"""The factorisation's envelope on the host: exact-zero tile flags, the envelope `tend`, the row profile, and executed
flops.

The device computes the same envelope from the values its fill stored (fill.cuh envelope_kernel); these functions
restate it for the tests and for tools/envelope_flops.py.  Tiles are NB x NB with front padding (the first
padded(N) - N rows and columns are the identity), as in the factorisation workspace.
"""
import numpy as np

from .constants import c_kms

NB = 128


def padded_tiles(N):
    return (int(N) + NB - 1) // NB


def tile_flags_from_matrix(K):
    """flags[I, J] (J <= I): does lower tile (I, J) of the padded matrix K [T*NB, T*NB] hold an entry != 0?"""
    T = K.shape[0] // NB
    B = K.reshape(T, NB, T, NB)
    return np.tril(np.any(B != 0.0, axis=(1, 3)))


def tile_flags_from_z(zs, amps, ls, sigma):
    """Exact-zero tile flags of K = sum_c amp_c^2 exp(p2_c (z_j - z_i)^2) + diag(sigma^2), padded as the device pads it,
    evaluated with numpy's exp of the same (p2 r) r.  zs: [ncomp, N] shifted ln-wavelengths."""
    zs = [np.asarray(z, dtype=np.float64) for z in zs]
    N = len(zs[0])
    T = padded_tiles(N)
    pad = T * NB - N
    flags = np.zeros((T, T), dtype=bool)
    p2s = [-0.5 * c_kms ** 2 / (l * l) for l in ls]
    for I in range(T):
        r0, r1 = max(I * NB - pad, 0), (I + 1) * NB - pad
        flags[I, I] = True   # the diagonal tile holds the diagonal (or the padding's identity)
        if r1 <= 0:
            continue
        nzcol = np.zeros(N, dtype=bool)
        for z, a, p2 in zip(zs, amps, p2s):
            r = z[None, :] - z[r0:r1, None]
            nzcol |= np.any(a * a * np.exp((p2 * r) * r) != 0.0, axis=0)
        cols = np.nonzero(nzcol[:r1])[0]   # lower tiles: columns up to the end of row tile I
        J = np.unique((cols + pad) // NB)
        flags[I, J] = True
    return flags


def row_profile(flags):
    """int[T]: F[I], the suffix minimum of the first non-zero block column f[I] of every row tile (I itself when the
    row has no non-zero tile before its diagonal).  Row tile I is exactly zero in block columns < F[I], in K and in L."""
    T = flags.shape[0]
    f = np.array([next((J for J in range(I) if flags[I, J]), I) for I in range(T)], dtype=np.int64)
    return np.minimum.accumulate(f[::-1])[::-1]


def tend_by_end(flags):
    """int[T + 1]: tend[e] = min{I >= e : F[I] >= e} (T when there is none), F = row_profile(flags); tend[0] = T."""
    T = flags.shape[0]
    F = row_profile(flags)
    tend = np.full(T + 1, T, dtype=np.int64)
    for e in range(1, T + 1):
        I = e
        while I < T and F[I] < e:
            I += 1
        tend[e] = I
    return tend


def group_starts(T, G):
    return list(range(0, T, G)) + [T]


def executed_flops(T, G, tend=None, prof=None):
    """DMMA flops the grouped factorisation executes for T row blocks and groups of G panels (uniform groups; chain 3
    panel solves, 2 * 128 * 64 * (64 + 128) per row block; trailing and in-group updates as 128 x 64 tiles, diagonal
    tiles in full).  tend None: the dense factorisation.  prof (row_profile; with tend): the update tiles of row block
    I start their k loop at panel max(a, prof[I]) of the group [a, e), and run at least one 16-column stage."""
    gs = group_starts(T, G)
    tile = 2.0 * NB * 64
    total = 0.0

    def k_len(I, a, kb):
        """k columns a 128 x 64 update tile of row block I runs over the panels [a, kb)."""
        if prof is None:
            return NB * (kb - a)
        return max(16, NB * (kb - max(a, int(prof[I]))))

    for q in range(len(gs) - 1):
        a, e = gs[q], gs[q + 1]
        end = T if tend is None else int(tend[e])
        for g in range(e - a):
            kb = a + g
            if g > 0:                                            # column update of block column kb, K <= 128 g
                total += sum(2 * tile * k_len(I, a, kb) for I in range(kb, end))
            total += 2 * max(end - kb - 1, 0) * tile * 96        # panel solve: two 128 x 64 tiles, K = 64 and 128
        # the group's trailing update: row block e + r owns 2 r + 2 tiles
        total += sum((2 * r + 2) * tile * k_len(e + r, a, e) for r in range(end - e))
    return total


def sorted_chunk_z(chunk, model_vel):
    """A chunk's pixels in wavelength order and its per-component shifted ln-wavelengths in that order.
    model_vel: [ncomp, n_epochs] velocities (km/s).  Returns (order, zs [ncomp, N])."""
    order = np.argsort(np.asarray(chunk["lwl"]), kind="stable")
    lwl = np.asarray(chunk["lwl"], dtype=np.float64)[order]
    ep = np.asarray(chunk["epoch"])[order]
    zs = np.array([lwl + (-np.asarray(v, dtype=np.float64)[ep]) / c_kms for v in model_vel])
    return order, zs
