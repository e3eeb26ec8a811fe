"""The envelope-restricted factorisation on covariances with a constructed exact-zero pattern and a closed-form likelihood.

Pixels come in clusters of identical ln-wavelengths, cluster centres DZ = 1e-2 apart in z.  Inside a cluster r = 0, so
exp_neg(-0.0) = 1 and K_ij = sum_c amp_c^2 exactly; between clusters p2 r^2 <= -9e4 (l <= 7 km/s), far below the -745.2
where exp_neg returns an exact +0.  With dyadic amplitudes and integer sigma, K is exact in FP64 and its tile zero
pattern is known on the host without any exponential.  The pixel order is free: placing a cluster's members anywhere
couples any chosen row and column tiles, which gives gapped profiles, rows that reach back past earlier rows, empty
rows, and envelopes that end on or one past a panel group's end.

With identical z for every component, K is block diagonal up to the pixel permutation, each block A 11^T + diag(sigma^2)
(A = sum_c amp_c^2), so Sherman-Morrison and the matrix determinant lemma give the likelihood in O(N):

    quad   = sum_clusters [ S_rr - A S_r^2 / (1 + A S_1) ]      S_1 = sum 1/sigma^2, S_r = sum r/sigma^2, S_rr = sum r^2/sigma^2
    logdet = sum_pixels log sigma^2 + sum_clusters log(1 + A S_1)

quad is an exact rational here (r = fl - mu is a multiple of 1/64); logdet is evaluated by mpmath at 40 digits.  This
reference knows nothing about tiles, and its cost does not depend on how the matrix is factored.

CPU: each pattern's exact K, tile flags (envelope.tile_flags_from_matrix) and envelope (envelope.tend_by_end) have the
property the pattern is built for; the closed form agrees with a dense scipy Cholesky of the same K.
GPU (-m gpu): the device envelope equals the host one; psoap_lnlike on the unsorted pixels against the closed form at
N = 1 .. 24577 and 1 to 3 components; the restricted lnlike == the unrestricted gradient elimination's under launch
switches that give both the same plan, also with a different cluster assignment per component; the farm (SB1, SB2, ST3
with zero orbital velocities) against the closed form in graph and direct issue, and against lone psoap_lnlike calls.
"""
import ctypes
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from psoap_b200 import envelope  # noqa: E402
from psoap_b200.constants import c_kms  # noqa: E402
from test_envelope import SAME_PLAN_ENVS  # noqa: E402

gpu = pytest.mark.gpu
NB = envelope.NB
Z0, DZ = 8.5, 1e-2
MU = 1.0
AMPS = (1.0, 0.5, 0.75)      # dyadic: amp^2 and every sum of them exact
LS = (5.0, 7.0, 6.0)
# |got - closed form| <= TOL (|quad| + |logdet|) for quad, logdet and lnlike.  scipy's Cholesky of the same K stays
# below 3e-16 on every pattern at N <= 6000 and 1 to 3 components (test_closed_form_matches_scipy asserts TOL / 10 at
# N <= 2049); TOL leaves room for the chains' explicit inverses of the diagonal blocks (cond * eps, DESIGN §6), as
# test_factor_exact does.
TOL = 1e-12
SIZES = [1, 127, 128, 129, 1000, 2049, 6000]
LARGE_N = 24577               # T = 193: the direct API takes chain 3 and G = 4 by itself


def geometry(N):
    """(T, pad): row blocks and front padding of the factorisation workspace; pixel i sits at padded row i + pad."""
    T = envelope.padded_tiles(N)
    return T, T * NB - N


# ---------------------------------------------------------------------------------------------- patterns
# Each builder returns one cluster label per pixel (pixel order = row order of psoap_lnlike).
def _diag(N):
    """Every pixel alone: K is diagonal, tend[e] == e (every trailing update and panel solve is empty)."""
    return np.arange(N)


def _dense(N):
    """One cluster: every tile is non-zero, tend == T."""
    return np.zeros(N, dtype=np.int64)


def _band(N, width):
    """Clusters of `width` tiles that start and end in the middle of a tile: row tile I reaches back `width` tiles at
    most."""
    _, pad = geometry(N)
    L = width * NB
    return (np.arange(N) + pad + L - NB // 2) // L


def _band1(N):
    return _band(N, 1)


def _band3(N):
    return _band(N, 3)


def _widening(N):
    """Contiguous clusters whose length grows from half a tile at the ends to several tiles in the middle."""
    T, pad = geometry(N)
    Np = T * NB
    wmax = max(1, T // 6)
    starts, b = [0], NB // 2
    while b < Np:
        starts.append(b)
        w = 1 + int(round(wmax * (1.0 - abs(2.0 * b / Np - 1.0))))
        b += w * NB
    return np.searchsorted(np.array(starts), np.arange(N) + pad, side="right") - 1


def _gapped(N):
    """Row tile I >= 2 is coupled to its diagonal tile and to ONE earlier tile J <= I - 2, zero tiles between: the first
    pixel of tile I shares a cluster with one pixel taken in order from tile 0 on (tile 0 while it has pixels left)."""
    T, pad = geometry(N)
    lab = np.arange(N)
    receivers = [I * NB - pad for I in range(2, T)]
    taken = set(receivers)
    donors = (i for i in range(N) if i not in taken)
    for I, rcv in zip(range(2, T), receivers):
        d = next(donors)
        assert (d + pad) // NB <= I - 2
        lab[d] = lab[rcv]
    return lab


def _out_of_order(N):
    """band1, and the first pixel of row tile T - 2 joins the band cluster of the first pixel of the matrix: that row
    reaches back to column 0 past every earlier row, so only the suffix minimum of f keeps the earlier groups' rows up to
    it."""
    T, pad = geometry(N)
    lab = _band1(N)
    if T >= 4:
        lab[(T - 2) * NB - pad] = lab[0]
    return lab


def _group_edges(N):
    """Whole-tile blocks [0, 8), [8, 17), [17, 24), [24, 33), ...: the envelope of the group that ends at 8 j + 8 ends
    on the group end (j even) or one row block past it (j odd) for G = 1, 2, 4 and 8."""
    T, pad = geometry(N)
    bounds = [0] + sorted([16 * j + 8 for j in range(T // 16 + 1)] + [16 * j + 17 for j in range(T // 16 + 1)])
    return np.searchsorted(np.array(bounds), (np.arange(N) + pad) // NB, side="right") - 1


def _pad_only(N):
    """The pixels of tile 0 (which holds the front padding) and the first pixel of tile 1 form one cluster; every other
    pixel is alone: the only off-diagonal tile is (1, 0)."""
    T, pad = geometry(N)
    lab = np.arange(N) + 1
    lab[:min(N, NB - pad + 1)] = 0
    return lab


PATTERNS = {"diag": _diag, "dense": _dense, "band1": _band1, "band3": _band3, "widening": _widening,
            "gapped": _gapped, "out_of_order": _out_of_order, "group_edges": _group_edges, "pad_only": _pad_only}
# the farm orders pixels by ln-wavelength: only patterns whose labels already rise with the pixel index reach it intact
SORTED = ["diag", "dense", "band1", "band3", "widening", "group_edges", "pad_only"]
# components 2 and 3 of the mixed cases take these patterns' labels (dense would make every union dense)
_CYCLE = ["diag", "band1", "band3", "widening", "gapped", "out_of_order", "group_edges", "pad_only"]


def companions(name, ncomp):
    i = _CYCLE.index(name) if name in _CYCLE else 0
    return [name] + [_CYCLE[(i + 3 * c) % len(_CYCLE)] for c in range(1, ncomp)]


def make_case(name, N, ncomp, mixed=False, seed=0):
    """Inputs of one case: per-component labels and z, fl = MU + k/64, integer sigma in 1..3, amplitudes, lengths."""
    names = companions(name, ncomp) if mixed else [name] * ncomp
    labels = [np.asarray(PATTERNS[n](N), dtype=np.int64) for n in names]
    rng = np.random.default_rng(1000 * N + 17 * ncomp + seed)
    k = rng.integers(-32, 33, size=N)
    return dict(name=name, N=N, labels=labels, zs=[Z0 + DZ * lab for lab in labels], fl=MU + k / 64.0,
                sigma=rng.integers(1, 4, size=N).astype(np.float64), amps=list(AMPS[:ncomp]), ls=list(LS[:ncomp]),
                A=sum(a * a for a in AMPS[:ncomp]))


def cluster_flags(labels, N):
    """Tile flags of the padded K from the cluster labels alone (lower tiles (I, J) that share a cluster, and the
    diagonal)."""
    T, pad = geometry(N)
    flags = np.eye(T, dtype=bool)
    tile = (np.arange(N) + pad) // NB
    for lab in labels:
        pairs = np.unique(np.stack([lab, tile], axis=1), axis=0)
        _, start, count = np.unique(pairs[:, 0], return_index=True, return_counts=True)
        for s, c in zip(start[count > 1], count[count > 1]):
            ts = pairs[s:s + c, 1]
            flags[np.ix_(ts, ts)] = True
    return np.tril(flags)


def exact_K(case):
    """The padded matrix the device fills, from z with numpy's exp (identity front padding)."""
    N = case["N"]
    T, pad = geometry(N)
    K = np.diag(case["sigma"] ** 2)
    for z, a, l in zip(case["zs"], case["amps"], case["ls"]):
        p2 = -0.5 * c_kms ** 2 / (l * l)
        D = z[None, :] - z[:, None]
        K += a * a * np.exp((p2 * D) * D)
    W = np.eye(T * NB)
    W[pad:, pad:] = K
    return W


def first_cols(flags):
    """f[I]: first non-zero block column of row tile I (I when none before the diagonal)."""
    return np.array([np.flatnonzero(flags[I, :I + 1])[0] for I in range(flags.shape[0])])


def closed_form(labels, fl, sigma, A, mu=MU):
    """(quad, logdet, lnlike) as mpmath numbers: quad exact, logdet at 40 digits.  labels: one cluster label per pixel
    (the same for every component), A = sum_c amp_c^2."""
    import mpmath
    k = np.rint((np.asarray(fl) - mu) * 64.0).astype(np.int64)
    assert np.array_equal(mu + k / 64.0, fl), "fl - mu must be a multiple of 1/64"
    s2 = np.rint(np.asarray(sigma) ** 2).astype(np.int64)
    assert np.array_equal(s2.astype(np.float64), np.asarray(sigma) ** 2), "sigma must be an integer"
    D = int(np.lcm.reduce(np.unique(s2)))
    w = D // s2                                        # 1/sigma^2 = w / D, integers
    _, inv = np.unique(labels, return_inverse=True)
    S1 = np.bincount(inv, weights=w)                   # every partial sum an integer below 2^53
    Sr = np.bincount(inv, weights=w * k)
    Srr = np.bincount(inv, weights=w * k * k)
    Af = Fraction(A)
    quad = Fraction(0)
    for s1, sr, srr in zip(S1, Sr, Srr):
        s1, sr, srr = Fraction(int(s1), D), Fraction(int(sr), 64 * D), Fraction(int(srr), 4096 * D)
        quad += srr - Af * sr * sr / (1 + Af * s1)
    with mpmath.workdps(40):
        vals, cnt = np.unique(s2, return_counts=True)
        logdet = mpmath.fsum(int(c) * mpmath.log(int(v)) for v, c in zip(vals, cnt))
        vals, cnt = np.unique(S1, return_counts=True)
        logdet += mpmath.fsum(int(c) * mpmath.log(1 + mpmath.mpf(A) * int(v) / D) for v, c in zip(vals, cnt))
        q = mpmath.mpf(quad.numerator) / quad.denominator
        return dict(quad=+q, logdet=+logdet, lnlike=-(q + logdet) / 2)


def rel_err(got, ref):
    """max over quad, logdet and lnlike of |got - ref| / (|quad| + |logdet|), as a float."""
    import mpmath
    with mpmath.workdps(40):
        scale = abs(ref["quad"]) + abs(ref["logdet"])
        return float(max(abs(mpmath.mpf(got[key]) - ref[key]) for key in ("quad", "logdet", "lnlike")) / scale)


# ---------------------------------------------------------------------------------------------- CPU
def _check_property(name, N, flags, tend):
    T, pad = geometry(N)
    f = first_cols(flags)
    off = np.tril(flags, -1)
    e = np.arange(1, T + 1)
    if name == "diag":
        assert not off.any() and np.array_equal(tend[1:], e)
    elif name == "dense":
        assert flags.all() if T == 1 else np.array_equal(flags, np.tril(np.ones((T, T), dtype=bool)))
        assert np.all(tend == T)
    elif name in ("band1", "band3"):
        w = 1 if name == "band1" else 3
        reach = np.arange(T) - f
        assert np.array_equal(reach[1:], [min((I - 1) % w + 1, I) for I in range(1, T)]), reach
        assert all(flags[I, f[I]:I + 1].all() for I in range(T))          # no gaps inside the band
        want = [min(e0 + w - (e0 - 1) % w, T) for e0 in range(1, T + 1)]
        assert np.array_equal(tend[1:], want), (tend, want)
    elif name == "widening":
        reach = np.arange(T) - f
        assert all(flags[I, f[I]:I + 1].all() for I in range(T))
        if T >= 40:
            mid = reach[T // 3:2 * T // 3].max()
            assert mid >= 4 and mid > reach[:T // 8].max() and mid > reach[-(T // 8):].max(), reach
    elif name == "gapped":
        for I in range(2, T):
            assert np.array_equal(np.flatnonzero(flags[I]), [f[I], I]) and f[I] <= I - 2, (I, f[I])
        if T > 1:
            assert not off[1].any()
        if NB - pad >= T - 2:
            assert np.all(f[2:] == 0)
    elif name == "out_of_order":
        if T >= 4:
            assert f[T - 2] == 0 and all(f[I] == I - 1 for I in range(1, T) if I != T - 2)
            assert np.all(tend[1:T - 1] == T - 1) and tend[T - 1] == T
            # without the suffix minimum the envelope of group e would end at e + 1 and cut row T - 2 off
            naive = [next((I for I in range(e0, T) if f[I] >= e0), T) for e0 in range(1, T + 1)]
            assert any(n < t for n, t in zip(naive, tend[1:]))
            if T >= 6:
                assert not flags[T - 2, 2:T - 3].any()                    # a gapped row
    elif name == "group_edges":
        if T >= 17:
            for G in (1, 2, 4, 8):
                ends = range(G, T, G)
                assert any(tend[x] == x for x in ends) and any(tend[x] == x + 1 for x in ends), (G, tend)
    elif name == "pad_only":
        assert set(zip(*np.nonzero(off))) == ({(1, 0)} if T >= 2 else set())
        if T >= 2:
            assert tend[1] == 2 and np.array_equal(tend[2:], e[1:])
    else:
        raise KeyError(name)


@pytest.mark.parametrize("name", list(PATTERNS))
def test_pattern_has_its_shape(name):
    """The exact K, its tile flags and its envelope, at every size the GPU tests use: the flags from the matrix
    (and from z, as test_envelope computes them) equal the flags from the labels where the matrix is affordable."""
    for N in SIZES + [LARGE_N]:
        case = make_case(name, N, 1)
        flags = cluster_flags(case["labels"], N)
        if N <= 2049:
            K = exact_K(case)
            T, pad = geometry(N)
            lab = case["labels"][0]
            same = lab[:, None] == lab[None, :]
            assert np.array_equal(K[pad:, pad:], np.where(same, case["A"], 0.0) + np.diag(case["sigma"] ** 2))
            assert np.array_equal(envelope.tile_flags_from_matrix(K), flags), (name, N)
            assert np.array_equal(envelope.tile_flags_from_z(case["zs"], case["amps"], case["ls"], case["sigma"]),
                                  flags), (name, N)
        tend = envelope.tend_by_end(flags)
        assert tend[0] == geometry(N)[0]
        _check_property(name, N, flags, tend)


def test_mixed_components_take_the_union():
    """A different cluster assignment per component: the zero pattern of K is the union of the components' patterns."""
    for name in PATTERNS:
        case = make_case(name, 1000, 3, mixed=True)
        flags = cluster_flags(case["labels"], 1000)
        parts = [cluster_flags([lab], 1000) for lab in case["labels"]]
        assert np.array_equal(flags, parts[0] | parts[1] | parts[2])
        assert np.array_equal(envelope.tile_flags_from_matrix(exact_K(case)), flags), name
        assert len(set(companions(name, 3))) == 3


def test_sorted_patterns_keep_their_order():
    """The farm sorts each chunk's pixels by ln-wavelength (stable): the SORTED patterns come through unchanged, the
    others would be rebuilt into contiguous clusters."""
    for name in PATTERNS:
        z = make_case(name, 2049, 1)["zs"][0]
        kept = np.array_equal(np.argsort(z, kind="stable"), np.arange(len(z)))
        assert kept == (name in SORTED), name


@pytest.mark.parametrize("N", [1, 127, 129, 1000, 2049])
def test_closed_form_matches_scipy(N):
    """The reference itself: a dense FP64 LAPACK Cholesky of the same K agrees with it at TOL / 10 or better."""
    from scipy.linalg import cho_factor, cho_solve
    worst = 0.0
    for name in PATTERNS:
        for ncomp in (1, 2, 3):
            case = make_case(name, N, ncomp)
            T, pad = geometry(N)
            cf = cho_factor(exact_K(case)[pad:, pad:], lower=True)
            r = case["fl"] - MU
            quad = float(r @ cho_solve(cf, r))
            logdet = 2.0 * float(np.sum(np.log(np.diagonal(cf[0]))))
            ref = closed_form(case["labels"][0], case["fl"], case["sigma"], case["A"])
            worst = max(worst, rel_err(dict(quad=quad, logdet=logdet, lnlike=-0.5 * (quad + logdet)), ref))
    assert worst <= TOL / 10, worst


def test_sizes_reach_their_plans():
    """The direct API takes chain 3 and groups of 4 at N = 24577 by itself; at N = 2049 the last group of every forced
    group size is partial."""
    from test_factor_exact import direct_plan
    big = direct_plan(LARGE_N, 0, nsm=148)
    assert (big["Tt"], big["chain"], big["G"]) == (193, 3, 4)
    for G in (2, 4, 8):
        groups = direct_plan(2049, 0, nsm=148, env={"PSOAP_GROUP": str(G)})["groups"]
        assert groups[-1] == (16, 1) and all(size == G for _, size in groups[:-1])


def test_closed_form_small_cases_by_hand():
    """One pixel, and two pixels in one cluster, written out."""
    import mpmath
    with mpmath.workdps(40):
        ref = closed_form(np.array([0]), np.array([1.5]), np.array([2.0]), 1.0)   # K = 1 + 4, r = 1/2
        assert abs(ref["quad"] - mpmath.mpf(1) / 20) < 1e-38 and abs(ref["logdet"] - mpmath.log(5)) < 1e-38
        # K = [[1 + 1, 1], [1, 1 + 4]]: det 9, K^-1 = [[5, -1], [-1, 2]] / 9; r = (1/2, -1/4): quad = 13/72
        ref = closed_form(np.array([3, 3]), np.array([1.5, 0.75]), np.array([1.0, 2.0]), 1.0)
        assert abs(ref["quad"] - mpmath.mpf(13) / 72) < 1e-38 and abs(ref["logdet"] - mpmath.log(9)) < 1e-38


# ---------------------------------------------------------------------------------------------- GPU helpers
def device_lnlike(case, zs=None, fl=None, sigma=None, amps=None, ls=None):
    """psoap_lnlike on the case's pixels as given (no sorting): (tend read from the workspace, [lnlike, logdet, quad,
    info])."""
    import torch
    from psoap_b200 import _lib
    lib = _lib.load()
    zs = case["zs"] if zs is None else zs
    fl = case["fl"] if fl is None else fl
    sigma = case["sigma"] if sigma is None else sigma
    amps = case["amps"] if amps is None else amps
    ls = case["ls"] if ls is None else ls
    N, ncomp = len(fl), len(zs)
    zd = [torch.tensor(np.ascontiguousarray(z), dtype=torch.float64, device="cuda") for z in zs]
    fd = torch.tensor(np.ascontiguousarray(fl), dtype=torch.float64, device="cuda")
    sd = torch.tensor(np.ascontiguousarray(sigma), dtype=torch.float64, device="cuda")
    nbytes = lib.psoap_lnlike_workspace_bytes(N)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    wp = (ws.data_ptr() + 255) // 256 * 256
    res = torch.full((4,), 7.0, dtype=torch.float64, device="cuda")
    ptrs = [z.data_ptr() for z in zd] + [None] * (3 - ncomp)
    _lib.check(lib.psoap_lnlike(ncomp, N, ptrs[0], ptrs[1], ptrs[2], fd.data_ptr(), sd.data_ptr(), _lib.dbl_array(amps),
                                _lib.dbl_array(ls), MU, wp, nbytes, res.data_ptr(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    tp, T = _lib.vp(), ctypes.c_int()
    _lib.check(lib.psoap_lnlike_envelope_view(wp, N, ctypes.byref(tp), ctypes.byref(T)))
    off = tp.value - ws.data_ptr()
    tend = ws[off:off + 4 * (T.value + 1)].view(torch.int32).cpu().numpy().astype(np.int64)
    return tend, res.cpu().numpy()


def as_result(res):
    return dict(lnlike=float(res[0]), logdet=float(res[1]), quad=float(res[2]))


def check_against_closed_form(case, res, what):
    assert res[3] == 0.0, (what, "info", res[3])
    ref = closed_form(case["labels"][0], case["fl"], case["sigma"], case["A"])
    err = rel_err(as_result(res), ref)
    assert err <= TOL, (what, err, as_result(res), {k: float(v) for k, v in ref.items()})


# ---------------------------------------------------------------------------------------------- GPU
@gpu
@pytest.mark.parametrize("name", list(PATTERNS))
def test_device_envelope_matches_host(name):
    """tend read through psoap_lnlike_envelope_view == tend_by_end of the exact flags, one component and three with
    different cluster assignments, at every size."""
    for N in SIZES + [LARGE_N]:
        for ncomp, mixed in ((1, False), (3, True)):
            if N == LARGE_N and mixed:
                continue
            case = make_case(name, N, ncomp, mixed=mixed)
            tend, _ = device_lnlike(case)
            want = envelope.tend_by_end(cluster_flags(case["labels"], N))
            assert np.array_equal(tend, want), (name, N, ncomp, tend, want)


@gpu
@pytest.mark.parametrize("N", SIZES)
@pytest.mark.parametrize("name", list(PATTERNS))
def test_restricted_factorisation_against_closed_form(name, N):
    """psoap_lnlike on the unsorted pixels, 1, 2 and 3 components with identical z: quad, logdet and lnlike within TOL
    of the closed form."""
    for ncomp in (1, 2, 3):
        case = make_case(name, N, ncomp)
        _, res = device_lnlike(case)
        check_against_closed_form(case, res, (name, N, ncomp))


@gpu
@pytest.mark.parametrize("name", list(PATTERNS))
def test_restricted_factorisation_large(name):
    """N = 24577 (T = 193): the direct API's own plan there is chain 3 with groups of 4."""
    import torch
    case = make_case(name, LARGE_N, 1)
    _, res = device_lnlike(case)
    check_against_closed_form(case, res, (name, LARGE_N))
    torch.cuda.empty_cache()


def _child_same_bits():
    """psoap_lnlike == the lnlike of the unrestricted gradient elimination (psoap_lnlike_grad) on every pattern."""
    from psoap_b200 import covariance
    n = 0
    for name in PATTERNS:
        for N in (1, 129, 1000, 2049, 6000):
            for ncomp, mixed in ((1, False), (2, True), (3, True)):
                case = make_case(name, N, ncomp, mixed=mixed)
                tend, res = device_lnlike(case)
                assert np.array_equal(tend, envelope.tend_by_end(cluster_flags(case["labels"], N))), (name, N, ncomp)
                g = covariance.lnlike_grad(case["zs"], case["fl"], case["sigma"], case["amps"], case["ls"], MU)
                assert res[0] == g.lnlike, (name, N, ncomp, res[0], g.lnlike)
                n += 1
    print("same bits ok: %d cases" % n)


@gpu
@pytest.mark.parametrize("cfg", sorted(SAME_PLAN_ENVS))
def test_restricted_equals_unrestricted(cfg):
    r = _run_child(["same-bits"], SAME_PLAN_ENVS[cfg])
    assert r.returncode == 0 and "same bits ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ------------------------------------------------------------------------------------ farm
# Zero orbital velocities (K = 0, gamma = 0): the farm's shifted z = lwl + (-0)/c are the lwl bits, the same for every
# component, so the closed form applies.  The farm sorts each chunk by lwl, so only the SORTED patterns reach it as
# built; that is the order every farm path factors in.
FARM_CHUNKS = [("band1", 2049), ("dense", 1500), ("group_edges", 2049), ("widening", 6000), ("band3", 3000),
               ("diag", 1000), ("pad_only", 129), ("dense", 1)]
FARM_ORBITS = {"SB1": [0.0, 0.2, 10.0, 10.0, 0.0, 0.0],
               "SB2": [0.2, 0.0, 0.2, 10.0, 10.0, 0.0, 0.0],
               "ST3": [0.4, 0.0, 0.2, 10.0, 10.0, 0.0, 0.2, 0.0, 0.2, 80.0, 100.0, 3.0, 0.0]}
FARM_NCOMP = {"SB1": 1, "SB2": 2, "ST3": 3}
FARM_K = 8                    # 8 chunks x 8 proposals = 64 pairs: chain 3 and rank-1024 updates (G = 8)
FEW = 3                       # 3 chunks x 1 proposal: chain 7 and look-ahead, the direct API's defaults
# under these switches a lone psoap_lnlike takes the G = 8 farm's plan (chain 3, groups of 8, no look-ahead)
FARM_PLAN_ENV = {"PSOAP_POTRF": "3", "PSOAP_GROUP": "8", "PSOAP_LOOKAHEAD": "0", "PSOAP_FARM_LOOKAHEAD": "0"}
FARM_ISSUES = {"graph": {}, "direct": {"PSOAP_FARM_DIRECT": "1"}, "g8-plan": FARM_PLAN_ENV}


def farm_chunk(name, N, seed):
    case = make_case(name, N, 1, seed=seed)
    assert name in SORTED
    return dict(lwl=case["zs"][0], fl=case["fl"], sigma=case["sigma"], epoch=(np.arange(N) % 3).astype(np.int32),
                date1D=np.array([0.5, 1.5, 2.5])), case["labels"][0]


def farm_proposals(model, K):
    """K vectors with zero velocities and distinct dyadic amplitudes (l in 5..7 km/s keeps clusters apart)."""
    amp_choices, nc = (1.0, 0.5, 0.75, 1.25), FARM_NCOMP[model]
    P = []
    for k in range(K):
        gp = []
        for c in range(nc):
            gp += [amp_choices[(k + c) % 4], 5.0 + (k + 2 * c) % 3]
        P.append(FARM_ORBITS[model] + gp)
    return np.array(P)


def _farm_check(model, farm, chunks, labels, P, same_plan, what):
    """Per-chunk lnlike, logdet and quad against the closed form, the sums against the closed form, and every chunk
    against a lone psoap_lnlike on the farm's sorted pixels (== when same_plan)."""
    import mpmath
    nc = FARM_NCOMP[model]
    K = P.shape[0]
    sums = farm.lnprob_many(P) if K > 1 else np.array([farm.lnprob(P[0])])
    res = farm._results.cpu().numpy()
    assert res.shape[:2] == (K, len(chunks))
    for k in range(K):
        amps, ls = list(P[k, -2 * nc::2]), list(P[k, -2 * nc + 1::2])
        A = sum(a * a for a in amps)
        refs = []
        for i, (ch, lab) in enumerate(zip(chunks, labels)):
            tag = (what, model, k, i, len(ch["fl"]))
            assert res[k, i, 3] == 0.0, tag
            ref = closed_form(lab, ch["fl"], ch["sigma"], A)
            refs.append(ref)
            assert rel_err(as_result(res[k, i]), ref) <= TOL, (tag, as_result(res[k, i]))
            order = np.argsort(ch["lwl"], kind="stable")
            assert np.array_equal(order, np.arange(len(order)))
            _, lone = device_lnlike(None, zs=[ch["lwl"][order]] * nc, fl=ch["fl"][order], sigma=ch["sigma"][order],
                                    amps=amps, ls=ls)
            if same_plan:
                assert lone[0] == res[k, i, 0], (tag, lone[0], res[k, i, 0])
            else:
                assert abs(lone[0] - res[k, i, 0]) <= TOL * float(abs(ref["quad"]) + abs(ref["logdet"])), tag
        with mpmath.workdps(40):
            total = mpmath.fsum(r["lnlike"] for r in refs)
            scale = mpmath.fsum(abs(r["quad"]) + abs(r["logdet"]) for r in refs)
            assert float(abs(mpmath.mpf(sums[k]) - total) / scale) <= TOL, (what, model, k, sums[k], float(total))


def farm_case(issue):
    """Every model: lnprob on FEW chunks (chain 7, look-ahead) and lnprob_many on 8 chunks x 8 proposals (chain 3,
    G = 8).  A lone call shares the few-chunk farm's plan under the defaults and the G = 8 farm's under FARM_PLAN_ENV."""
    from psoap_b200.farm import ChunkFarm
    for model in ("SB1", "SB2", "ST3"):
        built = [farm_chunk(name, N, seed=i) for i, (name, N) in enumerate(FARM_CHUNKS)]
        chunks, labels = [b[0] for b in built], [b[1] for b in built]
        few = ChunkFarm(model, chunks[:FEW])
        assert few._descs[0].reserved == 7 | (4 << 8)                    # chain 7 (look-ahead by branch count)
        _farm_check(model, few, chunks[:FEW], labels[:FEW], farm_proposals(model, 1), issue != "g8-plan", (issue, "few"))
        few.close()
        many = ChunkFarm(model, chunks, n_proposals=FARM_K)
        assert many._descs[0].reserved == 3 | (8 << 8)                   # chain 3, G = 8
        _farm_check(model, many, chunks, labels, farm_proposals(model, FARM_K), issue == "g8-plan", (issue, "many"))
        many.close()
    print("farm ok: " + issue)


@gpu
@pytest.mark.parametrize("issue", sorted(FARM_ISSUES))
def test_farm_plans_against_closed_form(issue):
    if issue == "graph":
        farm_case(issue)
        return
    r = _run_child(["farm", issue], FARM_ISSUES[issue])
    assert r.returncode == 0 and ("farm ok: " + issue) in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def _run_child(args, env_extra):
    """This file as a script in a child process: the launch switches are read once per process."""
    env = dict(os.environ, **env_extra)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    return subprocess.run([sys.executable, "-s", os.path.abspath(__file__)] + args, env=env, capture_output=True,
                          text=True, timeout=900)


if __name__ == "__main__":
    if sys.argv[1:] == ["same-bits"]:
        _child_same_bits()
    elif sys.argv[1:2] == ["farm"]:
        farm_case(sys.argv[2])
