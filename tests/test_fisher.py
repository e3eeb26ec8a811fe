"""Expected Fisher information of a chunk's likelihood (psoap_chunk_fisher, ChunkFarm.fisher, sample.fisher_jump).

CPU: a numpy reference np_fisher (K from the oracle, analytic dK/dp_a, 1/2 tr(K^-1 D_a K^-1 D_b)), its D_a checked
against central differences of the oracle's K and its F against second differences of the expected log-likelihood's
closed form; fisher_jump's subset, scaling and errors.
GPU (-m gpu): the device F against np_fisher (SB1, SB2, ST3; N = 1 .. ~1500; epoch-major and wavelength-sorted
pixels), a C4-sized chunk against a torch FP64 comparator, the exact properties (symmetry, the zero gamma row, bit
stability over calls and emulated ranks, result and gradient equal to psoap_chunk_lnprob_grad's), the k ranges against
the tile flags, the -inf conventions, and sample.run with fisher_jump.
"""
import ctypes

import numpy as np
import pytest

from test_gradient import C_KMS, NCOMP, NORB, np_velocity_jacobian

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- numpy reference
def chunk_z(model, chunk, p):
    """Shifted ln-wavelengths [ncomp, N] of the chunk's pixels (lwl + (-v)/c at each pixel's epoch), with a constant
    taken off lwl first: K depends on differences only, and small z keep finite differences free of rounding noise."""
    from oracle import oracle as orc
    vel = np.asarray(orc.get_velocities(model, p[:NORB[model]], chunk["date1D"]))
    lwl = np.asarray(chunk["lwl"]) - np.log(5000.0)
    return np.array([lwl + (-vel[c][chunk["epoch"]]) / C_KMS for c in range(NCOMP[model])])


def oracle_K(model, z, sigma, gp):
    from oracle import oracle as orc
    N = z.shape[1]
    K = np.empty((N, N))
    fill = {1: orc.fill_V11_f, 2: orc.fill_V11_f_g, 3: orc.fill_V11_f_g_h}[NCOMP[model]]
    fill(K, *z, *gp)
    K[np.diag_indices_from(K)] += np.asarray(sigma) ** 2
    return K


def np_dK(model, chunk, p):
    """[P, N, N] analytic dK/dp_a in the registered order (orbital, then amp_c, l_c)."""
    no, nc = NORB[model], NCOMP[model]
    z = chunk_z(model, chunk, p)
    J = np_velocity_jacobian(model, p[:no], chunk["date1D"])          # [ncomp, n_epochs, norb]
    ep = chunk["epoch"]
    N = len(ep)
    D = np.zeros((no + 2 * nc, N, N))
    for c in range(nc):
        amp, l = p[no + 2 * c], p[no + 2 * c + 1]
        p2 = -0.5 * C_KMS ** 2 / (l * l)
        r = z[c][None, :] - z[c][:, None]       # r_ij = z_j - z_i
        x = p2 * r * r
        e = np.exp(x)
        k = amp * amp * e
        D[no + 2 * c] = 2.0 * amp * e
        D[no + 2 * c + 1] = -2.0 * k * x / l
        u = -J[c][ep] / C_KMS                   # [N, norb]
        for a in range(no):
            D[a] += 2.0 * p2 * k * r * (u[None, :, a] - u[:, None, a])
    return D


def np_fisher(model, chunk, p, mu=1.0):
    """F [P, P] = 1/2 tr(K^-1 D_a K^-1 D_b) (mu does not enter: the mean is not a registered parameter)."""
    from scipy.linalg import cho_factor, cho_solve
    no = NORB[model]
    K = oracle_K(model, chunk_z(model, chunk, p), chunk["sigma"], p[no:])
    Kinv = cho_solve(cho_factor(K, lower=True), np.eye(len(K)))
    A = np.einsum("ij,ajk->aik", Kinv, np_dK(model, chunk, p))
    return 0.5 * np.einsum("aij,bji->ab", A, A)


def small_chunk(model, n_epochs, n_pix, seed, sort=False):
    from psoap_b200 import synthetic
    ch = synthetic.make_chunk(model, n_epochs, n_pix, seed=seed)
    if sort:
        order = np.argsort(ch["lwl"], kind="stable")
        for k in ("lwl", "fl", "sigma", "epoch"):
            ch[k] = np.ascontiguousarray(ch[k][order])
    return ch


def param_steps(model, p):
    from psoap_b200 import utils
    names = utils.registered_params[model]
    return np.array([1e-5 * max(abs(v), 1.0) for n, v in zip(names, p)])


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_dK_matches_central_differences(model):
    from psoap_b200 import synthetic, utils
    ch = small_chunk(model, 5, 12, seed=21)
    p = synthetic.default_params(model)
    no = NORB[model]
    D = np_dK(model, ch, p)
    h = param_steps(model, p)
    for a, name in enumerate(utils.registered_params[model]):
        up, dn = p.copy(), p.copy()
        up[a] += h[a]; dn[a] -= h[a]
        fd = (oracle_K(model, chunk_z(model, ch, up), ch["sigma"], up[no:])
              - oracle_K(model, chunk_z(model, ch, dn), ch["sigma"], dn[no:])) / (2 * h[a])
        if name == "gamma":
            assert np.all(D[a] == 0.0)
            assert np.abs(fd).max() <= 1e-9, np.abs(fd).max()
        else:
            assert np.abs(fd - D[a]).max() <= 1e-6 * np.abs(D[a]).max(), (name, np.abs(fd - D[a]).max(), np.abs(D[a]).max())


@pytest.mark.parametrize("model", ["SB1", "SB2"])
def test_fisher_matches_second_differences_of_expected_lnlike(model):
    """F_ab = -d^2/dt'_a dt'_b E_t[lnL(t')] at t' = t, E_t[lnL(t')] = -1/2 (tr(K(t')^-1 K(t)) + log det K(t'))."""
    from psoap_b200 import synthetic
    ch = small_chunk(model, 4, 10, seed=5)
    p = synthetic.default_params(model)
    no = NORB[model]
    K0 = oracle_K(model, chunk_z(model, ch, p), ch["sigma"], p[no:])

    def f(q):
        K = oracle_K(model, chunk_z(model, ch, q), ch["sigma"], q[no:])
        return -0.5 * (np.trace(np.linalg.solve(K, K0)) + np.linalg.slogdet(K)[1])

    F = np_fisher(model, ch, p)
    h = param_steps(model, p)
    P = len(p)
    fd = np.zeros((P, P))
    for a in range(P):
        for b in range(P):
            def at(sa, sb):
                q = p.copy()
                q[a] += sa * h[a]; q[b] += sb * h[b]
                return f(q)
            fd[a, b] = -(at(1, 1) - at(1, -1) - at(-1, 1) + at(-1, -1)) / (4 * h[a] * h[b])
    scale = np.sqrt(np.outer(np.diag(F), np.diag(F)))
    ok = np.abs(fd - F) <= 1e-4 * scale + 1e-6 * np.abs(F).max()
    assert ok.all(), (np.argwhere(~ok), fd[~ok], F[~ok])


def test_fisher_jump_subset_scaling_and_errors():
    from psoap_b200 import sample, utils
    names = utils.registered_params["SB2"]
    P = len(names)
    rng = np.random.default_rng(3)
    B = rng.standard_normal((P, P))
    F = B @ B.T + P * np.eye(P)
    g = names.index("gamma")
    F[g, :] = F[:, g] = 0.0
    fix = ["gamma", "T0"]
    keep = [i for i, n in enumerate(names) if n not in fix]
    cov = sample.fisher_jump(F, "SB2", fix)
    d = len(keep)
    assert cov.shape == (d, d)
    np.testing.assert_allclose(cov, 2.38 ** 2 / d * np.linalg.inv(F[np.ix_(keep, keep)]), rtol=1e-12)
    with pytest.raises(ValueError, match="gamma.*fix it"):
        sample.fisher_jump(F, "SB2", ["T0"])
    Fneg = F.copy()
    Fneg[0, 0] = -1.0
    with pytest.raises(ValueError, match="positive definite"):
        sample.fisher_jump(Fneg, "SB2", fix)


# ---------------------------------------------------------------------------------------------- GPU helpers
def _lib():
    from psoap_b200 import _lib as L
    return L, L.load()


def _desc(torch, ch, keep):
    from psoap_b200 import _lib as L
    t = {k: torch.from_numpy(np.ascontiguousarray(ch[k])).cuda() for k in ("lwl", "fl", "sigma", "date1D", "epoch")}
    keep.append(t)
    d = L.PsoapChunk()
    d.N, d.n_epochs = len(ch["fl"]), len(ch["date1D"])
    d.lwl, d.epoch, d.fl = t["lwl"].data_ptr(), t["epoch"].data_ptr(), t["fl"].data_ptr()
    d.sigma, d.dates = t["sigma"].data_ptr(), t["date1D"].data_ptr()
    return d


def chunk_fisher(model, ch, p, mu=1.0, views=False):
    """psoap_chunk_fisher on the chunk as given (no sorting): (result [4], grad_p [P], F [P, P]) and, with views,
    (flags [Tb, Tb], krange [Tb, 2])."""
    import torch
    L, lib = _lib()
    keep = []
    d = _desc(torch, ch, keep)
    m = L.MODELS[model]
    nb = lib.psoap_chunk_fisher_workspace_bytes(m, d.N, d.n_epochs)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    P = len(p)
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    gp = torch.empty(P, dtype=torch.float64, device="cuda")
    F = torch.empty((P, P), dtype=torch.float64, device="cuda")
    p_d = torch.from_numpy(np.asarray(p, dtype=np.float64)).cuda()
    L.check(lib.psoap_chunk_fisher(m, ctypes.byref(d), L.ptr(p_d), mu, L.ptr(ws), nb, L.ptr(res), L.ptr(gp), L.ptr(F),
                                   L.stream_ptr()))
    torch.cuda.synchronize()
    out = (res.cpu().numpy(), gp.cpu().numpy(), F.cpu().numpy())
    if not views:
        return out
    fl, kr, Tb = L.vp(), L.vp(), ctypes.c_int()
    L.check(lib.psoap_chunk_fisher_views(L.ptr(ws), m, d.N, d.n_epochs, ctypes.byref(fl), ctypes.byref(kr),
                                         ctypes.byref(Tb)))
    T = Tb.value
    base = ws.data_ptr()
    flags = ws[fl.value - base:fl.value - base + T * T].cpu().numpy().reshape(T, T)
    krange = ws[kr.value - base:kr.value - base + 8 * T].cpu().numpy().view(np.int32).reshape(T, 2)
    return out, flags, krange


def assert_fisher_close(got, ref, rtol):
    scale = np.sqrt(np.abs(np.outer(np.diag(ref), np.diag(ref))))
    err = np.abs(got - ref)
    assert np.all(err <= rtol * scale), (err / np.where(scale > 0, scale, 1)).max()


# ---------------------------------------------------------------------------------------------- GPU
SIZES = {1: (1, 1), 127: (1, 127), 128: (2, 64), 129: (3, 43), 700: (7, 100), 1500: (10, 150)}


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
@pytest.mark.parametrize("N", sorted(SIZES))
@pytest.mark.parametrize("order", ["epoch", "lwl"])
def test_chunk_fisher_matches_numpy(model, N, order):
    from psoap_b200 import synthetic
    ne, npix = SIZES[N]
    ch = small_chunk(model, ne, npix, seed=100 + N, sort=(order == "lwl"))
    p = synthetic.default_params(model)
    res, _, F = chunk_fisher(model, ch, p)
    assert res[3] == 0.0
    assert_fisher_close(F, np_fisher(model, ch, p), 1e-10)


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_farm_fisher_matches_numpy(model):
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [small_chunk(model, 4 + i, 60 + 40 * i, seed=200 + i) for i in range(3)]
    p = synthetic.default_params(model)
    farm = ChunkFarm(model, chunks)
    per = farm.chunk_fishers(p).cpu().numpy()
    for i, ch in enumerate(chunks):
        assert_fisher_close(per[i], np_fisher(model, ch, p), 1e-10)
    F = farm.fisher(p)
    assert np.array_equal(F, np.sum(per, axis=0))
    farm.close()


def _torch_fisher(torch, model, ch, p):
    """FP64 comparator on the device: K^-1 by cholesky_inverse, D_a as np_dK, A_a = K^-1 D_a by matmul."""
    no, nc = NORB[model], NCOMP[model]
    dev = dict(dtype=torch.float64, device="cuda")
    z = torch.tensor(chunk_z(model, ch, p), **dev)
    J = torch.tensor(np_velocity_jacobian(model, p[:no], ch["date1D"]), **dev)
    ep = torch.tensor(ch["epoch"], dtype=torch.int64, device="cuda")
    N = len(ch["fl"])
    K = torch.diag(torch.tensor(ch["sigma"], **dev) ** 2)
    terms = []
    for c in range(nc):
        amp, l = p[no + 2 * c], p[no + 2 * c + 1]
        p2 = -0.5 * C_KMS ** 2 / (l * l)
        r = z[c][None, :] - z[c][:, None]
        x = p2 * r * r
        e = torch.exp(x)
        K += amp * amp * e
        terms.append((amp, l, p2, r, x, e))
    Kinv = torch.cholesky_inverse(torch.linalg.cholesky(K))
    A = []
    for a in range(no + 2 * nc):
        D = torch.zeros((N, N), **dev)
        for c, (amp, l, p2, r, x, e) in enumerate(terms):
            k = amp * amp * e
            if a < no:
                u = -J[c][ep][:, a] / C_KMS
                D += 2.0 * p2 * k * r * (u[None, :] - u[:, None])
            elif a == no + 2 * c:
                D = 2.0 * amp * e
            elif a == no + 2 * c + 1:
                D = -2.0 * k * x / l
        A.append(Kinv @ D)
    P = len(A)
    F = np.zeros((P, P))
    for a in range(P):
        for b in range(a, P):
            F[a, b] = F[b, a] = 0.5 * float(torch.sum(A[a] * A[b].T))
    return F


@gpu
def test_c4_sized_chunk_against_torch():
    import torch
    from psoap_b200 import synthetic
    ch = small_chunk("SB2", 20, 300, seed=4255, sort=True)
    p = synthetic.default_params("SB2")
    res, _, F = chunk_fisher("SB2", ch, p)
    assert res[3] == 0.0 and len(ch["fl"]) == 6000
    assert_fisher_close(F, _torch_fisher(torch, "SB2", ch, p), 1e-9)


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_exact_properties(model):
    import torch
    from psoap_b200 import synthetic, utils
    from test_gradient import _chunk_grad
    ch = small_chunk(model, 6, 90, seed=31, sort=True)
    p = synthetic.default_params(model)
    res, gp, F = chunk_fisher(model, ch, p)
    assert np.array_equal(F, F.T)
    g = utils.registered_params[model].index("gamma")
    assert np.all(F[g, :] == 0.0) and np.all(F[:, g] == 0.0)
    res2, gp2, F2 = chunk_fisher(model, ch, p)
    assert np.array_equal(F, F2) and np.array_equal(res, res2) and np.array_equal(gp, gp2)
    ref_res, ref_gp = _chunk_grad(torch, model, ch, p)
    assert np.array_equal(res, ref_res) and np.array_equal(gp, ref_gp)


@gpu
def test_fisher_independent_of_rank_count():
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 4, 30 + 7 * i, seed=300 + i) for i in range(9)]
    p = synthetic.default_params("SB2")
    single = ChunkFarm("SB2", chunks)
    ref = single.chunk_fishers(p).cpu().numpy()
    ref_sum = single.fisher(p)
    assert np.array_equal(ref, single.chunk_fishers(p).cpu().numpy())
    for world in (1, 2, 4):
        total = np.zeros_like(ref)
        for r in range(world):
            f = ChunkFarm("SB2", chunks, rank=r, world_size=world)
            f.world_size = 1  # no process group here: take the un-reduced per-chunk tensor
            rows = f.chunk_fishers(p).cpu().numpy()
            for i in range(len(chunks)):
                if i not in f.mine:
                    assert np.all(rows[i] == 0.0)
            total = total + rows
            f.close()
        assert np.array_equal(total, ref)
        assert np.array_equal(np.sum(total, axis=0), ref_sum)
    single.close()


@gpu
def test_k_ranges_and_pixel_order():
    from psoap_b200 import synthetic
    p = synthetic.default_params("SB2")
    unsorted = small_chunk("SB2", 10, 400, seed=41)
    srt = small_chunk("SB2", 10, 400, seed=41, sort=True)
    (_, _, Fu), flags_u, kr_u = chunk_fisher("SB2", unsorted, p, views=True)
    (_, _, Fs), flags_s, kr_s = chunk_fisher("SB2", srt, p, views=True)
    for flags, kr in ((flags_u, kr_u), (flags_s, kr_s)):
        T = flags.shape[0]
        assert np.array_equal(flags, flags.T)
        host = np.array([[np.flatnonzero(flags[:, J]).min(), np.flatnonzero(flags[:, J]).max()] for J in range(T)])
        assert np.array_equal(kr, host)
    # every epoch spans the chunk's wavelengths: epoch-major blocks reach nearly every other block, sorted ones a band
    assert np.sum(kr_s[:, 1] - kr_s[:, 0] + 1) < np.sum(kr_u[:, 1] - kr_u[:, 0] + 1)
    assert_fisher_close(Fs, Fu, 1e-12)


@gpu
def test_minus_inf_gives_nan_fisher():
    from psoap_b200 import synthetic
    ch = small_chunk("SB2", 4, 60, seed=9)
    for k, v in ((7, -0.1), (1, 4e5)):   # a negative amp, |v| >= c
        p = synthetic.default_params("SB2")
        p[k] = v
        res, gp, F = chunk_fisher("SB2", ch, p)
        assert res[0] == -np.inf and np.isnan(gp).all() and np.isnan(F).all()
    # exactly singular K: two pixels at one ln-wavelength, sigma = 0, amp = 0.5
    sing = dict(lwl=np.full(2, np.log(5000.0)), fl=np.array([1.3, 0.7]), sigma=np.zeros(2),
                date1D=np.array([1.0]), epoch=np.zeros(2, dtype=np.int32))
    p = synthetic.default_params("SB1")
    p[6:] = [0.5, 5.0]
    res, gp, F = chunk_fisher("SB1", sing, p)
    assert res[3] == 2.0 and res[0] == -np.inf and np.isnan(gp).all() and np.isnan(F).all()
    # a valid call on a fresh workspace afterwards is finite
    res, gp, F = chunk_fisher("SB2", ch, synthetic.default_params("SB2"))
    assert np.isfinite(F).all()


@gpu
def test_sampler_takes_fisher_jump():
    from psoap_b200 import sample, synthetic, utils
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 5, 60, seed=500 + i) for i in range(2)]
    p = synthetic.default_params("SB2")
    names = utils.registered_params["SB2"]
    pars = dict(zip(names, p))
    fix = ["gamma"]
    config = dict(model="SB2", parameters=pars, fix_params=fix, samples=6, fisher_jump=True,
                  jumps={n: 0.1 for n in names})
    sampler = sample.run(config, chunks, verbose=False)
    farm = ChunkFarm("SB2", chunks)
    expect = sample.fisher_jump(farm.fisher(p), "SB2", fix)
    farm.close()
    assert np.array_equal(sampler.cov, expect)
    assert sampler.flatchain.shape == (6, len(names) - 1) and np.all(np.isfinite(sampler.lnprobability))
