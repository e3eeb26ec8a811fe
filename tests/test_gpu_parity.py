"""GPU parity tests (-m gpu): the CUDA path, called through the package / C ABI, against the golden vectors of
the unmodified reference and against the CPU oracle on seeded inputs.

Tolerances (BASELINE.json north_star): covariance entries 1e-12 relative (+1e-300 absolute floor for entries in
exp's denormal range) on bit-identical ln-wavelength inputs; lnlike 1e-10 relative.
"""
import ctypes
import os
import sys

import numpy as np
import pytest

from conftest import rel_close

pytestmark = pytest.mark.gpu

ENTRY_RTOL, ENTRY_FLOOR = 1e-12, 1e-300
LNLIKE_RTOL = 1e-10
N_ORB = {"SB1": 6, "SB2": 7, "ST1": 11, "ST2": 12, "ST3": 13}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


# ---------------------------------------------------------------------------------------------- fills
def test_fill_golden(golden, torch_cuda):
    from psoap_b200 import matrix_functions as mf
    g = golden["fills"]
    lw, lwp, amp, l = g["lwl"], g["lwl_predict"], g["amp"], g["l"]
    N, M = lw.shape[1], len(lwp)
    m = np.empty((N, N)); mf.fill_V11_f(m, lw[0], amp[0], l[0])
    assert rel_close(m, g["V11_f"], ENTRY_RTOL, ENTRY_FLOOR)
    m = np.empty((N, N)); mf.fill_V11_f_g(m, lw[0], lw[1], amp[0], l[0], amp[1], l[1])
    assert rel_close(m, g["V11_f_g"], ENTRY_RTOL, ENTRY_FLOOR)
    m = np.empty((N, N)); mf.fill_V11_f_g_h(m, lw[0], lw[1], lw[2], amp[0], l[0], amp[1], l[1], amp[2], l[2])
    assert rel_close(m, g["V11_f_g_h"], ENTRY_RTOL, ENTRY_FLOOR)
    assert np.array_equal(m, m.T) and np.array_equal(np.diag(m), np.diag(g["V11_f_g_h"]))
    m = np.empty((N, M)); mf.fill_V12_f(m, lw[0], lwp, amp[0], l[0])
    assert rel_close(m, g["V12_f"], ENTRY_RTOL, ENTRY_FLOOR)
    m = np.empty((33, 33)); mf.fill_V11_f(m, g["far_lwl"], 0.5, 5.0)
    assert rel_close(m, g["far_V11_f"], ENTRY_RTOL, ENTRY_FLOOR)
    # the host-buffer C entry (what a seam at matrix_functions.pyx binds), into a strided host matrix
    from psoap_b200 import _lib
    big = np.full((N, N + 7), -3.0)
    vecs = [np.ascontiguousarray(lw[c]) for c in range(3)]
    _lib.check(_lib.load().psoap_fill_v11_host(3, big.ctypes.data_as(_lib.c_double_p), N + 7, N,
                                               *[v.ctypes.data_as(_lib.c_double_p) for v in vecs],
                                               _lib.dbl_array(amp[:3]), _lib.dbl_array(l[:3])))
    assert rel_close(big[:, :N], g["V11_f_g_h"], ENTRY_RTOL, ENTRY_FLOOR) and (big[:, N:] == -3.0).all()


@pytest.mark.parametrize("N", [1, 63, 64, 65, 257, 1000])
def test_fill_vs_oracle_ragged_sizes(N, oracle, torch_cuda):
    from psoap_b200 import matrix_functions as mf
    rng = np.random.default_rng(N)
    lw = np.log(5100.0) + rng.uniform(0, 500.0, size=(3, N)) / oracle.c_kms
    ref = np.empty((N, N)); oracle.fill_V11_f_g_h(ref, lw[0], lw[1], lw[2], 0.1, 5.0, 0.05, 7.0, 0.03, 6.0)
    got = np.empty((N, N)); mf.fill_V11_f_g_h(got, lw[0], lw[1], lw[2], 0.1, 5.0, 0.05, 7.0, 0.03, 6.0)
    assert rel_close(got, ref, ENTRY_RTOL, ENTRY_FLOOR)
    # device tensor, strided view (ld > N), in place
    big = torch_cuda.full((N + 3, N + 5), -7.0, dtype=torch_cuda.float64, device="cuda")
    mf.fill_V11_f_g(big[:N, :N], lw[0], lw[1], 0.1, 5.0, 0.05, 7.0)
    ref2 = np.empty((N, N)); oracle.fill_V11_f_g(ref2, lw[0], lw[1], 0.1, 5.0, 0.05, 7.0)
    assert rel_close(big[:N, :N].cpu().numpy(), ref2, ENTRY_RTOL, ENTRY_FLOOR)
    assert (big[N:, :] == -7.0).all() and (big[:, N:] == -7.0).all()  # nothing outside the view is touched
    M = max(1, N // 2 + 1)
    lwp = np.log(5100.0) + rng.uniform(0, 500.0, size=M) / oracle.c_kms
    ref3 = np.empty((N, M)); oracle.fill_V12_f(ref3, lw[0], lwp, 0.2, 4.0)
    got3 = np.empty((N, M)); mf.fill_V12_f(got3, lw[0], lwp, 0.2, 4.0)
    assert rel_close(got3, ref3, ENTRY_RTOL, ENTRY_FLOOR)


def test_fill_rejects_wrong_dtype(torch_cuda):
    from psoap_b200 import matrix_functions as mf
    with pytest.raises(ValueError):
        mf.fill_V11_f(np.empty((4, 4), dtype=np.float32), np.zeros(4), 0.1, 5.0)


# ---------------------------------------------------------------------------------------------- orbit / shift
def test_orbit_golden(golden, torch_cuda):
    from psoap_b200 import orbit
    g = golden["orbits"]
    dates = g["dates"]
    for k in [k[:-2] for k in g.files if k.endswith("_p")]:
        model = k.split("_")[0]
        v = orbit.models[model](*g[k + "_p"], dates).get_velocities()
        assert v.shape == g[k + "_v"].shape
        # the reference's fsolve lands within ~3e-13 rad of the Kepler root (SURVEY.md §7)
        assert np.all(np.abs(v - g[k + "_v"]) <= 1e-10 * np.abs(g[k + "_v"]) + 1e-10), k
    o = orbit.SB2(q=0.2, K=5.0, e=0.2, omega=10.0, P=10.0, T0=0.0, gamma=5.0, obs_dates=dates)
    assert np.all(np.abs(o.get_velocities() - g["SB2_0_v"]) <= 1e-10)
    with pytest.raises(AssertionError):
        orbit.SB1(5.0, 1.2, 10.0, 10.0, 0.0, 5.0)


def test_replicate_wls_bit_exact(golden, torch_cuda):
    from psoap_b200 import data
    g = golden["lnlike"]
    for k in range(4):
        pre = f"case{k}_"
        out = data.replicate_wls(g[pre + "lwl"], g[pre + "vel"], g[pre + "mask"])
        assert np.array_equal(out, g[pre + "lwls"])


# ---------------------------------------------------------------------------------------------- lnlike
def test_lnlike_golden(golden, torch_cuda):
    from psoap_b200 import covariance
    g = golden["lnlike"]
    for k in range(4):
        pre = f"case{k}_"
        model = str(g[pre + "model"])
        pg = g[pre + "p"][N_ORB[model]:]
        lwls, fl, sigma = g[pre + "lwls"], g[pre + "fl"], g[pre + "sigma"]
        N = len(fl)
        V11 = np.empty((N, N))
        got = covariance.lnlike[model](V11, *lwls, fl, sigma, *pg)
        assert rel_close(got, g[pre + "lnlike"], LNLIKE_RTOL), (k, got, float(g[pre + "lnlike"]))
        got = covariance.lnlike[model](V11, *lwls, fl, sigma, *pg, mu_GP=0.9)
        assert rel_close(got, g[pre + "lnlike_mu09"], LNLIKE_RTOL)
        pn = pg.copy(); pn[0] = -0.1
        assert covariance.lnlike[model](V11, *lwls, fl, sigma, *pn) == -np.inf
        lw2 = lwls.copy(); lw2[:, 1] = lw2[:, 0]
        assert covariance.lnlike[model](V11, *lw2, fl, np.zeros_like(sigma), *pg) == -np.inf  # not PD
        # C ABI host-buffer entry
        got = covariance.lnlike_host(list(lwls), fl, sigma, pg[0::2], pg[1::2])
        assert rel_close(got, g[pre + "lnlike"], LNLIKE_RTOL)


@pytest.mark.parametrize("model,n_epochs,n_pix,mask_frac", [("SB1", 7, 100, 0.0), ("SB2", 10, 128, 0.0),
                                                            ("SB2", 9, 150, 0.02), ("ST3", 8, 161, 0.05),
                                                            ("SB2", 1, 1, 0.0), ("SB2", 3, 43, 0.0)])
def test_lnlike_vs_oracle(model, n_epochs, n_pix, mask_frac, oracle, torch_cuda):
    from psoap_b200 import covariance, synthetic
    ch = synthetic.make_chunk(model, n_epochs, n_pix, seed=n_pix, mask_frac=mask_frac)
    p = synthetic.default_params(model)
    vel = oracle.get_velocities(model, p[:N_ORB[model]], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    V11 = np.empty((ch["N"], ch["N"]))
    ref = oracle.lnlike[model](V11, *lwls, ch["fl"], ch["sigma"], *p[N_ORB[model]:])
    got = covariance.lnlike[model](None, *lwls, ch["fl"], ch["sigma"], *p[N_ORB[model]:])
    assert rel_close(got, ref, LNLIKE_RTOL), (got, ref)
    # device-resident inputs give the same value
    t = torch_cuda
    got_dev = covariance.lnlike[model](None, *[t.from_numpy(x).cuda() for x in lwls], t.from_numpy(ch["fl"]).cuda(),
                                       t.from_numpy(ch["sigma"]).cuda(), *p[N_ORB[model]:])
    assert got_dev == got


def test_lnlike_empty_chunk(oracle, torch_cuda):
    """A chunk whose mask removes every pixel: the reference returns -0.0 (fill, factorisation and sums over nothing),
    -inf if a hyper-parameter is negative; so do the Python mirror and both C entry points."""
    from psoap_b200 import _lib, covariance
    e = np.empty(0)
    ref = oracle.lnlike_f_g(np.empty((0, 0)), e, e, e, e, 0.1, 5.0, 0.05, 7.0)
    got = covariance.lnlike_f_g(None, e, e, e, e, 0.1, 5.0, 0.05, 7.0)
    assert got == ref == 0.0 and np.signbit(got) and np.signbit(ref)
    assert covariance.lnlike_f_g(None, e, e, e, e, -0.1, 5.0, 0.05, 7.0) == -np.inf
    lib = _lib.load()
    res = _lib.PsoapResult()
    amp, l = _lib.dbl_array([0.1, 0.05]), _lib.dbl_array([5.0, 7.0])
    _lib.check(lib.psoap_lnlike_host(2, 0, None, None, None, None, None, amp, l, 1.0, ctypes.byref(res)))
    assert res.lnlike == 0.0 and np.signbit(res.lnlike) and res.info == 0.0
    dres = torch_cuda.full((4,), 7.0, dtype=torch_cuda.float64, device="cuda")
    _lib.check(lib.psoap_lnlike(2, 0, None, None, None, None, None, amp, l, 1.0, None, 0, _lib.ptr(dres), _lib.stream_ptr()))
    torch_cuda.cuda.synchronize()
    out = dres.cpu().numpy()
    assert out[0] == 0.0 and np.signbit(out[0]) and not out[1:].any()


@pytest.mark.parametrize("n_pix", [127, 128, 129, 255, 256, 257, 383, 384, 385, 511, 513, 640, 897])
def test_lnlike_tile_boundaries(n_pix, oracle, torch_cuda):
    """Sizes around the 128-row tile / 2- and 4-panel group boundaries (front padding, partial groups)."""
    from psoap_b200 import covariance, synthetic
    ch = synthetic.make_chunk("SB2", 1, n_pix, seed=n_pix, dv_pix=1.4)
    p = synthetic.default_params("SB2")
    vel = oracle.get_velocities("SB2", p[:7], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    V11 = np.empty((ch["N"], ch["N"]))
    ref = oracle.lnlike_f_g(V11, lwls[0], lwls[1], ch["fl"], ch["sigma"], *p[7:])
    got = covariance.lnlike_f_g(None, lwls[0], lwls[1], ch["fl"], ch["sigma"], *p[7:])
    assert rel_close(got, ref, LNLIKE_RTOL), (n_pix, got, ref)


def test_lnlike_materialize_v11(oracle, torch_cuda):
    from psoap_b200 import covariance, synthetic
    ch = synthetic.make_chunk("SB2", 4, 50, seed=3)
    p = synthetic.default_params("SB2")
    vel = oracle.get_velocities("SB2", p[:7], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    V11 = np.empty((ch["N"], ch["N"]))
    covariance.MATERIALIZE_V11 = True
    try:
        covariance.lnlike_f_g(V11, lwls[0], lwls[1], ch["fl"], ch["sigma"], *p[7:])
    finally:
        covariance.MATERIALIZE_V11 = False
    ref = np.empty_like(V11); oracle.fill_V11_f_g(ref, lwls[0], lwls[1], *p[7:])
    ref[np.diag_indices_from(ref)] += ch["sigma"] ** 2
    assert rel_close(V11, ref, ENTRY_RTOL, ENTRY_FLOOR)


# ---------------------------------------------------------------------------------------------- predict
def test_predict_golden(golden, torch_cuda):
    from psoap_b200 import covariance
    g = golden["predict"]
    lwls, fl, sigma, lwp, amp, l = g["lwls"], g["fl"], g["sigma"], g["lwl_predict"], g["amp"], g["l"]

    def close(mu, Sig, kmu, kS):
        scale = np.abs(g[kS]).max()
        assert np.all(np.abs(mu - g[kmu]) <= 1e-9 * np.maximum(1.0, np.abs(g[kmu]))), kmu
        assert np.all(np.abs(Sig - g[kS]) <= 1e-9 * scale), kS
        assert np.array_equal(Sig, Sig.T)

    mu, Sig = covariance.predict_f_g(lwls[0], lwls[1], fl, sigma, lwp[0], lwp[1], 0.7, amp[0], l[0], 0.3, amp[1], l[1])
    close(mu, Sig, "fg_mu", "fg_Sigma")
    mu = covariance.predict_f_g(lwls[0], lwls[1], fl, sigma, lwp[0], lwp[1], 0.7, amp[0], l[0], 0.3, amp[1], l[1],
                                get_Sigma=False)
    assert np.all(np.abs(mu - g["fg_mu_only"]) <= 1e-9)
    mu, Sig = covariance.predict_f_g_sum(lwls[0], lwls[1], fl, sigma, lwp[0], lwp[1], 1.0, amp[0], l[0], amp[1], l[1])
    close(mu, Sig, "fgsum_mu", "fgsum_Sigma")
    mu, Sig = covariance.predict_f_g_h(lwls[0], lwls[1], lwls[2], fl, sigma, lwp[0], lwp[1], lwp[2], 0.5, 0.3, 0.2,
                                       amp[0], l[0], amp[1], l[1], amp[2], l[2])
    close(mu, Sig, "fgh_mu", "fgh_Sigma")
    mu, Sig = covariance.predict_f_g_h_sum(lwls[0], lwls[1], lwls[2], fl, sigma, lwls[0], lwls[1], lwls[2], 1.0,
                                           amp[0], l[0], amp[1], l[1], amp[2], l[2])
    close(mu, Sig, "fghsum_mu", "fghsum_Sigma")
    with pytest.raises(ValueError):  # covariance.py:294: V12.T only conforms when M == N
        covariance.predict_f_g_h_sum(lwls[0], lwls[1], lwls[2], fl, sigma, lwp[0], lwp[1], lwp[2], 1.0, amp[0], l[0],
                                     amp[1], l[1], amp[2], l[2])


def test_predict_f_vs_oracle(oracle, torch_cuda):
    from psoap_b200 import covariance, synthetic
    ch = synthetic.make_chunk("SB1", 3, 90, seed=9)
    grid = np.linspace(ch["lwl"].min(), ch["lwl"].max(), 140)
    mu_r, S_r = oracle.predict_f(ch["lwl"], ch["fl"], ch["sigma"], grid, 0.1, 5.0, mu_GP=1.0)
    mu, S = covariance.predict_f(ch["lwl"], ch["fl"], ch["sigma"], grid, 0.1, 5.0, mu_GP=1.0)
    assert np.all(np.abs(mu - mu_r) <= 1e-9) and np.all(np.abs(S - S_r) <= 1e-9 * np.abs(S_r).max())


@pytest.mark.parametrize("n_epochs,n_pix,m", [(30, 300, 600), (8, 250, 2000)], ids=["retrieve-n9000-m600", "predict-n2000-m2000"])
def test_predict_at_script_sizes(n_epochs, n_pix, m, oracle, torch_cuda):
    """predict_f_g at the sizes the reference's scripts use: psoap_retrieve_SB2.py:76-105 predicts each component on
    a 2 x n_pix grid from all N = n_epochs x n_pix pixels (here N = 9000, 600 points per component: C is 1200 x 9000),
    psoap_predict_SB2.py:75 predicts on as many points as there are data (n = m = 2000, Sigma is 4000 x 4000).
    Tolerance: 1e-9 of the largest entry for Sigma, 1e-9 for the mean (the data are of order one)."""
    from psoap_b200 import covariance, synthetic
    ch = synthetic.make_chunk("SB2", n_epochs, n_pix, seed=31 + m)
    p = synthetic.default_params("SB2")
    vel = oracle.get_velocities("SB2", p[:7], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    lo, hi = ch["lwl"].min() - 30.0 / oracle.c_kms, ch["lwl"].max() + 30.0 / oracle.c_kms
    grid_f, grid_g = np.linspace(lo, hi, m), np.linspace(lo, hi, m) + 0.3 * (hi - lo) / m
    args = (lwls[0], lwls[1], ch["fl"], ch["sigma"], grid_f, grid_g, 0.8, p[7], p[8], 0.2, p[9], p[10])
    mu_r, S_r = oracle.predict_f_g(*args)
    mu, S = covariance.predict_f_g(*args)
    assert mu.shape == (2 * m,) and S.shape == (2 * m, 2 * m)
    assert np.all(np.abs(mu - mu_r) <= 1e-9 * np.maximum(1.0, np.abs(mu_r))), np.abs(mu - mu_r).max()
    assert np.all(np.abs(S - S_r) <= 1e-9 * np.abs(S_r).max()), np.abs(S - S_r).max()
    assert np.array_equal(S, S.T)
    mu_only = covariance.predict_f_g(*args, get_Sigma=False)
    assert np.array_equal(mu_only, mu)


def test_predict_host_entry(oracle, torch_cuda):
    """psoap_predict_host: host arrays in, host arrays out, no Python glue between fill, elimination and read-out;
    the three modes against the oracle's predict_f_g_h / predict_f_g_sum / predict_f_g_h_sum."""
    from psoap_b200 import _lib, synthetic
    lib = _lib.load()
    ch = synthetic.make_chunk("ST3", 5, 60, seed=8)
    p = synthetic.default_params("ST3")
    vel = oracle.get_velocities("ST3", p[:13], ch["date1D"])
    lwls = [np.ascontiguousarray(x) for x in oracle.replicate_wls(ch["lwl"], vel, ch["mask"])]
    n = ch["N"]
    amps, ls = p[13::2], p[14::2]

    def call(ncomp, mode, grids, resid_mu, nugget):
        m = len(grids[0])
        M = ncomp * m if mode == 0 else m
        dp = (_lib.c_double_p * ncomp)(*[x.ctypes.data_as(_lib.c_double_p) for x in lwls[:ncomp]])
        pp = (_lib.c_double_p * ncomp)(*[g.ctypes.data_as(_lib.c_double_p) for g in grids[:ncomp]])
        delta, Sig, res = np.empty(M), np.empty((M, M)), _lib.PsoapResult()
        _lib.check(lib.psoap_predict_host(ncomp, mode, n, m, dp, ch["fl"].ctypes.data_as(_lib.c_double_p),
                                          ch["sigma"].ctypes.data_as(_lib.c_double_p), pp, _lib.dbl_array(amps[:ncomp]),
                                          _lib.dbl_array(ls[:ncomp]), resid_mu, nugget,
                                          delta.ctypes.data_as(_lib.c_double_p), Sig.ctypes.data_as(_lib.c_double_p),
                                          ctypes.byref(res)))
        assert res.info == 0.0
        return delta, Sig

    def close(a, b):
        return np.all(np.abs(a - b) <= 1e-9 * max(1.0, np.abs(b).max()))

    grids = [np.ascontiguousarray(np.linspace(x.min(), x.max(), 77)) for x in lwls]
    mu_r, S_r = oracle.predict_f_g_h(*lwls, ch["fl"], ch["sigma"], *grids, 0.5, 0.3, 0.2, *p[13:])
    delta, Sig = call(3, 0, grids, 1.0, 0.0)
    assert close(np.concatenate([np.full(77, v) for v in (0.5, 0.3, 0.2)]) + delta, mu_r) and close(Sig, S_r)
    mu_r, S_r = oracle.predict_f_g_sum(lwls[0], lwls[1], ch["fl"], ch["sigma"], grids[0], grids[1], 1.0, *p[13:17])
    delta, Sig = call(2, 1, grids, 1.0, 1e-8)
    assert close(1.0 + delta, mu_r) and close(Sig, S_r)
    mu_r, S_r = oracle.predict_f_g_h_sum(*lwls, ch["fl"], ch["sigma"], *lwls, 1.0, *p[13:])   # M == N quirk (covariance.py:294)
    delta, _ = call(3, 2, lwls, 1.0, 0.0)
    _, Sig = call(3, 1, lwls, 1.0, 0.0)
    assert close(1.0 + delta, mu_r) and close(Sig, S_r)


# ---------------------------------------------------------------------------------------------- farm
def test_farm_vs_oracle(oracle, torch_cuda):
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    specs = [(5, 60, 0.0), (6, 45, 0.03), (4, 128, 0.0), (7, 33, 0.1), (5, 77, 0.0), (3, 20, 0.0), (6, 64, 0.0)]
    for model in ("SB2", "ST3", "SB1"):
        chunks = [synthetic.make_chunk(model, ne, npx, seed=100 + i, mask_frac=mf, wl0=5000.0 + 3 * i)
                  for i, (ne, npx, mf) in enumerate(specs)]
        p = synthetic.default_params(model)
        farm = ChunkFarm(model, chunks, nbranch=3)
        total_ref, per_ref = oracle.farm_lnprob(model, p, chunks)
        lnl = farm.chunk_lnlikes(p).cpu().numpy()
        assert rel_close(lnl, per_ref, LNLIKE_RTOL), (model, lnl, per_ref)
        assert rel_close(farm.lnprob(p), total_ref, LNLIKE_RTOL)
        # second proposal through the same graph
        p2 = p.copy(); p2[1 if model != "SB1" else 0] *= 1.3; p2[-1] *= 0.9
        total_ref2, _ = oracle.farm_lnprob(model, p2, chunks)
        assert rel_close(farm.lnprob(p2), total_ref2, LNLIKE_RTOL)
        # sentinels: |v| >= c (sample_parallel.py:186-187) and negative hyper-parameters -> -inf
        p3 = p.copy(); p3[1 if model != "SB1" else 0] = 4e5
        assert farm.lnprob(p3) == -np.inf and oracle.farm_lnprob(model, p3, chunks)[0] == -np.inf
        p4 = p.copy(); p4[-2] = -0.01
        assert farm.lnprob(p4) == -np.inf
        assert rel_close(farm.lnprob(p), total_ref, LNLIKE_RTOL)  # and the farm recovers afterwards
        farm.close()


def test_farm_skips_empty_chunk(oracle, torch_cuda):
    """A fully masked chunk adds -0.0 in the reference; the farm gives the same total with or without it."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 4, 50, seed=21 + i) for i in range(3)]
    empty = dict(chunks[0], lwl=np.empty(0), fl=np.empty(0), sigma=np.empty(0),
                 mask=np.zeros_like(chunks[0]["mask"], dtype=bool))
    p = synthetic.default_params("SB2")
    full = ChunkFarm("SB2", chunks).lnprob(p)
    with_empty = ChunkFarm("SB2", chunks[:1] + [empty] + chunks[1:])
    assert with_empty.lnprob(p) == full
    per_chunk = with_empty.chunk_lnlikes(p).cpu().numpy()
    assert per_chunk.shape == (4,) and per_chunk[1] == 0.0 and np.all(per_chunk[[0, 2, 3]] != 0.0)
    assert rel_close(full, oracle.farm_lnprob("SB2", p, chunks)[0], LNLIKE_RTOL)


def test_farm_direct_mode_large_chunk(oracle, torch_cuda):
    """A one-chunk farm with N >= 7000 issues its pipeline directly instead of replaying the graph (api.cu
    psoap_farm.direct); the value must be the one the operator surface gives for the same chunk, call after call."""
    from psoap_b200 import covariance, synthetic
    from psoap_b200.farm import ChunkFarm
    ch = synthetic.make_chunk("SB2", 22, 320, seed=4)          # N = 7040
    p = synthetic.default_params("SB2")
    farm = ChunkFarm("SB2", [ch])
    got = [farm.lnprob(p) for _ in range(3)]
    assert got[0] == got[1] == got[2]
    vel = oracle.get_velocities("SB2", p[:7], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    ref = covariance.lnlike_f_g(None, lwls[0], lwls[1], ch["fl"], ch["sigma"], *p[7:])
    assert rel_close(got[0], ref, LNLIKE_RTOL), (got[0], ref)
    p2 = p.copy(); p2[1] *= 1.1                                 # another proposal through the same farm
    vel2 = oracle.get_velocities("SB2", p2[:7], ch["date1D"])
    lw2 = oracle.replicate_wls(ch["lwl"], vel2, ch["mask"])
    assert rel_close(farm.lnprob(p2), covariance.lnlike_f_g(None, lw2[0], lw2[1], ch["fl"], ch["sigma"], *p2[7:]), LNLIKE_RTOL)


def test_farm_partition_matches_single(oracle, torch_cuda):
    """Emulated ranks on one GPU: the per-rank vectors (zero outside own chunks) sum to the single-rank answer."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm, combine_chunk_lnlikes
    chunks = [synthetic.make_chunk("SB2", 4, 30 + 7 * i, seed=300 + i) for i in range(9)]
    p = synthetic.default_params("SB2")
    single = ChunkFarm("SB2", chunks)
    ref_vec = single.chunk_lnlikes(p).cpu().numpy().copy()
    vecs = []
    for r in range(4):
        f = ChunkFarm("SB2", chunks, rank=r, world_size=4)
        f.world_size = 1  # no process group here: take the un-reduced vector
        vecs.append(f.chunk_lnlikes(p).cpu().numpy().copy())
        f.close()
    total, vec = combine_chunk_lnlikes(vecs)
    assert np.array_equal(vec, ref_vec)
    assert total == float(np.sum(ref_vec))
    single.close()


# ---------------------------------------------------------------------------------------------- full size
def _torch_reference_lnlike(torch, lwls, fl, sigma, pg, mu=1.0):
    """Independent full-size check: our operator-surface fill + cuSOLVER Cholesky through torch."""
    from psoap_b200 import matrix_functions as mf
    N = len(fl)
    K = torch.empty((N, N), dtype=torch.float64, device="cuda")
    fills = {1: mf.fill_V11_f, 2: mf.fill_V11_f_g, 3: mf.fill_V11_f_g_h}
    fills[len(lwls)](K, *lwls, *pg)
    K.diagonal().add_(torch.from_numpy(sigma).cuda() ** 2)
    L = torch.linalg.cholesky(K)
    r = (torch.from_numpy(fl).cuda() - mu)[:, None]
    y = torch.linalg.solve_triangular(L, r, upper=False)
    logdet = 2.0 * torch.log(torch.diagonal(L)).sum()
    return float(-0.5 * ((y * y).sum() + logdet))


@pytest.mark.parametrize("cfg", ["C1", "C2", "C3"])
def test_full_size_configs(cfg, oracle, torch_cuda):
    """BASELINE.json configs at full size: agreement with an independent GPU factorisation (cuSOLVER via torch)
    and invariance under a random permutation of the pixels (a different elimination order)."""
    from psoap_b200 import covariance, synthetic
    model, chunks = synthetic.config_chunks(cfg)
    ch = chunks[0]
    p = synthetic.default_params(model)
    vel = oracle.get_velocities(model, p[:N_ORB[model]], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    pg = p[N_ORB[model]:]
    got = covariance.lnlike[model](None, *lwls, ch["fl"], ch["sigma"], *pg)
    ref = _torch_reference_lnlike(torch_cuda, list(lwls), ch["fl"], ch["sigma"], pg)
    assert np.isfinite(got) and rel_close(got, ref, LNLIKE_RTOL), (got, ref)
    perm = np.random.default_rng(1).permutation(ch["N"])
    got_p = covariance.lnlike[model](None, *[x[perm] for x in lwls], ch["fl"][perm], ch["sigma"][perm], *pg)
    assert rel_close(got_p, got, LNLIKE_RTOL), (got_p, got)


def _reference_cpu_lnprob(oracle, model, p, ch):
    """The reference's CPU path for one chunk (sample_parallel.py:168-198): fsolve orbits, numpy Doppler shift, the
    reference's own compiled Cython fill when oracle/_ref holds it (C restatement otherwise), scipy cho_factor/solve."""
    return oracle.chunk_lnprob(model, p, ch, use_ref_fill=True)


@pytest.mark.parametrize("cfg", ["C1", "C2", "C3"])
def test_full_size_vs_reference_cpu(cfg, oracle, torch_cuda):
    """BASELINE.json configs C1-C3 at FULL size against the reference CPU path (matrix_functions.pyx fill +
    scipy LAPACK, covariance.py:299-376), through the operator surface and through the ChunkFarm (device orbit
    solve + fused Doppler shift): 1e-10 relative on lnlike."""
    from psoap_b200 import covariance, synthetic
    from psoap_b200.farm import ChunkFarm
    model, chunks = synthetic.config_chunks(cfg)
    ch = chunks[0]
    p = synthetic.default_params(model)
    ref = _reference_cpu_lnprob(oracle, model, p, ch)
    vel = oracle.get_velocities(model, p[:N_ORB[model]], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    got = covariance.lnlike[model](None, *lwls, ch["fl"], ch["sigma"], *p[N_ORB[model]:])
    assert np.isfinite(ref) and rel_close(got, ref, LNLIKE_RTOL), (cfg, got, ref)
    farm = ChunkFarm(model, chunks)
    got_farm = farm.lnprob(p)
    farm.close()
    assert rel_close(got_farm, ref, LNLIKE_RTOL), (cfg, got_farm, ref)


def test_c4_chunks_vs_reference_cpu(oracle, torch_cuda):
    """Four chunks of the bench workload C4 (N = 2000, 3320, 4660, 6000: the smallest, two interior and the largest)
    through the ChunkFarm against the reference CPU path, per chunk."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    model, chunks = synthetic.config_chunks("C4")
    pick = [chunks[i] for i in (0, 85, 170, 255)]
    assert [c["N"] for c in pick] == [2000, 3320, 4660, 6000]
    p = synthetic.default_params(model)
    farm = ChunkFarm(model, pick, nbranch=4)
    got = farm.chunk_lnlikes(p).cpu().numpy().copy()
    farm.close()
    ref = np.array([_reference_cpu_lnprob(oracle, model, p, c) for c in pick])
    assert rel_close(got, ref, LNLIKE_RTOL), (got, ref)


def test_package_default_hyperparameters_large(oracle, torch_cuda):
    """amp = 0.5, l = 5 km/s for every component (the package defaults, psoap/data/config.SB2.yaml:29-32): a
    signal-to-noise (amp/sigma)^2 some 25-100x above the other tests', i.e. the worst conditioning the explicit
    inverse of the 128 x 128 diagonal blocks sees.  N = 4000 (SB2) and N = 4200 (ST3) against the reference CPU path."""
    from psoap_b200 import covariance, synthetic
    for model, ne, npx in (("SB2", 20, 200), ("ST3", 20, 210)):
        ch = synthetic.make_chunk(model, ne, npx, seed=77)
        p = synthetic.default_params(model)
        p[N_ORB[model]:] = [0.5, 5.0] * synthetic.NCOMP[model]
        ref = _reference_cpu_lnprob(oracle, model, p, ch)
        vel = oracle.get_velocities(model, p[:N_ORB[model]], ch["date1D"])
        lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
        got = covariance.lnlike[model](None, *lwls, ch["fl"], ch["sigma"], *p[N_ORB[model]:])
        assert np.isfinite(ref) and rel_close(got, ref, LNLIKE_RTOL), (model, got, ref)


@pytest.mark.parametrize("model,n_epochs,n_pix,mask_frac", [("SB1", 3, 100, 0.0), ("SB2", 5, 200, 0.01),
                                                            ("ST3", 7, 184, 0.0), ("SB2", 20, 128, 0.0),
                                                            ("SB2", 1, 5, 0.0)])
def test_fill_lower_entrywise_vs_reference(model, n_epochs, n_pix, mask_frac, oracle, torch_cuda):
    """The fill the likelihood ACTUALLY uses (fill_lower_kernel: lower triangle, front padding, interior-tile fast
    path, Doppler shift fused from the base ln-wavelengths + epoch index + velocity table) entry by entry against
    matrix_functions.pyx:125-144 on data.py:40-63's shifted vectors plus covariance.py:322's sigma^2 diagonal:
    |delta| <= 1e-12 |ref| + 1e-300.  Covers pad != 0 (N = 300, 995, 1288, 5) and pad == 0 (N = 2560)."""
    from psoap_b200 import _lib, synthetic
    t = torch_cuda
    lib = _lib.load()
    ch = synthetic.make_chunk(model, n_epochs, n_pix, seed=n_pix + n_epochs, mask_frac=mask_frac)
    N, ncomp = ch["N"], synthetic.NCOMP[model]
    p = synthetic.default_params(model)
    vel = oracle.get_velocities(model, p[:N_ORB[model]], ch["date1D"])
    lwls = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
    pg = p[N_ORB[model]:]
    ref = np.empty((N, N))
    mf = oracle.ref_matrix_functions() or oracle
    {1: mf.fill_V11_f, 2: mf.fill_V11_f_g, 3: mf.fill_V11_f_g_h}[ncomp](ref, *lwls, *pg)
    ref[np.diag_indices_from(ref)] += ch["sigma"] ** 2
    Np = (N + 127) // 128 * 128
    pad = Np - N
    amp, l = _lib.dbl_array(pg[0::2]), _lib.dbl_array(pg[1::2])
    fl, sg = t.from_numpy(ch["fl"]).cuda(), t.from_numpy(ch["sigma"]).cuda()
    for fused in (True, False):
        W = t.full((Np, Np), -7.0, dtype=t.float64, device="cuda")     # column-major: W[c, r] is entry (r, c)
        rvec = t.full((Np,), -7.0, dtype=t.float64, device="cuda")
        if fused:
            lw = [t.from_numpy(ch["lwl"]).cuda(), None, None]
            ep, vd = t.from_numpy(ch["epoch"]).cuda(), t.from_numpy(np.ascontiguousarray(vel)).cuda()
        else:
            lw = [t.from_numpy(np.ascontiguousarray(x)).cuda() for x in lwls] + [None] * (3 - ncomp)
            ep, vd = None, None
        _lib.check(lib.psoap_debug_fill_lower(ncomp, N, _lib.ptr(lw[0]), _lib.ptr(lw[1]), _lib.ptr(lw[2]), _lib.ptr(ep),
                                              _lib.ptr(vd), len(ch["date1D"]), _lib.ptr(fl), _lib.ptr(sg), amp, l, 0.9,
                                              _lib.ptr(W), Np, _lib.ptr(rvec), _lib.stream_ptr()))
        M = W.cpu().numpy().T                                           # M[r, c] = entry (r, c)
        low = np.tril_indices(N)
        got = M[pad:, pad:]
        assert rel_close(got[low], ref[low], ENTRY_RTOL, ENTRY_FLOOR), (fused, np.abs(got[low] - ref[low]).max())
        # identity in the front padding, nothing written above the diagonal
        P = M[:, :pad]
        assert np.array_equal(np.tril(P), np.tril(np.eye(Np)[:, :pad]))
        assert np.array_equal(np.tril(M[:pad, :]), np.tril(np.eye(Np)[:pad, :]))
        # tiles strictly above the diagonal are never touched; diagonal tiles are written whole (both halves agree)
        blk = np.arange(Np) // 128
        assert (M[blk[:, None] < blk[None, :]] == -7.0).all()
        for k in range(Np // 128):
            D = M[128 * k:128 * (k + 1), 128 * k:128 * (k + 1)]
            assert np.array_equal(D, D.T)
        r = rvec.cpu().numpy()
        assert np.array_equal(r[pad:], ch["fl"] - 0.9) and not r[:pad].any()


def test_block_additivity(oracle, torch_cuda):
    """Two pixel sets far apart in wavelength have exactly zero cross-covariance (exp underflow), so the joint
    log-likelihood is the sum of the parts."""
    from psoap_b200 import covariance, synthetic
    a = synthetic.make_chunk("SB2", 6, 200, seed=21, wl0=5000.0)
    b = synthetic.make_chunk("SB2", 5, 333, seed=22, wl0=5400.0)
    p = synthetic.default_params("SB2")
    parts, lw_all = [], []
    for ch in (a, b):
        vel = oracle.get_velocities("SB2", p[:7], ch["date1D"])
        lw = oracle.replicate_wls(ch["lwl"], vel, ch["mask"])
        lw_all.append(lw)
        parts.append(covariance.lnlike_f_g(None, lw[0], lw[1], ch["fl"], ch["sigma"], *p[7:]))
    lw = np.concatenate(lw_all, axis=1)
    joint = covariance.lnlike_f_g(None, lw[0], lw[1], np.concatenate([a["fl"], b["fl"]]),
                                  np.concatenate([a["sigma"], b["sigma"]]), *p[7:])
    assert rel_close(joint, parts[0] + parts[1], LNLIKE_RTOL)


def test_repeatable_bits(oracle, torch_cuda):
    """The same evaluation repeated gives the same bits (the TMA/mbarrier pipeline once raced here, DESIGN.md §4),
    with and without an intervening synchronisation, and through the farm graph."""
    from psoap_b200 import covariance, synthetic
    from psoap_b200.farm import ChunkFarm
    ch = synthetic.make_chunk("SB2", 20, 300, seed=1)  # N = 6000: several tiles per persistent CTA
    p = synthetic.default_params("SB2")
    vel = synthetic.host_velocities("SB2", p[:7], ch["date1D"])
    t = torch_cuda
    lw = [t.from_numpy(ch["lwl"] - vel[c][ch["epoch"]] / synthetic.c_kms).cuda() for c in range(2)]
    fl, sg = t.from_numpy(ch["fl"]).cuda(), t.from_numpy(ch["sigma"]).cuda()
    vals = {covariance.lnlike_f_g(None, lw[0], lw[1], fl, sg, *p[7:]) for _ in range(6)}
    assert len(vals) == 1, vals
    farm = ChunkFarm("SB2", [ch, synthetic.make_chunk("SB2", 20, 150, seed=2)])
    fv = {farm.lnprob(p) for _ in range(4)}
    assert len(fv) == 1, fv
    farm.close()


def test_c5_large_single_chunk(torch_cuda):
    """BASELINE config C5 (N = 32768, 8.6 GB matrix) through size-independent properties: the data are laid out as
    two far-apart halves (exactly zero cross-covariance), so the joint log-likelihood must equal the sum of the
    halves, each of which is small enough to be cross-checked against cuSOLVER."""
    from psoap_b200 import covariance, synthetic
    p = synthetic.default_params("SB2")
    halves, lws = [], []
    for k, wl0 in enumerate((5000.0, 5600.0)):
        ch = synthetic.make_chunk("SB2", 32, 512, seed=50 + k, wl0=wl0)  # 16384 pixels each
        vel = synthetic.host_velocities("SB2", p[:7], ch["date1D"])
        lw = np.stack([ch["lwl"] - vel[c][ch["epoch"]] / synthetic.c_kms for c in range(2)])
        halves.append((ch, lw))
        lws.append(lw)
    parts = [covariance.lnlike_f_g(None, lw[0], lw[1], ch["fl"], ch["sigma"], *p[7:]) for ch, lw in halves]
    ref0 = _torch_reference_lnlike(torch_cuda, list(halves[0][1]), halves[0][0]["fl"], halves[0][0]["sigma"], p[7:])
    assert rel_close(parts[0], ref0, LNLIKE_RTOL), (parts[0], ref0)
    lw = np.concatenate(lws, axis=1)
    fl = np.concatenate([h[0]["fl"] for h in halves])
    sg = np.concatenate([h[0]["sigma"] for h in halves])
    assert lw.shape[1] == 32768
    torch_cuda.cuda.empty_cache()
    joint = covariance.lnlike_f_g(None, lw[0], lw[1], fl, sg, *p[7:])
    assert np.isfinite(joint) and rel_close(joint, parts[0] + parts[1], LNLIKE_RTOL), (joint, parts)


def test_sampler_chain_matches_oracle_at_visited_points(oracle, torch_cuda, tmp_path):
    """psoap_b200.sample.run (the psoap-sample-parallel replacement): every stored lnprob is the oracle's farm
    log-likelihood at the stored chain position; outputs are written like sample_parallel.py:442-443."""
    from psoap_b200 import sample, synthetic, utils
    chunks = [synthetic.make_chunk("SB2", 5, 40 + 9 * i, seed=700 + i, mask_frac=0.02 * i) for i in range(3)]
    names = utils.registered_params["SB2"]
    pars = dict(zip(names, synthetic.default_params("SB2")))
    jumps = dict(q=0.002, K=0.02, e=0.002, omega=0.05, P=0.001, T0=0.001, gamma=0.01, amp_f=0.002, l_f=0.05,
                 amp_g=0.002, l_g=0.05)
    config = dict(model="SB2", parameters=pars, jumps=jumps, fix_params=["gamma"], samples=12, soften=1.0,
                  outdir=str(tmp_path), opt_jump="does-not-exist.npy")
    s = sample.run(config, chunks, run_index=3, seed=5, verbose=False)
    assert s.flatchain.shape == (12, 10) and s.lnprobability.shape == (12,)
    assert np.array_equal(np.load(tmp_path / "run03" / "flatchain.npy"), s.flatchain)
    assert np.array_equal(np.load(tmp_path / "run03" / "lnprob.npy"), s.lnprobability)
    for i in (0, 5, 11):
        p_orb, p_GP = utils.convert_vector(s.flatchain[i], "SB2", ["gamma"], **pars)
        ref, _ = oracle.farm_lnprob("SB2", np.concatenate([p_orb, p_GP]), chunks)
        assert rel_close(s.lnprobability[i], ref, LNLIKE_RTOL), (i, s.lnprobability[i], ref)
    assert s.naccepted >= 1


def test_calibration_golden(golden, oracle, torch_cuda):
    """covariance.optimize_calibration / _static (covariance.py:560-711) through two device Schur complements."""
    from psoap_b200 import covariance
    g = golden["calibration"]
    amp, l = float(g["amp"]), float(g["l"])
    args = (float(g["lwl0"]), float(g["lwl1"]), g["lwl_cal"], g["fl_cal"], g["sigma_cal"], g["lwl_fixed"], g["fl_fixed"],
            g["sigma_fixed"], amp, l)
    for order in (1, 2):
        fl_cor, X = covariance.optimize_calibration_static(*args, order=order, mu_GP=1.0)
        assert rel_close(X, g[f"static_o{order}_X"], 1e-7, 1e-10), (X, g[f"static_o{order}_X"])
        assert rel_close(fl_cor, g[f"static_o{order}_fl"], 1e-8)
    n_cal, n_fix = len(g["lwl_cal"]), len(g["lwl_fixed"])
    A = np.empty((n_cal, n_cal)); oracle.fill_V11_f(A, g["lwl_cal"], amp, l); A[np.diag_indices_from(A)] += g["sigma_cal"] ** 2
    B = np.empty((n_fix, n_fix)); oracle.fill_V11_f(B, g["lwl_fixed"], amp, l); B[np.diag_indices_from(B)] += g["sigma_fixed"] ** 2
    C = np.empty((n_cal, n_fix)); oracle.fill_V12_f(C, g["lwl_cal"], g["lwl_fixed"], amp, l)
    fl_cor, X = covariance.optimize_calibration(float(g["lwl0"]), float(g["lwl1"]), g["lwl_cal"], g["fl_cal"],
                                                g["fl_fixed"], A, B, C, order=1, mu_GP=1.0)
    assert rel_close(X, g["general_X"], 1e-7, 1e-10) and rel_close(fl_cor, g["general_fl"], 1e-8)
    # Nelder-Mead hyper-parameter fit (covariance.py:408-424): same optimum as the reference's
    lw2, fl2, sg2 = g["lwl_fixed"][:60], g["fl_fixed"][:60], g["sigma_fixed"][:60]
    fit = covariance.optimize_GP_f(lw2, fl2, sg2, 0.2, 8.0)
    assert np.all(np.abs(fit - g["gp_fit"]) <= 1e-3 * np.abs(g["gp_fit"])), (fit, g["gp_fit"])
    # the cycle driver (covariance.py:714-748, with the evident call) against the same loop over the oracle
    wl = np.stack([g["lwl_cal"]] + [g["lwl_fixed"][60 * k:60 * (k + 1)] for k in range(3)])
    fl = np.stack([g["fl_cal"]] + [g["fl_fixed"][60 * k:60 * (k + 1)] for k in range(3)])
    sg = np.stack([g["sigma_cal"]] + [g["sigma_fixed"][60 * k:60 * (k + 1)] for k in range(3)])
    out = covariance.cycle_calibration(wl, fl, sg, amp, l, 1, order=1)
    ref = np.copy(fl)
    for i in range(4):
        rem = lambda a: np.delete(a, i, axis=0)[0:3].flatten()
        ref[i], _ = oracle.optimize_calibration_static(wl.min(), wl.max(), wl[i], ref[i], sg[i], rem(wl), rem(ref),
                                                       rem(sg), amp, l, order=1, mu_GP=1.0)
    assert out.shape == fl.shape and rel_close(out, ref, 1e-7)


def test_farm_many_proposals(oracle, torch_cuda):
    """Ensemble evaluation: K proposals x all chunks in one graph launch equal K single evaluations / the oracle."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 4, 35 + 11 * i, seed=900 + i, mask_frac=0.03 * (i % 2)) for i in range(4)]
    p = synthetic.default_params("SB2")
    P = np.stack([p * (1.0 + 0.01 * k * np.array([0, 1, 0, 0, 0, 0, 0, 1, 0, 0, 1])) for k in range(5)])
    P[3, 1] = 4e5   # |v| >= c for proposal 3 only
    farm = ChunkFarm("SB2", chunks, n_proposals=5, nbranch=6)
    got = farm.lnprob_many(P)
    per = farm.chunk_lnlikes(P).cpu().numpy()
    assert got.shape == (5,) and per.shape == (5, 4)
    for k in range(5):
        ref, ref_vec = oracle.farm_lnprob("SB2", P[k], chunks)
        if k == 3:
            assert got[k] == -np.inf and ref == -np.inf
        else:
            assert rel_close(got[k], ref, LNLIKE_RTOL) and rel_close(per[k], ref_vec, LNLIKE_RTOL), (k, got[k], ref)
    farm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"PSOAP_POTRF": "3"}, {"PSOAP_POTRF": "7", "PSOAP_GROUP": "4"},
                                 {"PSOAP_PDL": "0", "PSOAP_LOOKAHEAD": "0"}, {"PSOAP_PDL": "100000"},
                                 {"PSOAP_TAIL": "1"}, {"PSOAP_YIELD_LOOKAHEAD": "1"}, {"PSOAP_FARM_LOOKAHEAD": "0"}],
                         ids=["inverse-chain-everywhere", "blocked-chain-everywhere-group4", "no-pdl-no-lookahead", "pdl-everywhere",
                              "quarter-tile-tail", "one-tile-per-cta-bulk", "farm-without-lookahead"])
def test_alternative_kernel_paths(env, torch_cuda):
    """The library's environment switches select alternative kernels / launch modes for the same contract (the blocked
    diagonal factorisation + blocked panel solve of csrc/chain.cuh, launch attributes).  They are read once at load
    time, so the parity tests are re-run in a child process for each."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    child_env = dict(os.environ, **env)
    cmd = [sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", os.path.join(root, "tests", "test_gpu_parity.py"),
           "-k", "lnlike_golden or tile_boundaries or predict_golden or farm_vs_oracle or package_default_hyperparameters_large"]
    out = subprocess.run(cmd, cwd=root, env=child_env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert " passed" in out.stdout and "failed" not in out.stdout


@pytest.mark.gpu
def test_second_device_in_one_process_is_refused(torch_cuda):
    """The library binds to the device of its first call (one process per GPU); another current device is an error,
    not an invalid-resource-handle launch later."""
    import ctypes
    from psoap_b200 import _lib
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    lib = _lib.load()
    ms, fl = ctypes.c_double(), ctypes.c_double()
    _lib.check(lib.psoap_bench_syrk(256, 128, 1, ctypes.byref(ms), ctypes.byref(fl)))     # binds to the current device
    cur = torch.cuda.current_device()
    try:
        torch.cuda.set_device((cur + 1) % torch.cuda.device_count())
        with pytest.raises(_lib.PsoapError, match="one process per GPU"):
            _lib.check(lib.psoap_bench_syrk(256, 128, 1, ctypes.byref(ms), ctypes.byref(fl)))
    finally:
        torch.cuda.set_device(cur)
