"""Gradient of the log-likelihood (psoap_lnlike_grad, psoap_chunk_lnprob_grad, psoap_orbit_jacobian).

CPU: a numpy gradient helper and a numpy orbit Jacobian, each checked against central differences of the oracle.
GPU (-m gpu): the restricted identity-border elimination against an unrestricted psoap_schur of the same matrix (==),
the device gradient against the numpy helper (and, at N = 12289, a torch comparator), the chunk chain rule, directional
derivatives of ChunkFarm.lnprob, the -inf conventions, bit stability and an L-BFGS-B fit.

Scale of a gradient entry: S_theta = 1/2 sum_ij |W_ij dK_ij/dtheta| (W = alpha alpha^T - K^-1), the size of the terms
the entry is a sum of; entries are compared within a multiple of it.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C_KMS = 2.99792458e5
NORB = {"SB1": 6, "SB2": 7, "ST1": 11, "ST2": 12, "ST3": 13}
NCOMP = {"SB1": 1, "SB2": 2, "ST1": 1, "ST2": 2, "ST3": 3}


# ---------------------------------------------------------------------------------------------- numpy helpers
def np_lnlike_grad(lwls, fl, sigma, amps, ls, mu=1.0):
    """Exact gradient in numpy/scipy: returns (lnlike, grads, scales) with grads/scales dicts of
    amp [ncomp], l [ncomp], mu (float), lwl [ncomp, N]; also cond(K)."""
    from scipy.linalg import cho_factor, cho_solve
    lwls = [np.asarray(z, dtype=np.float64) for z in lwls]
    N = len(fl)
    K = np.diag(np.asarray(sigma, dtype=np.float64) ** 2)
    terms = []
    for z, a, l in zip(lwls, amps, ls):
        p2 = -0.5 * C_KMS ** 2 / (l * l)
        D = z[None, :] - z[:, None]  # D_ij = z_j - z_i
        x = p2 * D * D
        E = np.exp(x)
        terms.append((D, x, E, a, l, p2))
        K = K + a * a * E
    cf = cho_factor(K, lower=True)
    r = np.asarray(fl, dtype=np.float64) - mu
    alpha = cho_solve(cf, r)
    Kinv = cho_solve(cf, np.eye(N))
    logdet = 2.0 * np.sum(np.log(np.diag(cf[0])))
    W = np.outer(alpha, alpha) - Kinv
    g = dict(amp=[], l=[], lwl=[])
    s = dict(amp=[], l=[], lwl=[])
    for D, x, E, a, l, p2 in terms:
        k = a * a * E
        dA = 2.0 * a * E
        dL = -2.0 * k * x / l
        dZ = W * (2.0 * p2 * (-D) * k)  # dZ[i, j] = W_ij dK_ij/dz_i
        g["amp"].append(0.5 * np.sum(W * dA)); s["amp"].append(0.5 * np.sum(np.abs(W * dA)))
        g["l"].append(0.5 * np.sum(W * dL)); s["l"].append(0.5 * np.sum(np.abs(W * dL)))
        g["lwl"].append(dZ.sum(axis=1)); s["lwl"].append(np.abs(dZ).sum(axis=1))
    g["mu"], s["mu"] = float(np.sum(alpha)), float(np.sum(np.abs(alpha)))
    for key in ("amp", "l", "lwl"):
        g[key], s[key] = np.array(g[key]), np.array(s[key])
    lnl = -0.5 * (r @ alpha + logdet)
    ev = np.linalg.eigvalsh(K)
    return lnl, g, s, ev[-1] / ev[0]


def np_kepler(t, T0, P, e):
    """(f, E) of orbit.py:47-72 by Newton to convergence (vectorised)."""
    tp = np.mod(t - T0, P)
    M = 2 * np.pi * tp / P
    E = M.copy()
    for _ in range(100):
        E = E - (E - e * np.sin(E) - M) / (1 - e * np.cos(E))
    th = 2 * np.arctan(np.sqrt((1 + e) / (1 - e)) * np.tan(E / 2.0))
    return np.where(E < np.pi, th, th + 2 * np.pi), E


def np_rv_grad(K, e, om, P, T0, t):
    """d rv / d(K, e, omega, P, T0), each [n_dates]."""
    f, E = np_kepler(t, T0, P, e)
    w = om * np.pi / 180
    den = 1 - e * np.cos(E)
    se = np.sqrt(1 - e * e)
    dfdM = se / den ** 2
    dfde = se * np.sin(E) / den ** 2 + np.sin(f) / (1 - e * e)
    dvdf = -K * np.sin(w + f)
    return [np.cos(w + f) + e * np.cos(w), dvdf * dfde + K * np.cos(w), -K * (np.sin(w + f) + e * np.sin(w)) * np.pi / 180,
            dvdf * dfdM * (-2 * np.pi * (t - T0) / P ** 2), dvdf * dfdM * (-2 * np.pi / P)]


def np_velocity_jacobian(model, p, dates):
    """[ncomp, n_dates, norb] Jacobian of oracle.get_velocities."""
    t = np.asarray(dates, dtype=np.float64)
    nc, no = NCOMP[model], NORB[model]
    J = np.zeros((nc, len(t), no))
    J[:, :, no - 1] = 1.0

    def term(c, o, iq, q, K, e, om, P, T0):
        g = np_rv_grad(K / q, e, om, P, T0, t)
        J[c, :, o] += g[0] / q
        if iq >= 0:
            J[c, :, iq] += -K / q ** 2 * g[0]
        for k in range(1, 5):
            J[c, :, o + k] += g[k]

    if model in ("SB1", "SB2"):
        o = 1 if model == "SB2" else 0
        K, e, om, P, T0 = p[o:o + 5]
        term(0, o, -1, 1.0, K, e, om, P, T0)
        if model == "SB2":
            term(1, o, 0, p[0], K, e, om + 180, P, T0)
        return J
    o = 0 if model == "ST1" else 1
    oo = o + 5 + (1 if model == "ST3" else 0)
    Ki, ei, omi, Pi, T0i = p[o:o + 5]
    Ko, eo, omo, Po, T0o = p[oo:oo + 5]
    term(0, o, -1, 1.0, Ki, ei, omi, Pi, T0i)
    term(0, oo, -1, 1.0, Ko, eo, omo, Po, T0o)
    if model != "ST1":
        term(1, o, 0, p[0], Ki, ei, omi + 180, Pi, T0i)
        term(1, oo, -1, 1.0, Ko, eo, omo, Po, T0o)
    if model == "ST3":
        term(2, oo, o + 5, p[o + 5], Ko, eo, omo + 180, Po, T0o)
    return J


def make_problem(N, ncomp, seed, amps=(0.1, 0.07, 0.05), ls=(5.0, 6.0, 7.0), sig=0.03):
    """Shifted ln-wavelengths of ncomp components on one 2.8 km/s pixel grid, flux around 1."""
    rng = np.random.default_rng(seed)
    dpix = 2.8 / C_KMS
    base = np.log(5000.0) + np.arange(N) * dpix + rng.uniform(-0.2, 0.2, N) * dpix
    lwls = [base - v / C_KMS for v in (0.0, 17.0, -31.0)[:ncomp]]
    fl = 1.0 + 0.1 * rng.standard_normal(N)
    sigma = sig * (1.0 + 0.2 * rng.uniform(size=N))
    return lwls, fl, sigma, list(amps[:ncomp]), list(ls[:ncomp])


ORBITS = {
    "SB1": [5.0, 0.2, 10.0, 10.0, 3.0, 5.0],
    "SB2": [0.2, 5.0, 0.2, 10.0, 10.0, 3.0, 5.0],
    "ST1": [5.0, 0.2, 10.0, 10.0, 3.0, 4.0, 0.3, 80.0, 100.0, 20.0, 5.0],
    "ST2": [0.4, 5.0, 0.2, 10.0, 10.0, 3.0, 4.0, 0.3, 80.0, 100.0, 20.0, 5.0],
    "ST3": [0.4, 5.0, 0.2, 10.0, 10.0, 3.0, 0.2, 4.0, 0.3, 80.0, 100.0, 20.0, 5.0],
}
ECC = {"SB1": [1], "SB2": [2], "ST1": [1, 6], "ST2": [2, 7], "ST3": [2, 8]}


def orbit_case(model, ecc):
    p = np.array(ORBITS[model], dtype=np.float64)
    for k in ECC[model]:
        p[k] = ecc
    # dates over several periods on both sides of T0, so that the modulus of orbit.py:60 wraps
    dates = np.array([-251.3, -37.7, -9.1, -0.4, 2.2, 7.9, 13.3, 26.6, 58.1, 311.7])
    return p, dates


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_numpy_gradient_matches_central_differences(ncomp, oracle):
    lwls, fl, sigma, amps, ls = make_problem(40, ncomp, seed=10 + ncomp)
    lnl_fn = oracle.lnlike[{1: "SB1", 2: "SB2", 3: "ST3"}[ncomp]]

    def f(lw, am, ll, mu):
        return lnl_fn(np.empty((40, 40)), *lw, fl, sigma, *[x for pair in zip(am, ll) for x in pair], mu_GP=mu)

    lnl, g, s, cond = np_lnlike_grad(lwls, fl, sigma, amps, ls)
    print("cond(K) = %.3g" % cond)
    assert cond <= 1e5
    assert abs(lnl - f(lwls, amps, ls, 1.0)) <= 1e-12 * abs(lnl)
    tol = 1e-6
    for c in range(ncomp):
        for key, vals in (("amp", amps), ("l", ls)):
            h = 1e-5 * vals[c]
            up, dn = list(vals), list(vals)
            up[c] += h; dn[c] -= h
            if key == "amp":
                fd = (f(lwls, up, ls, 1.0) - f(lwls, dn, ls, 1.0)) / (2 * h)
            else:
                fd = (f(lwls, amps, up, 1.0) - f(lwls, amps, dn, 1.0)) / (2 * h)
            assert abs(fd - g[key][c]) <= tol * s[key][c], (key, c, fd, g[key][c], s[key][c])
        h = 1e-3 * 2.8 / C_KMS
        for i in range(40):
            up = [z.copy() for z in lwls]; dn = [z.copy() for z in lwls]
            up[c][i] += h; dn[c][i] -= h
            fd = (f(up, amps, ls, 1.0) - f(dn, amps, ls, 1.0)) / (2 * h)
            assert abs(fd - g["lwl"][c][i]) <= 1e-5 * s["lwl"][c][i], (c, i, fd, g["lwl"][c][i], s["lwl"][c][i])
    h = 1e-5
    fd = (f(lwls, amps, ls, 1.0 + h) - f(lwls, amps, ls, 1.0 - h)) / (2 * h)
    assert abs(fd - g["mu"]) <= tol * s["mu"]


@pytest.mark.parametrize("model", ["SB1", "SB2", "ST1", "ST2", "ST3"])
@pytest.mark.parametrize("ecc", [0.0, 0.9])
def test_numpy_orbit_jacobian_matches_central_differences(model, ecc, oracle):
    p, dates = orbit_case(model, ecc)
    J = np_velocity_jacobian(model, p, dates)
    v0 = oracle.get_velocities(model, p, dates)
    assert J.shape == (NCOMP[model], len(dates), NORB[model]) and v0.shape == J.shape[:2]
    # step per parameter: 1e-6 of its size (1e-6 days / degrees / km/s where it is zero)
    for k in range(NORB[model]):
        h = 1e-6 * max(abs(p[k]), 1.0)
        up, dn = p.copy(), p.copy()
        up[k] += h; dn[k] -= h
        if k in ECC[model] and dn[k] < 0.0:  # e >= 0 is asserted: one-sided second-order difference at e = 0
            up2 = p.copy(); up2[k] += 2 * h
            fd = (-3 * v0 + 4 * oracle.get_velocities(model, up, dates) - oracle.get_velocities(model, up2, dates)) / (2 * h)
        else:
            fd = (oracle.get_velocities(model, up, dates) - oracle.get_velocities(model, dn, dates)) / (2 * h)
        scale = np.abs(J[:, :, k]) + 1e-3 * np.max(np.abs(J)) + 1e-9
        assert np.all(np.abs(fd - J[:, :, k]) <= 1e-5 * scale), (k, fd, J[:, :, k])


# ---------------------------------------------------------------------------------------------- GPU helpers
def _lib():
    from psoap_b200 import _lib as L
    return L, L.load()


def _flat_view(torch, buf, addr, count):
    off = addr - buf.data_ptr()
    assert off % 8 == 0
    return buf[off:off + 8 * count].view(torch.float64)


def _lower_block(torch, buf, addr, ld, N):
    """Column-major lower-triangular [N, N] block at device address addr: returns Bt with Bt[j, i] = B(i, j)."""
    flat = _flat_view(torch, buf, addr, (N - 1) * ld + N)
    return torch.triu(flat.as_strided((N, N), (ld, 1)))


def _grad_call(lwls_d, fl_d, sg_d, amps, ls, mu=1.0, ws=None):
    """psoap_lnlike_grad through the C ABI: returns (result [4], grad_hyp, grad_lwl, workspace)."""
    import torch
    L, lib = _lib()
    ncomp, N = len(lwls_d), fl_d.numel()
    nbytes = lib.psoap_lnlike_grad_workspace_bytes(ncomp, N)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    gh = torch.empty(2 * ncomp + 1, dtype=torch.float64, device="cuda")
    gl = torch.empty((ncomp, max(N, 1)), dtype=torch.float64, device="cuda")
    p = [L.ptr(v) for v in lwls_d] + [L.vp(None)] * (3 - ncomp)
    L.check(lib.psoap_lnlike_grad(ncomp, N, p[0], p[1], p[2], L.ptr(fl_d), L.ptr(sg_d), L.dbl_array(amps),
                                  L.dbl_array(ls), float(mu), L.ptr(ws), nbytes, L.ptr(res), L.ptr(gh), L.ptr(gl),
                                  L.stream_ptr()))
    torch.cuda.synchronize()
    return res.cpu().numpy(), gh.cpu().numpy(), gl[:, :N].cpu().numpy(), ws


def restriction_case(N, ncomp=2):
    """-K^-1 and -alpha of the gradient entry against an unrestricted psoap_schur of the same identity-bordered
    matrix (built here: the internal fill through psoap_debug_fill_lower, the border written by hand)."""
    import torch
    L, lib = _lib()
    lwls, fl, sigma, amps, ls = make_problem(N, ncomp, seed=N)
    lw = [torch.from_numpy(z).cuda() for z in lwls]
    fl_d, sg_d = torch.from_numpy(fl).cuda(), torch.from_numpy(sigma).cuda()
    Nn = (N + 127) // 128 * 128
    Nt, pad = 2 * Nn, Nn - N
    St = torch.zeros((Nt, Nt), dtype=torch.float64, device="cuda")  # S(i, j) = St[j, i]
    nbytes = lib.psoap_schur_workspace_bytes(N, N)
    sws = torch.zeros(nbytes + 256, dtype=torch.uint8, device="cuda")
    rv, acc, info = L.vp(), L.vp(), L.vp()
    L.check(lib.psoap_schur_views(L.ptr(sws), N, N, ctypes.byref(rv), ctypes.byref(acc), ctypes.byref(info)))
    p = [L.ptr(v) for v in lw] + [L.vp(None)] * (3 - ncomp)
    L.check(lib.psoap_debug_fill_lower(ncomp, N, p[0], p[1], p[2], None, None, 0, L.ptr(fl_d), L.ptr(sg_d),
                                       L.dbl_array(amps), L.dbl_array(ls), 1.0, L.ptr(St), Nt, L.vp(rv.value),
                                       L.stream_ptr()))
    a = torch.arange(N, device="cuda")
    St[pad + a, Nn + a] = 1.0                      # S(Nn + a, pad + a) = 1
    dead = torch.arange(Nn + N, Nt, device="cuda")
    St[dead, dead] = 1.0
    _flat_view(torch, sws, rv.value, Nt)[Nn:] = 0.0
    _flat_view(torch, sws, acc.value, 8).zero_()
    sws[info.value - sws.data_ptr():info.value - sws.data_ptr() + 8].zero_()
    sres = torch.empty(4, dtype=torch.float64, device="cuda")
    L.check(lib.psoap_schur(L.ptr(St), Nt, N, N, L.ptr(sws), nbytes, L.ptr(sres), L.stream_ptr()))
    ref_blk = torch.triu(St[Nn:Nn + N, Nn:Nn + N])
    ref_alpha = _flat_view(torch, sws, rv.value, Nt)[Nn:Nn + N].clone()
    res, gh, gl, ws = _grad_call(lw, fl_d, sg_d, amps, ls)
    kinv, ld, nal = L.vp(), ctypes.c_int64(), L.vp()
    L.check(lib.psoap_lnlike_grad_views(L.ptr(ws), N, ctypes.byref(kinv), ctypes.byref(ld), ctypes.byref(nal)))
    blk = _lower_block(torch, ws, kinv.value, ld.value, N)
    alpha = _flat_view(torch, ws, nal.value, N)
    assert float(sres[3]) == 0.0 and res[3] == 0.0
    assert float(sres[1]) == res[1] and float(sres[2]) == res[2]
    assert torch.equal(blk, ref_blk), float((blk - ref_blk).abs().max())
    assert torch.equal(alpha, ref_alpha)
    return True


# ---------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("N", [1, 127, 128, 129, 2000, 4000, 6145, 12289])
def test_restricted_elimination_is_exact(N):
    assert restriction_case(N)


RESTRICT_ENVS = {"potrf3": {"PSOAP_POTRF": "3"}, "group1": {"PSOAP_GROUP": "1"}, "group8": {"PSOAP_GROUP": "8"},
                 "no-lookahead": {"PSOAP_LOOKAHEAD": "0"}, "yield1": {"PSOAP_YIELD_LOOKAHEAD": "1"},
                 "yield2": {"PSOAP_YIELD_LOOKAHEAD": "2"}, "no-pdl": {"PSOAP_PDL": "0"}}


@gpu
@pytest.mark.parametrize("cfg", sorted(RESTRICT_ENVS))
def test_restricted_elimination_launch_paths(cfg):
    env = dict(os.environ, **RESTRICT_ENVS[cfg])
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), "restrict", "2000"], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "restrict ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def _assert_grad_close(got_lnl, gh, gl, lnl, g, s, ncomp, rtol=1e-10):
    assert abs(got_lnl - lnl) <= 1e-12 * abs(lnl), (got_lnl, lnl)
    for c in range(ncomp):
        assert abs(gh[2 * c] - g["amp"][c]) <= rtol * s["amp"][c], ("amp", c, gh[2 * c], g["amp"][c])
        assert abs(gh[2 * c + 1] - g["l"][c]) <= rtol * s["l"][c], ("l", c, gh[2 * c + 1], g["l"][c])
    assert abs(gh[-1] - g["mu"]) <= rtol * s["mu"]
    err = np.abs(gl - g["lwl"]) / s["lwl"]
    assert np.all(err <= rtol), float(err.max())


@gpu
@pytest.mark.parametrize("ncomp,N", [(1, 129), (1, 256), (2, 300), (3, 1000), (2, 2000), (3, 2048), (2, 4000)])
def test_gradient_matches_numpy(ncomp, N):
    import torch
    from psoap_b200 import covariance
    lwls, fl, sigma, amps, ls = make_problem(N, ncomp, seed=100 * ncomp + N)
    lnl, g, s, cond = np_lnlike_grad(lwls, fl, sigma, amps, ls)
    print("N = %d ncomp = %d cond(K) = %.3g" % (N, ncomp, cond))
    assert cond <= 1e5
    out = covariance.lnlike_grad(lwls, fl, sigma, amps, ls, mu_GP=1.0)
    gh = np.empty(2 * ncomp + 1)
    gh[0:2 * ncomp:2], gh[1:2 * ncomp:2], gh[-1] = out.amp, out.l, out.mu_GP
    assert isinstance(out.lwl, np.ndarray) and out.lwl.shape == (ncomp, N)
    _assert_grad_close(out.lnlike, gh, out.lwl, lnl, g, s, ncomp)
    ref = covariance._lnlike(None, lwls, fl, sigma, amps, ls, 1.0)
    assert abs(out.lnlike - ref) <= 1e-12 * abs(ref)
    # device inputs give a device per-pixel gradient with the same bits
    dev = covariance.lnlike_grad([torch.from_numpy(z).cuda() for z in lwls], torch.from_numpy(fl).cuda(),
                                 torch.from_numpy(sigma).cuda(), amps, ls)
    assert dev.lwl.is_cuda and np.array_equal(dev.lwl.cpu().numpy(), out.lwl) and dev.lnlike == out.lnlike


def _torch_grad(torch, lwls, fl, sigma, amps, ls, mu=1.0):
    """Test-only comparator on the GPU: operator-surface fill, torch Cholesky / cholesky_inverse, contraction in torch."""
    from psoap_b200 import matrix_functions as mf
    N, ncomp = len(fl), len(lwls)
    z = [torch.from_numpy(v).cuda() for v in lwls]
    K = torch.empty((N, N), dtype=torch.float64, device="cuda")
    {1: mf.fill_V11_f, 2: mf.fill_V11_f_g, 3: mf.fill_V11_f_g_h}[ncomp](K, *z, *[x for p in zip(amps, ls) for x in p])
    K.diagonal().add_(torch.from_numpy(sigma).cuda() ** 2)
    Lc = torch.linalg.cholesky(K)
    r = torch.from_numpy(fl).cuda() - mu
    alpha = torch.cholesky_solve(r[:, None], Lc)[:, 0]
    W = torch.cholesky_inverse(Lc).neg_().addr_(alpha, alpha)
    del K
    g, s = dict(amp=[], l=[], lwl=[]), dict(amp=[], l=[], lwl=[])
    for c in range(ncomp):
        p2 = -0.5 * C_KMS ** 2 / (ls[c] ** 2)
        D = z[c][None, :] - z[c][:, None]
        x = p2 * D * D
        k = amps[c] ** 2 * torch.exp(x)
        T = W * k                                      # W_ij k_ij
        g["amp"].append(float(T.sum()) / amps[c]); s["amp"].append(float(T.abs().sum()) / amps[c])
        T.mul_(x)
        g["l"].append(-float(T.sum()) / ls[c]); s["l"].append(float(T.abs().sum()) / ls[c])
        T = W * k * (-2.0 * p2) * D
        g["lwl"].append(T.sum(dim=1).cpu().numpy()); s["lwl"].append(T.abs().sum(dim=1).cpu().numpy())
        del D, x, k, T
    g["mu"], s["mu"] = float(alpha.sum()), float(alpha.abs().sum())
    for key in ("amp", "l", "lwl"):
        g[key], s[key] = np.array(g[key]), np.array(s[key])
    lnl = float(-0.5 * (r @ alpha + 2.0 * torch.log(torch.diagonal(Lc)).sum()))
    return lnl, g, s


@gpu
def test_gradient_large_against_torch():
    import torch
    from psoap_b200 import covariance
    N, ncomp = 12289, 2
    lwls, fl, sigma, amps, ls = make_problem(N, ncomp, seed=12289)
    out = covariance.lnlike_grad(lwls, fl, sigma, amps, ls)
    gh = np.empty(2 * ncomp + 1)
    gh[0:2 * ncomp:2], gh[1:2 * ncomp:2], gh[-1] = out.amp, out.l, out.mu_GP
    lnl, g, s = _torch_grad(torch, lwls, fl, sigma, amps, ls)
    torch.cuda.empty_cache()
    _assert_grad_close(out.lnlike, gh, out.lwl, lnl, g, s, ncomp)


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST1", "ST2", "ST3"])
def test_orbit_jacobian_device(model):
    from psoap_b200 import orbit
    for ecc in (0.0, 0.5, 0.9):
        p, dates = orbit_case(model, ecc)
        J = orbit.velocity_jacobian(model, p, dates).cpu().numpy()
        ref = np_velocity_jacobian(model, p, dates)
        assert np.all(np.abs(J - ref) <= 1e-10 * (np.abs(ref) + 1.0)), np.abs(J - ref).max()


def _chunk_desc(torch, ch, keep):
    from psoap_b200 import _lib as L
    t = {k: torch.from_numpy(np.ascontiguousarray(ch[k])).cuda() for k in ("lwl", "fl", "sigma", "date1D", "epoch")}
    keep.append(t)
    d = L.PsoapChunk()
    d.N, d.n_epochs = len(ch["fl"]), len(ch["date1D"])
    d.lwl, d.epoch, d.fl = t["lwl"].data_ptr(), t["epoch"].data_ptr(), t["fl"].data_ptr()
    d.sigma, d.dates = t["sigma"].data_ptr(), t["date1D"].data_ptr()
    return d


def _chunk_grad(torch, model, ch, p, mu=1.0):
    L, lib = _lib()
    keep = []
    d = _chunk_desc(torch, ch, keep)
    nb = lib.psoap_chunk_lnprob_grad_workspace_bytes(L.MODELS[model], d.N, d.n_epochs)
    ws = torch.empty(nb + 256, dtype=torch.uint8, device="cuda")
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    gp = torch.empty(len(p), dtype=torch.float64, device="cuda")
    p_d = torch.from_numpy(np.asarray(p, dtype=np.float64)).cuda()
    L.check(lib.psoap_chunk_lnprob_grad(L.MODELS[model], ctypes.byref(d), L.ptr(p_d), mu, L.ptr(ws), nb, L.ptr(res),
                                        L.ptr(gp), L.stream_ptr()))
    torch.cuda.synchronize()
    return res.cpu().numpy(), gp.cpu().numpy()


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_chunk_chain_rule(model):
    """psoap_chunk_lnprob_grad = the direct entry's per-pixel gradient, summed per epoch and composed with the
    orbit Jacobian in Python."""
    import torch
    from psoap_b200 import covariance, data, orbit, synthetic
    ch = synthetic.make_chunk(model, 8, 150, seed=41, mask_frac=0.05)
    p = synthetic.default_params(model)
    no, nc = NORB[model], NCOMP[model]
    res, gp = _chunk_grad(torch, model, ch, p)
    vel = orbit.velocities(model, p[:no], ch["date1D"])
    lwls = data.replicate_wls(torch.from_numpy(ch["lwl"]).cuda(), vel, ch["mask"])
    out = covariance.lnlike_grad([lwls[c] for c in range(nc)], ch["fl"], ch["sigma"], list(p[no::2]), list(p[no + 1::2]))
    assert res[0] == out.lnlike
    gz = np.asarray(out.lwl)
    ep = ch["epoch"]
    gv = np.array([[-gz[c][ep == e].sum() / C_KMS for e in range(len(ch["date1D"]))] for c in range(nc)])
    J = orbit.velocity_jacobian(model, p[:no], ch["date1D"]).cpu().numpy()
    terms = gv[:, :, None] * J
    g_orb, scale = terms.sum(axis=(0, 1)), np.abs(terms).sum(axis=(0, 1))
    assert np.all(np.abs(gp[:no] - g_orb) <= 1e-12 * scale + 1e-300), (gp[:no], g_orb)
    g_gp = np.empty(2 * nc)
    g_gp[0::2], g_gp[1::2] = out.amp, out.l
    assert np.all(np.abs(gp[no:] - g_gp) <= 1e-12 * np.abs(g_gp)), (gp[no:], g_gp)


# per-parameter step scales of the directional checks (units of the parameter)
STEP = {"q": 1e-3, "q_in": 1e-3, "q_out": 1e-3, "K": 0.1, "K_in": 0.1, "K_out": 0.1, "e": 1e-3, "e_in": 1e-3,
        "e_out": 1e-3, "omega": 0.1, "omega_in": 0.1, "omega_out": 0.1, "P": 1e-3, "P_in": 1e-3, "P_out": 1e-2,
        "T0": 1e-2, "T0_in": 1e-2, "T0_out": 1e-2, "gamma": 0.1, "amp_f": 1e-3, "amp_g": 1e-3, "amp_h": 1e-3,
        "l_f": 1e-2, "l_g": 1e-2, "l_h": 1e-2}


@gpu
@pytest.mark.parametrize("case", ["SB1", "SB2", "ST3", "SB2-defaults-N4000"])
def test_farm_gradient_directional(case):
    from psoap_b200 import synthetic, utils
    from psoap_b200.farm import ChunkFarm
    model = case.split("-")[0]
    if case.endswith("N4000"):
        chunks = [synthetic.make_chunk(model, 20, 200, seed=77)]
        p = synthetic.default_params(model)
        p[NORB[model]:] = [0.5, 5.0] * NCOMP[model]   # the package defaults amp = 0.5, l = 5
    else:
        chunks = [synthetic.make_chunk(model, 6, 70 + 10 * i, seed=60 + i, mask_frac=0.03) for i in range(3)]
        p = synthetic.default_params(model)
    farm = ChunkFarm(model, chunks)
    lnp, g = farm.lnprob_and_grad(p)
    assert lnp == farm.lnprob(p)
    rng = np.random.default_rng(5)
    steps = np.array([STEP[n] for n in utils.registered_params[model]])
    for _ in range(3):
        u = rng.standard_normal(len(p)) * steps
        t = 1e-3
        fd = (farm.lnprob(p + t * u) - farm.lnprob(p - t * u)) / (2 * t)
        scale = np.sum(np.abs(g * u))
        assert abs(fd - g @ u) <= 1e-5 * scale, (fd, g @ u, scale)
    farm.close()


@gpu
def test_minus_inf_conventions():
    import torch
    from psoap_b200 import covariance, synthetic
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    lwls, fl, sigma, amps, ls = make_problem(300, 2, seed=3)
    out = covariance.lnlike_grad(lwls, fl, sigma, [0.1, -0.05], ls)
    assert out.lnlike == -np.inf and np.isnan(out.amp).all() and np.isnan(out.l).all() and np.isnan(out.mu_GP)
    assert np.isnan(out.lwl).all()
    # a negative GP value and |v| >= c in the farm's vector
    ch = synthetic.make_chunk("SB2", 4, 60, seed=9)
    farm = ChunkFarm("SB2", [ch])
    for bad in (dict(k=7, v=-0.1), dict(k=1, v=4e5)):
        p = synthetic.default_params("SB2")
        p[bad["k"]] = bad["v"]
        lnp, g = farm.lnprob_and_grad(p)
        assert lnp == -np.inf and np.isnan(g).all()
    farm.close()
    # N = 0: -0.0 and zeros
    out = covariance.lnlike_grad([np.zeros(0)], np.zeros(0), np.zeros(0), [0.1], [5.0])
    assert out.lnlike == 0.0 and np.signbit(out.lnlike) and out.amp[0] == 0.0 and out.mu_GP == 0.0
    assert out.lwl.shape == (1, 0)
    # exactly singular K: N = 2, identical z, sigma = 0, amp = 0.5 (amp^2, L_11, L_21 exact, second pivot 0)
    z = torch.full((2,), np.log(5000.0), dtype=torch.float64, device="cuda")
    fl2, sg2 = torch.tensor([1.3, 0.7], dtype=torch.float64, device="cuda"), torch.zeros(2, dtype=torch.float64, device="cuda")
    Wm = torch.zeros((128, 128), dtype=torch.float64, device="cuda")
    rv = torch.zeros(128, dtype=torch.float64, device="cuda")
    L.check(lib.psoap_debug_fill_lower(1, 2, L.ptr(z), None, None, None, None, 0, L.ptr(fl2), L.ptr(sg2),
                                       L.dbl_array([0.5]), L.dbl_array([5.0]), 1.0, L.ptr(Wm), 128, L.ptr(rv),
                                       L.stream_ptr()))
    assert float(Wm[126, 127]) == 0.25          # S(127, 126) = amp^2 exp_neg(0): exp_neg(0) is exactly 1
    res, gh, gl, ws = _grad_call([z], fl2, sg2, [0.5], [5.0])
    assert res[3] == 2.0 and res[0] == -np.inf and np.isnan(gh).all() and np.isnan(gl).all()
    # the next valid call on the same workspace is correct
    lwls, fl, sigma, amps, ls = make_problem(2, 1, seed=4)
    res, gh, gl, _ = _grad_call([torch.from_numpy(lwls[0]).cuda()], torch.from_numpy(fl).cuda(),
                                torch.from_numpy(sigma).cuda(), amps, ls, ws=ws)
    lnl, g, s, _ = np_lnlike_grad(lwls, fl, sigma, amps, ls)
    assert res[3] == 0.0
    _assert_grad_close(res[0], gh, gl, lnl, g, s, 1)


@gpu
def test_gradient_bit_stability():
    import torch
    from psoap_b200 import covariance, synthetic
    from psoap_b200.farm import ChunkFarm
    lwls, fl, sigma, amps, ls = make_problem(3000, 3, seed=8)
    a = covariance.lnlike_grad(lwls, fl, sigma, amps, ls)
    b = covariance.lnlike_grad(lwls, fl, sigma, amps, ls)
    assert a.lnlike == b.lnlike and np.array_equal(a.amp, b.amp) and np.array_equal(a.l, b.l)
    assert a.mu_GP == b.mu_GP and np.array_equal(a.lwl, b.lwl)
    # emulated ranks (as test_farm_partition_matches_single): identical per-chunk rows, the same summed gradient
    chunks = [synthetic.make_chunk("SB2", 4, 30 + 7 * i, seed=300 + i) for i in range(9)]
    p = synthetic.default_params("SB2")
    single = ChunkFarm("SB2", chunks)
    ref = single.chunk_lnlike_grads(p).cpu().numpy()
    ref_sum = single.lnprob_and_grad(p)
    total = np.zeros_like(ref)
    for r in range(4):
        f = ChunkFarm("SB2", chunks, rank=r, world_size=4)
        f.world_size = 1  # no process group here: take the un-reduced rows
        rows = f.chunk_lnlike_grads(p).cpu().numpy()
        for i in f.mine:
            assert np.array_equal(rows[i], ref[i])
        total = total + rows
        f.close()
    assert np.array_equal(total, ref)
    assert float(np.sum(total[:, 0])) == ref_sum[0] and np.array_equal(np.sum(total[:, 1:], axis=0), ref_sum[1])
    assert ref_sum[0] == single.lnprob(p)
    single.close()


@gpu
def test_lbfgs_with_gradient_reaches_nelder_mead_optimum():
    from scipy.optimize import minimize
    from psoap_b200 import covariance, synthetic
    ch = synthetic.make_chunk("SB1", 3, 120, seed=12)
    lw, fl, sg = ch["lwl"], ch["fl"], ch["sigma"]
    x_nm = covariance.optimize_GP_f(lw, fl, sg, 0.1, 5.0)
    f_nm = -covariance.lnlike_f(None, lw, fl, sg, *x_nm)

    def fun(x):
        out = covariance.lnlike_grad([lw], fl, sg, [x[0]], [x[1]])
        return -out.lnlike, -np.array([out.amp[0], out.l[0]])

    r = minimize(fun, np.array([0.1, 5.0]), method="L-BFGS-B", jac=True, bounds=[(1e-4, None), (1e-2, None)])
    print("Nelder-Mead", x_nm, f_nm, "L-BFGS-B", r.x, r.fun, r.nfev)
    assert r.fun <= f_nm + 1e-9 * abs(f_nm)


if __name__ == "__main__":
    if sys.argv[1] == "restrict":
        import torch
        assert torch.cuda.is_available()
        restriction_case(int(sys.argv[2]))
        print("restrict ok")
