"""Free per-epoch radial velocities (PSOAP_FREE1..3, psoap_farm_create_free, ChunkFarm(free_velocities=True) and
sample.fit_epoch_velocities): the radial velocity of every component at every epoch in place of an orbit.

The free path feeds the fill the same velocity table the orbit path computes when the free vector holds the orbit's
velocities, so likelihoods and predictions are the orbit path's bits there; gradients and Fisher matrices are the
orbit's through the chain rule.  The CPU tests cover the epoch maps, the argument checks and the fit driver's gauge.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NORB = {"SB1": 6, "SB2": 7, "ST3": 13}
NCOMP = {"SB1": 1, "SB2": 2, "ST3": 3}
C_KMS = 2.99792458e5
gpu = pytest.mark.gpu


def _lib():
    from psoap_b200 import _lib as L
    return L, L.load()


def chunks_on(model, dates, subsets, n_pix, seed):
    """Synthetic chunks that observe the given subsets of one date list (chunk i: dates[subsets[i]])."""
    from psoap_b200 import synthetic
    out = []
    for i, (sub, npx) in enumerate(zip(subsets, n_pix)):
        ch = synthetic.make_chunk(model, len(sub), npx, seed=seed + i, wl0=5000.0 + 3.0 * i)
        ch["date1D"] = np.asarray(dates, dtype=np.float64)[list(sub)]
        out.append(ch)
    return out


def proposals(model, K, seed):
    from psoap_b200 import synthetic
    p = synthetic.default_params(model)
    rng = np.random.default_rng(seed)
    return np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])


def device_velocities(model, p, dates):
    """psoap_orbit_velocities on the device: [ncomp, n_dates]."""
    import torch
    L, lib = _lib()
    pd = torch.from_numpy(np.ascontiguousarray(p, dtype=np.float64)).cuda()
    dd = torch.from_numpy(np.ascontiguousarray(dates, dtype=np.float64)).cuda()
    vel = torch.empty((NCOMP[model], len(dates)), dtype=torch.float64, device="cuda")
    L.check(lib.psoap_orbit_velocities(L.MODELS[model], L.ptr(pd), L.ptr(dd), len(dates), L.ptr(vel), None,
                                       L.stream_ptr()))
    return vel.cpu().numpy()


def device_jacobian(model, p, dates):
    """psoap_orbit_jacobian on the device: [ncomp, n_dates, norb]."""
    import torch
    L, lib = _lib()
    pd = torch.from_numpy(np.ascontiguousarray(p[:NORB[model]], dtype=np.float64)).cuda()
    dd = torch.from_numpy(np.ascontiguousarray(dates, dtype=np.float64)).cuda()
    jac = torch.empty((NCOMP[model], len(dates), NORB[model]), dtype=torch.float64, device="cuda")
    L.check(lib.psoap_orbit_jacobian(L.MODELS[model], L.ptr(pd), L.ptr(dd), len(dates), L.ptr(jac), L.stream_ptr()))
    return jac.cpu().numpy()


def free_of(model, p, epochs):
    """The free vector [V, gp] at the orbit's device velocities for the registered vector p."""
    return np.concatenate([device_velocities(model, p, epochs).reshape(-1), p[NORB[model]:]])


def chain_matrix(model, p, epochs):
    """d(free vector) / d(registered vector): [ncomp Ng + 2 ncomp, norb + 2 ncomp]."""
    ncomp, norb = NCOMP[model], NORB[model]
    Ng = len(epochs)
    J = np.zeros((ncomp * Ng + 2 * ncomp, norb + 2 * ncomp))
    J[:ncomp * Ng, :norb] = device_jacobian(model, p, epochs).reshape(ncomp * Ng, norb)
    J[ncomp * Ng:, norb:] = np.eye(2 * ncomp)
    return J


# Chunks of the GPU tests: 4 global epochs seen by every chunk in part, one epoch seen by one chunk only, and a chunk
# with 9 epochs (18 or 27 velocities: its Fisher matrix takes the blocked contraction, the 4-epoch ones the other).
DATES = np.array([1.5, 4.0, 7.25, 9.0, 12.5, 15.0, 20.0, 22.5, 30.0, 41.0])
SUBSETS = [(0, 1, 2, 3), (2, 3, 4, 5), (1, 3, 5, 6, 7, 8, 9, 0, 4)]


# ---------------------------------------------------------------------------------------------- CPU
def test_epoch_maps_of_overlapping_and_disjoint_dates():
    from psoap_b200.farm import epoch_maps, free_index, global_epochs
    over = [np.array([3.0, 1.0, 2.0]), np.array([2.0, 5.0]), np.array([1.0, 5.0, 7.5])]
    ep = global_epochs(over)
    assert np.array_equal(ep, [1.0, 2.0, 3.0, 5.0, 7.5])
    maps = epoch_maps(over, ep)
    assert [m.tolist() for m in maps] == [[2, 0, 1], [1, 3], [0, 3, 4]]
    assert all(m.dtype == np.int32 for m in maps)
    disj = [np.array([10.0, 11.0]), np.array([1.0, 2.0, 3.0])]
    ep = global_epochs(disj)
    assert np.array_equal(ep, [1.0, 2.0, 3.0, 10.0, 11.0])
    assert [m.tolist() for m in epoch_maps(disj, ep)] == [[3, 4], [0, 1, 2]]
    # a chunk's own vector [v_0[e], v_1[e], gp] inside the farm's [v_0[0..5), v_1[0..5), gp]
    assert free_index(2, 5, [3, 4]).tolist() == [3, 4, 8, 9, 10, 11, 12, 13]


def test_epoch_map_validation():
    from psoap_b200.farm import epoch_maps
    with pytest.raises(ValueError, match="not in the global epoch list"):
        epoch_maps([np.array([1.0, 2.5])], np.array([1.0, 2.0, 3.0]))
    with pytest.raises(ValueError, match="not in the global epoch list"):
        epoch_maps([np.array([9.0])], np.array([1.0, 2.0]))       # beyond the last epoch
    with pytest.raises(ValueError, match="twice"):
        epoch_maps([np.array([2.0, 2.0])], np.array([1.0, 2.0]))


def test_c_entries_take_the_free_ids_and_check_arguments():
    from psoap_b200 import _build
    _build.build_library()
    L, lib = _lib()
    for m, nc in ((6, 1), (7, 2), (8, 3)):
        assert lib.psoap_model_ncomp(m) == nc and lib.psoap_model_norb(m) == 0
    assert [lib.psoap_model_ncomp(m) for m in (1, 2, 3, 4, 5)] == [1, 2, 1, 2, 3]
    assert [lib.psoap_model_norb(m) for m in (1, 2, 3, 4, 5)] == [6, 7, 11, 12, 13]
    assert lib.psoap_model_ncomp(9) == 0 and lib.psoap_model_ncomp(0) == 0
    # the chunk workspaces grow with the chunk's own velocity count
    g = [lib.psoap_chunk_lnprob_grad_workspace_bytes(7, 1000, ne) for ne in (4, 20)]
    f = [lib.psoap_chunk_fisher_workspace_bytes(7, 1000, ne) for ne in (4, 20)]
    assert 0 < g[0] < g[1] and 0 < f[0] < f[1]
    Nn = 1024   # padded N: one N^2 product per parameter besides the gradient's 4 N^2 and its scratch
    assert (4 + 2 * 20 + 4) * 8 * Nn * Nn <= f[1] < (4 + 2 * 20 + 4 + 8) * 8 * Nn * Nn
    assert lib.psoap_chunk_fisher_workspace_bytes(9, 1000, 4) == 0
    N = (ctypes.c_int64 * 2)(100, 200)
    ne = (ctypes.c_int32 * 2)(3, 4)
    assert lib.psoap_farm_free_workspace_bytes(2, 6, 2, N, ne, 1, 2) > 0
    assert lib.psoap_farm_free_workspace_bytes(4, 6, 2, N, ne, 1, 2) == 0
    assert lib.psoap_farm_free_workspace_bytes(2, 0, 2, N, ne, 1, 2) == 0
    farm = L.vp(None)
    assert lib.psoap_farm_create_free(ctypes.byref(farm), 0, 6, 2, None, None, 1, 2, 1.0, None, 0) == -1
    assert b"psoap_farm_create_free" in lib.psoap_last_error()


class QuadraticFarm:
    """Stand-in for a free-velocity ChunkFarm: a gauge-invariant quadratic log-likelihood in the velocity differences
    v_c[e] - v_c[0] and the GP values, recording every vector it is asked about."""
    model = "SB2"
    free = True

    def __init__(self, Ng, seed):
        rng = np.random.default_rng(seed)
        self.epochs = np.arange(Ng, dtype=np.float64)
        self.Ng = Ng
        self.n_params = 2 * Ng + 4
        D = np.zeros((2 * (Ng - 1) + 4, self.n_params))
        for c in range(2):
            for e in range(1, Ng):
                D[c * (Ng - 1) + e - 1, c * Ng + e] = 1.0
                D[c * (Ng - 1) + e - 1, c * Ng] = -1.0
        D[2 * (Ng - 1):, 2 * Ng:] = np.eye(4)
        W = rng.uniform(0.5, 2.0, D.shape[0])
        self.H = D.T @ (W[:, None] * D)
        self.t = np.concatenate([rng.normal(0.0, 10.0, 2 * Ng), [0.1, 5.0, 0.05, 7.0]])
        self.seen = []

    def lnprob_and_grad(self, p):
        self.seen.append(np.array(p))
        r = p - self.t
        return -0.5 * r @ self.H @ r, -self.H @ r

    def fisher(self, p):
        return self.H


@pytest.mark.parametrize("ref_epoch", [0, 3])
@pytest.mark.parametrize("fix_gp", [False, True])
def test_fit_holds_the_gauge_entries(ref_epoch, fix_gp):
    from psoap_b200 import sample
    farm = QuadraticFarm(6, seed=ref_epoch)
    v0 = np.arange(12, dtype=np.float64).reshape(2, 6) * 0.5
    gp0 = np.array([0.2, 4.0, 0.1, 6.0])
    fit = sample.fit_epoch_velocities(farm, v0, gp0, ref_epoch=ref_epoch, fix_gp=fix_gp,
                                      options=dict(ftol=1e-15, gtol=1e-10))
    fixed = [ref_epoch, 6 + ref_epoch] + ([12, 13, 14, 15] if fix_gp else [])
    assert len(farm.seen) > 1
    for p in farm.seen:
        assert np.array_equal(p[fixed], np.concatenate([v0.reshape(-1), gp0])[fixed])
    assert np.array_equal(fit.v[:, ref_epoch], v0[:, ref_epoch])
    assert fit.sigma_v[0, ref_epoch] == 0.0 and fit.sigma_v[1, ref_epoch] == 0.0
    assert np.all(fit.sigma_v[:, [e for e in range(6) if e != ref_epoch]] > 0)
    assert fit.cov.shape == (len(fit.free), len(fit.free)) and not set(fixed) & set(fit.free.tolist())
    # the optimum: the targets' differences, shifted by the held reference velocity
    for c in range(2):
        want = farm.t[c * 6:(c + 1) * 6] - farm.t[c * 6 + ref_epoch] + v0[c, ref_epoch]
        assert np.allclose(fit.v[c], want, atol=1e-5)
    assert np.array_equal(fit.gp, gp0) if fix_gp else np.allclose(fit.gp, farm.t[12:], atol=1e-5)
    assert np.allclose(fit.cov, np.linalg.inv(farm.H[np.ix_(fit.free, fit.free)]))


def test_fit_arguments_are_checked():
    from psoap_b200 import sample
    farm = QuadraticFarm(4, seed=1)
    with pytest.raises(ValueError, match="v0 must be"):
        sample.fit_epoch_velocities(farm, np.zeros((2, 5)), [0.1, 5.0, 0.1, 5.0])
    with pytest.raises(ValueError, match="ref_epoch"):
        sample.fit_epoch_velocities(farm, np.zeros((2, 4)), [0.1, 5.0, 0.1, 5.0], ref_epoch=4)
    farm.free = False
    with pytest.raises(ValueError, match="free_velocities=True"):
        sample.fit_epoch_velocities(farm, np.zeros((2, 4)), [0.1, 5.0, 0.1, 5.0])


# ---------------------------------------------------------------------------------------------- GPU
def farm_pair(model, K, n_pix=(30, 40, 25), seed=11, **kw):
    from psoap_b200.farm import ChunkFarm
    chunks = chunks_on(model, DATES, SUBSETS, n_pix, seed)
    return (ChunkFarm(model, chunks, n_proposals=K, **kw),
            ChunkFarm(model, chunks, n_proposals=K, free_velocities=True, **kw), chunks)


@gpu
@pytest.mark.parametrize("model", ["SB2", "ST3"])
def test_free_mode_is_the_orbit_paths_bits(model):
    """Free vector at the orbit's device velocities: lnprob, the per-chunk records and the predicted components are the
    orbit farm's bits."""
    import torch
    K = 2
    orb, fre, chunks = farm_pair(model, K)
    assert np.array_equal(fre.epochs, DATES) and fre.n_params == NCOMP[model] * len(DATES) + 2 * NCOMP[model]
    P = proposals(model, K, seed=3)
    V = np.stack([free_of(model, p, fre.epochs) for p in P])
    assert np.array_equal(fre.lnprob_many(V), orb.lnprob_many(P))
    ro = orb.lnprob_device(torch.from_numpy(P).cuda()).clone()
    rf = fre.lnprob_device(torch.from_numpy(V).cuda()).clone()
    assert torch.isfinite(ro[..., 0]).all() and torch.equal(ro, rf)
    grids = [np.linspace(ch["lwl"].min(), ch["lwl"].max(), 37 + 5 * i) for i, ch in enumerate(chunks)]
    mus = [1.0] * NCOMP[model]
    for f in (orb, fre):
        f.attach_prediction_grids(grids, predict_nbranch=2)
    po, pf = orb.predict_components(P, mus), fre.predict_components(V, mus)
    for (mo, so), (mf, sf) in zip(po, pf):
        assert torch.equal(mo, mf) and torch.equal(so, sf)
    orb.close()
    fre.close()


def rel_err(a, b):
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


@gpu
@pytest.mark.parametrize("model", ["SB2", "ST3"])
def test_chain_rule_to_the_orbit_gradient_and_fisher(model):
    orb, fre, _ = farm_pair(model, 1)
    p = proposals(model, 1, seed=5)[0]
    v = free_of(model, p, fre.epochs)
    J = chain_matrix(model, p, fre.epochs)
    nv = NCOMP[model] * len(DATES)
    ro = orb.chunk_lnlike_grads_many(p[None]).cpu().numpy()[0]
    rf = fre.chunk_lnlike_grads_many(v[None]).cpu().numpy()[0]
    assert np.isfinite(ro).all() and np.isfinite(rf).all()
    assert np.array_equal(ro[:, 0], rf[:, 0])
    assert np.array_equal(ro[:, 1 + NORB[model]:], rf[:, 1 + nv:])          # GP entries, chunk by chunk
    g_orb, g_free = ro[:, 1:].sum(axis=0), rf[:, 1:].sum(axis=0)
    assert rel_err(J.T @ g_free, g_orb) <= 1e-12, rel_err(J.T @ g_free, g_orb)
    F_orb, F_free = orb.fisher(p), fre.fisher(v)
    assert np.array_equal(F_free, F_free.T)
    assert rel_err(J.T @ F_free @ J, F_orb) <= 1e-12, rel_err(J.T @ F_free @ J, F_orb)
    orb.close()
    fre.close()


@gpu
def test_velocity_gradient_matches_oracle_differences():
    """d lnlike / d v_c[g] of every global epoch against differences of the CPU oracle's likelihood (the reference's
    replicate_wls shift and dense Cholesky).  The oracle's lnlike carries rounding noise of about cond(K) eps |quad|
    (1e-8 here, quad ~ 1e4), which a two-point difference at a step small enough for its truncation error divides by
    the step.  So the derivative is taken from a least-squares quartic through 11 points v_k + j h, |j| <= 5,
    h = 2e-3 km/s: the spectra vary on the scale of a line width (2 - 4 pixels of 2.8 km/s), so the quintic term left
    out is below 1e-12 of the gradient, and the fit's residuals measure the noise.  The error allowed is five standard
    errors of the fitted slope, and at least 1e-9 of the largest velocity gradient."""
    from oracle import oracle as orc
    from psoap_b200.farm import ChunkFarm
    model = "SB2"
    chunks = chunks_on(model, DATES, SUBSETS, (30, 40, 25), seed=21)
    farm = ChunkFarm(model, chunks, free_velocities=True)
    p = proposals(model, 1, seed=7)[0]
    v = free_of(model, p, farm.epochs)
    Ng, nv = len(DATES), 2 * len(DATES)
    _, g = farm.lnprob_and_grad(v)
    maps = [np.searchsorted(DATES, ch["date1D"]) for ch in chunks]

    def lnl(q):
        V = q[:nv].reshape(2, Ng)
        tot = 0.0
        for ch, m in zip(chunks, maps):
            N = len(ch["fl"])
            lw = [ch["lwl"] - V[c][m][ch["epoch"]] / C_KMS for c in range(2)]
            tot += orc.lnlike_f_g(np.empty((N, N)), lw[0], lw[1], ch["fl"], ch["sigma"], *q[nv:], mu_GP=farm.mu_GP)
        return tot

    l0 = lnl(v)
    assert abs(l0 - farm.lnprob(v)) <= 1e-9 * abs(l0)
    h = 2e-3
    j = np.arange(-5, 6, dtype=np.float64)
    A = np.vander(j, 5, increasing=True)                  # 1, j, .., j^4
    AtA_inv = np.linalg.inv(A.T @ A)
    floor = 1e-9 * np.max(np.abs(g[:nv]))
    for k in range(nv):
        y = np.empty(len(j))
        for n, jj in enumerate(j):
            q = v.copy()
            q[k] += jj * h
            y[n] = lnl(q)
        y -= l0
        coef, *_ = np.linalg.lstsq(A, y, rcond=None)
        res = y - A @ coef
        se = np.sqrt(res @ res / (len(j) - 5) * AtA_inv[1, 1]) / h
        d = coef[1] / h
        assert abs(g[k] - d) <= max(5 * se, floor), (k, g[k], d, se)
    farm.close()


@gpu
@pytest.mark.parametrize("model", ["SB2", "ST3"])
def test_gauge_identities(model):
    from psoap_b200.farm import ChunkFarm
    chunks = chunks_on(model, DATES, SUBSETS, (30, 40, 25), seed=31)
    farm = ChunkFarm(model, chunks, free_velocities=True)
    ncomp, Ng = NCOMP[model], len(DATES)
    v = free_of(model, proposals(model, 1, seed=2)[0], farm.epochs)
    _, g = farm.lnprob_and_grad(v)
    F = farm.fisher(v)
    for c in range(ncomp):
        blk = slice(c * Ng, (c + 1) * Ng)
        assert abs(np.sum(g[blk])) <= 1e-9 * np.linalg.norm(g), (c, np.sum(g[blk]), np.linalg.norm(g))
        rows = np.sum(F[:, blk], axis=1)
        assert np.max(np.abs(rows)) <= 1e-9 * np.max(np.abs(F)), (c, np.max(np.abs(rows)), np.max(np.abs(F)))
    # the same per chunk, where the gauge holds for each chunk's own velocities
    for r, ch in zip(farm.chunk_lnlike_grads(v).cpu().numpy(), chunks):
        for c in range(ncomp):
            assert abs(np.sum(r[1 + c * Ng:1 + (c + 1) * Ng])) <= 1e-9 * np.linalg.norm(r[1:])
    farm.close()


@gpu
def test_rows_scatter_to_the_observed_epochs_and_match_the_chunk_entry():
    """Fewer than 8 (proposal, chunk) pairs: the gradient graph runs the direct API's launch plan, so the farm's rows are
    the bits of one psoap_chunk_lnprob_grad call per chunk on its own velocities (ChunkFarm.chunk_lnlike_grads)."""
    import torch
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    model, K = "SB2", 2
    chunks = chunks_on(model, DATES, SUBSETS, (30, 40, 25), seed=41)
    farm = ChunkFarm(model, chunks, n_proposals=K, free_velocities=True)
    Ng = len(DATES)
    V = np.stack([free_of(model, p, farm.epochs) for p in proposals(model, K, seed=9)])
    rows = farm.chunk_lnlike_grads_many(V).cpu().numpy()
    assert np.isfinite(rows).all()
    for i, sub in enumerate(SUBSETS):
        seen = np.zeros(Ng, dtype=bool)
        seen[list(sub)] = True
        for c in range(2):
            blk = rows[:, i, 1 + c * Ng:1 + (c + 1) * Ng]
            assert np.all(blk[:, ~seen] == 0.0) and not np.signbit(blk[:, ~seen]).any()
            assert np.all(blk[:, seen] != 0.0)
    for k in range(K):
        assert np.array_equal(rows[k], farm.chunk_lnlike_grads(V[k]).cpu().numpy())
    # and the chunk entry directly, on the chunk's own vector [v_0[e], v_1[e], gp] (PSOAP_FREE2)
    ch = chunks[1]
    m = np.searchsorted(DATES, ch["date1D"])
    loc = np.concatenate([V[0, :Ng][m], V[0, Ng:2 * Ng][m], V[0, 2 * Ng:]])
    k1 = farm.mine.index(1)
    d = farm._descs[k1]
    nbytes = lib.psoap_chunk_lnprob_grad_workspace_bytes(7, d.N, d.n_epochs)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    gl = torch.empty(loc.size, dtype=torch.float64, device="cuda")
    L.check(lib.psoap_chunk_lnprob_grad(7, ctypes.byref(d), L.ptr(torch.from_numpy(loc).cuda()), farm.mu_GP, L.ptr(ws),
                                        nbytes, L.ptr(res), L.ptr(gl), L.stream_ptr()))
    gl = gl.cpu().numpy()
    assert res[0].item() == rows[0, 1, 0]
    assert np.array_equal(gl[:len(m)], rows[0, 1, 1 + m]) and np.array_equal(gl[len(m):2 * len(m)], rows[0, 1, 1 + Ng + m])
    assert np.array_equal(gl[2 * len(m):], rows[0, 1, 1 + 2 * Ng:])
    farm.close()


@gpu
def test_a_bad_velocity_touches_only_its_items():
    """|v| >= c at an epoch only chunk 2 observes: that item is -inf with a NaN row, every other item (the same proposal's
    other chunks included) keeps the bits it has in an all-valid batch; likewise a negative GP value for all chunks."""
    model, K = "SB2", 4
    from psoap_b200.farm import ChunkFarm
    chunks = chunks_on(model, DATES, SUBSETS, (30, 40, 25), seed=51)
    farm = ChunkFarm(model, chunks, n_proposals=K, free_velocities=True, grad_nbranch=1)
    Ng = len(DATES)
    good = np.stack([free_of(model, p, farm.epochs) for p in proposals(model, K, seed=4)])
    bad = good.copy()
    only2 = 8                       # observed by chunk 2 alone
    assert [only2 in s for s in SUBSETS] == [False, False, True]
    bad[1, Ng + only2] = 3.1e5      # v_1 beyond c
    bad[2, 2 * Ng] = -0.1           # amp_f < 0
    rb, rg = farm.chunk_lnlike_grads_many(bad).cpu().numpy(), farm.chunk_lnlike_grads_many(good).cpu().numpy()
    lb, lg = farm.chunk_lnlikes(bad).cpu().numpy(), farm.chunk_lnlikes(good).cpu().numpy()
    assert np.isfinite(rg).all()
    assert rb[1, 2, 0] == -np.inf and np.isnan(rb[1, 2, 1:]).all() and lb[1, 2] == -np.inf
    assert np.array_equal(rb[1, :2], rg[1, :2]) and np.array_equal(lb[1, :2], lg[1, :2])
    assert np.all(rb[2, :, 0] == -np.inf) and np.isnan(rb[2, :, 1:]).all() and np.all(lb[2] == -np.inf)
    for k in (0, 3):
        assert np.array_equal(rb[k], rg[k]) and np.array_equal(lb[k], lg[k])
    # the sequential path writes the same -inf and NaN row
    seq = farm.chunk_lnlike_grads(bad[1]).cpu().numpy()
    assert seq[2, 0] == -np.inf and np.isnan(seq[2, 1:]).all() and np.isfinite(seq[:2]).all()
    farm.close()


@gpu
def test_rows_are_bit_stable_across_calls_branches_and_ranks():
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    model, K = "SB2", 2
    subsets = [(0, 1, 2, 3), (2, 3, 4, 5), (1, 3, 5, 6), (0, 4, 7, 8), (5, 6, 7, 8, 9), (0, 9)]
    chunks = chunks_on(model, DATES, subsets, [40 + 35 * i for i in range(6)], seed=61)
    single = ChunkFarm(model, chunks, n_proposals=K, free_velocities=True, grad_nbranch=8)
    V = np.stack([free_of(model, p, single.epochs) for p in proposals(model, K, seed=8)])
    ref = single.chunk_lnlike_grads_many(V).cpu().numpy()
    assert np.isfinite(ref).all()
    assert np.array_equal(single.chunk_lnlike_grads_many(V).cpu().numpy(), ref)
    other = ChunkFarm(model, chunks, n_proposals=K, free_velocities=True, grad_nbranch=3)
    assert np.array_equal(other.chunk_lnlike_grads_many(V).cpu().numpy(), ref)
    other.close()
    total = np.zeros_like(ref)
    for r in range(2):
        f = ChunkFarm(model, chunks, n_proposals=K, rank=r, world_size=2, free_velocities=True)
        f.world_size = 1  # no process group here: take the un-reduced rows
        assert np.array_equal(f.epochs, single.epochs)
        rows = f.chunk_lnlike_grads_many(V).cpu().numpy()
        for i in f.mine:
            assert np.array_equal(rows[:, i], ref[:, i])
        total = total + rows
        f.close()
    assert np.array_equal(total, ref)
    single.close()


@gpu
def test_fit_recovers_synthetic_sb2_velocities():
    """One SB2 chunk made from known per-epoch velocities: the fit, started 1.5 km/s off with each component's first
    epoch held at its true value (the gauge), lands within 4 Cramer-Rao sigma of the truth at every epoch."""
    from psoap_b200 import sample, synthetic
    from psoap_b200.farm import ChunkFarm
    ch = synthetic.make_chunk("SB2", 8, 400, seed=71)
    truth = synthetic.host_velocities("SB2", synthetic.ORBIT_PARAMS["SB2"], ch["date1D"])
    farm = ChunkFarm("SB2", [ch], free_velocities=True)
    rng = np.random.default_rng(3)
    v0 = truth + rng.uniform(-1.5, 1.5, truth.shape)
    v0[:, 0] = truth[:, 0]
    fit = sample.fit_epoch_velocities(farm, v0, synthetic.GP_PARAMS["SB2"], ref_epoch=0)
    assert fit.opt.success, fit.opt.message
    pull = (fit.v - truth)[:, 1:] / fit.sigma_v[:, 1:]
    assert np.all(np.abs(pull) < 4.0), pull
    assert np.array_equal(fit.v[:, 0], truth[:, 0])
    farm.close()


@gpu
def test_sb1_wrapper():
    from psoap_b200 import sample, synthetic
    chunks = [synthetic.make_chunk("SB1", 6, 150, seed=81)]
    truth = synthetic.host_velocities("SB1", synthetic.ORBIT_PARAMS["SB1"], chunks[0]["date1D"])[0]
    fit = sample.fit_sb1_epoch_velocities(chunks, truth + 0.5 * (np.arange(6) > 0), 0.1, 5.0, fix_gp=True)
    assert fit.v.shape == (1, 6) and np.array_equal(fit.gp, [0.1, 5.0]) and fit.cov.shape == (5, 5)
    assert np.all(np.abs(fit.v[0, 1:] - truth[1:]) < 4.0 * fit.sigma_v[0, 1:])
