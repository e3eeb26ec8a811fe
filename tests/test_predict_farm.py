"""The farm's prediction graph (psoap_farm_predict_attach / psoap_farm_predict, ChunkFarm.attach_prediction_grids and
predict_components): the component spectra of every (proposal, chunk) item, psoap_predict mode 0 on the chunk's resident
pixels shifted by the proposal's velocities, in one graph launch.

The lone psoap_predict call on the same pixels, shifted on the host from the device velocities, is the exact reference:
under launch switches that give both paths one plan the outputs are the same bits.  The oracle's predict_f / _f_g /
_f_g_h on epoch-major pixels is the parity reference.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NORB = {"SB1": 6, "SB2": 7, "ST1": 11, "ST2": 12, "ST3": 13}
NCOMP = {"SB1": 1, "SB2": 2, "ST1": 1, "ST2": 2, "ST3": 3}
C_KMS = 2.99792458e5
gpu = pytest.mark.gpu
EXACT_ENV = {"PSOAP_POTRF": "3", "PSOAP_GROUP": "4", "PSOAP_LOOKAHEAD": "0", "PSOAP_FARM_LOOKAHEAD": "0"}


def _lib():
    from psoap_b200 import _lib as L
    return L, L.load()


def proposals(model, K, seed):
    from psoap_b200 import synthetic
    p = synthetic.default_params(model)
    rng = np.random.default_rng(seed)
    return np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])


def grid_of(ch, m):
    """m rest-frame ln-wavelength points over the chunk's range (not on the pixels)."""
    lo, hi = ch["lwl"].min(), ch["lwl"].max()
    return lo + (hi - lo) * (np.arange(m) + 0.37) / m


def mus_of(model):
    return np.linspace(0.4, 0.6, NCOMP[model])


def run_child(*args, env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__)] + list(args), env=env, capture_output=True,
                       text=True, timeout=1500)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def raw_predict(farm, P):
    """One psoap_farm_predict call on this rank's items: (delta, sigma, results [K, n_mine, 4], offsets [2, nitems + 1])
    as numpy arrays."""
    import torch
    L, lib = _lib()
    off = farm._pred["off"]
    K = farm.n_proposals
    p = torch.from_numpy(np.ascontiguousarray(P, dtype=np.float64)).cuda()
    d = torch.full((max(1, int(off[0, -1])),), 7.0, dtype=torch.float64, device="cuda")
    s = torch.full((max(1, int(off[1, -1])),), 7.0, dtype=torch.float64, device="cuda")
    r = torch.empty((K, len(farm.mine), 4), dtype=torch.float64, device="cuda")
    L.check(lib.psoap_farm_predict(farm._farm, L.ptr(p), L.ptr(d), L.ptr(s), L.ptr(r), L.stream_ptr()))
    return d.cpu().numpy(), s.cpu().numpy(), r.cpu().numpy(), off


# ---------------------------------------------------------------------------------------------- CPU
def test_predict_entries_reject_a_null_farm():
    from psoap_b200 import _build
    _build.build_library()
    L, lib = _lib()
    assert lib.psoap_version() >= 104
    m = (ctypes.c_int64 * 2)(10, 20)
    assert lib.psoap_farm_predict_workspace_bytes(None, 4, m, 0) == 0
    off = (ctypes.c_int64 * 8)()
    assert lib.psoap_farm_predict_attach(None, 4, m, None, 0, None, 0, off) == -1
    assert b"psoap_farm_predict_attach" in lib.psoap_last_error()
    assert lib.psoap_farm_predict(None, None, None, None, None, None) == -1
    assert b"psoap_farm_predict" in lib.psoap_last_error()
    assert lib.psoap_launch_count() == 0


def test_prediction_grids_are_checked():
    from psoap_b200.farm import prediction_grids
    g = np.linspace(8.5, 8.6, 7)
    out = prediction_grids([g, np.zeros(0)], [40, 0], 2)
    assert out[0].shape == (2, 7) and np.array_equal(out[0][1], g) and out[1].shape == (2, 0)
    two = np.stack([g, g + 1e-4])
    assert np.array_equal(prediction_grids([two], [5], 2)[0], two)
    with pytest.raises(ValueError, match="one prediction grid per chunk"):
        prediction_grids([g], [40, 30], 2)
    with pytest.raises(ValueError, match="chunk 0"):
        prediction_grids([np.stack([g, g, g])], [40], 2)
    with pytest.raises(ValueError, match="chunk 0"):
        prediction_grids([np.zeros((2, 2, 2))], [40], 2)
    bad = g.copy()
    bad[3] = np.nan
    with pytest.raises(ValueError, match="non-finite"):
        prediction_grids([g, bad], [40, 30], 1)
    with pytest.raises(ValueError, match="no pixels"):
        prediction_grids([g, g], [40, 0], 1)


def _bare_farm():
    """A ChunkFarm with only the host attributes the argument checks read (no device needed)."""
    from psoap_b200.farm import ChunkFarm
    f = ChunkFarm.__new__(ChunkFarm)
    f.model, f.n_chunks, f.n_proposals, f.n_params = "SB2", 2, 2, 11
    f._n_pix, f._pred, f.mine, f._farm = [40, 0], None, [0], None
    return f


def test_method_arguments_are_checked():
    f = _bare_farm()
    g = np.linspace(8.5, 8.6, 7)
    with pytest.raises(ValueError, match="sigma"):
        f.attach_prediction_grids([g, []], sigma="upper")
    with pytest.raises(ValueError, match="predict_nbranch"):
        f.attach_prediction_grids([g, []], predict_nbranch=0)
    with pytest.raises(ValueError, match="no pixels"):
        f.attach_prediction_grids([g, g])
    with pytest.raises(ValueError, match="one prediction grid per chunk"):
        f.attach_prediction_grids([g])
    P = np.zeros((2, 11))
    with pytest.raises(ValueError, match="P must hold"):
        f.predict_components(P[:1], [0.5, 0.5])
    with pytest.raises(ValueError, match="mus"):
        f.predict_components(P, [0.5])
    with pytest.raises(RuntimeError, match="attach_prediction_grids"):
        f.predict_components(P, [0.5, 0.5])
    f._pred = {}
    with pytest.raises(RuntimeError, match="already attached"):
        f.attach_prediction_grids([g, []])


def test_combine_predictions_is_the_law_of_total_variance():
    from psoap_b200.farm import combine_predictions
    rng = np.random.default_rng(11)
    for K, M in ((1, 5), (8, 300), (3, 1)):
        mu = rng.normal(1.0, 0.1, (K, M))
        var = rng.uniform(0.0, 1e-3, (K, M))
        mean, v = combine_predictions(mu, var)
        assert np.allclose(mean, mu.mean(axis=0), rtol=1e-14, atol=0)
        assert np.allclose(v, var.mean(axis=0) + mu.var(axis=0), rtol=1e-12, atol=1e-18)
        m2, v2 = combine_predictions(mu, var)
        assert np.array_equal(mean, m2) and np.array_equal(v, v2)


# ---------------------------------------------------------------------------------------------- GPU
def _chunks(model, n_pix, seed, n_epochs=4, **kw):
    from psoap_b200 import synthetic
    return [synthetic.make_chunk(model, n_epochs, n, seed=seed + i, wl0=5000.0 + 3.0 * i, **kw) for i, n in enumerate(n_pix)]


@gpu
def test_attach_arguments_and_workspace_size():
    import torch
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    chunks = _chunks("SB2", [40, 70, 100], seed=510)
    farm = ChunkFarm("SB2", chunks, n_proposals=2)
    f = farm._farm
    m = (ctypes.c_int64 * 3)(50, 90, 0)
    grids = [torch.from_numpy(np.tile(grid_of(ch, 90), 2)).cuda() for ch in chunks]
    ptrs = (L.vp * 6)(*[L.vp(grids[i // 2].data_ptr() + (i % 2) * 90 * 8) for i in range(6)])
    sizes = [lib.psoap_farm_predict_workspace_bytes(f, nb, m, 0) for nb in (1, 2, 4)]
    assert all(a < b for a, b in zip(sizes, sizes[1:])), sizes
    assert lib.psoap_farm_predict_workspace_bytes(f, 4, m, 1) < sizes[2]
    assert lib.psoap_farm_predict_workspace_bytes(f, 0, m, 0) == 0
    assert lib.psoap_farm_predict_workspace_bytes(f, 2, m, 2) == 0
    assert lib.psoap_farm_predict_workspace_bytes(f, 2, (ctypes.c_int64 * 3)(50, -1, 0), 0) == 0
    ws = torch.empty(sizes[1] + 512, dtype=torch.uint8, device="cuda")
    off = (ctypes.c_int64 * (2 * 7))()
    P = torch.from_numpy(proposals("SB2", 2, 1)).cuda()
    out = torch.empty(10 ** 6, dtype=torch.float64, device="cuda")
    res = torch.empty((2, 3, 4), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    n0 = lib.psoap_launch_count()
    assert lib.psoap_farm_predict(f, L.ptr(P), L.ptr(out), L.ptr(out), L.ptr(res), L.stream_ptr()) == -1   # before attach
    assert lib.psoap_farm_predict_attach(f, 2, (ctypes.c_int64 * 3)(50, -1, 0), ptrs, 0, L.ptr(ws), sizes[1], off) == -1
    assert lib.psoap_farm_predict_attach(f, 2, m, ptrs, 3, L.ptr(ws), sizes[1], off) == -1
    assert lib.psoap_farm_predict_attach(f, 2, m, None, 0, L.ptr(ws), sizes[1], off) == -1
    nullg = (L.vp * 6)(*([ptrs[0], None] + list(ptrs[2:])))
    assert lib.psoap_farm_predict_attach(f, 2, m, nullg, 0, L.ptr(ws), sizes[1], off) == -1
    assert lib.psoap_farm_predict_attach(f, 2, m, ptrs, 0, L.ptr(ws), sizes[1] - 1, off) == -3
    assert lib.psoap_farm_predict_attach(f, 2, m, ptrs, 0, L.vp(ws.data_ptr() + 8), sizes[1], off) == -3
    assert lib.psoap_launch_count() == n0
    assert lib.psoap_farm_predict_attach(f, 2, m, ptrs, 0, L.ptr(ws), sizes[1], off) == 0
    assert lib.psoap_farm_predict_attach(f, 2, m, ptrs, 0, L.ptr(ws), sizes[1], off) == -1   # one prediction graph per farm
    o = np.frombuffer(off, dtype=np.int64).reshape(2, 7)
    # chunk after chunk, proposals side by side; item = proposal * 3 + chunk
    assert list(o[0]) == [0, 200, 560, 100, 380, 560, 560]
    assert list(o[1]) == [0, 2 * 100 ** 2, 2 * 100 ** 2 + 2 * 180 ** 2, 100 ** 2, 2 * 100 ** 2 + 180 ** 2] + [o[1, 6]] * 2
    L.check(lib.psoap_farm_predict(f, L.ptr(P), L.ptr(out), L.ptr(out[600:]), L.ptr(res), L.stream_ptr()))
    torch.cuda.synchronize()
    assert lib.psoap_launch_count() > n0
    farm.close()


def exact_case(model, K):
    """Graph outputs == lone psoap_predict calls on the farm's wavelength-sorted pixels shifted on the host from the
    device velocities (run in a child process under EXACT_ENV).  At least 8 items, so that the farm's chain from
    psoap_chunk.reserved is 3 like the lone call's.  Chunks of 1 to 6 row blocks; m not a multiple of 128, and M
    crossing a tile boundary."""
    import torch
    from psoap_b200 import covariance
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    n_pix = [30, 60, 95, 130, 160, 190, 45, 110]     # x 4 epochs: N = 120 .. 760
    nch = 8 if K == 1 else 3
    chunks = _chunks(model, n_pix[:nch], seed=700, mask_frac=0.02)
    blocks = sorted({(len(ch["fl"]) + 127) // 128 for ch in chunks})
    assert blocks[0] == 1 and (K > 1 or blocks[-1] == 6), blocks
    ncomp, norb = NCOMP[model], NORB[model]
    ms = [45 + 47 * i for i in range(nch)]
    assert any(ncomp * m > 128 for m in ms) and all(m % 128 for m in ms)
    grids = [np.stack([grid_of(ch, m) + 2e-5 * c for c in range(ncomp)]) for ch, m in zip(chunks, ms)]
    farm = ChunkFarm(model, chunks, n_proposals=K)
    farm.attach_prediction_grids(grids, predict_nbranch=3)
    P = proposals(model, K, seed=K)
    mus = mus_of(model)
    got = farm.predict_components(P, mus)
    for k in range(K):
        p = torch.from_numpy(P[k].copy()).cuda()
        for i, ch in enumerate(chunks):
            order = np.argsort(ch["lwl"], kind="stable")
            lwl, fl, sg, ep = (np.ascontiguousarray(ch[key][order]) for key in ("lwl", "fl", "sigma", "epoch"))
            dates = torch.from_numpy(ch["date1D"].copy()).cuda()
            vel = torch.empty((ncomp, len(ch["date1D"])), dtype=torch.float64, device="cuda")
            L.check(lib.psoap_orbit_velocities(L.MODELS[model], L.ptr(p), L.ptr(dates), len(ch["date1D"]), L.ptr(vel),
                                               None, L.stream_ptr()))
            v = vel.cpu().numpy()
            lw = [torch.from_numpy(lwl + (-v[c][ep]) / C_KMS).cuda() for c in range(ncomp)]
            lp = [torch.from_numpy(grids[i][c].copy()).cuda() for c in range(ncomp)]
            Sigma, delta = covariance._predict_device(0, lw, torch.from_numpy(fl).cuda(), torch.from_numpy(sg).cuda(),
                                                      lp, list(P[k, norb::2]), list(P[k, norb + 1::2]), farm.mu_GP)
            mu = delta + torch.from_numpy(np.repeat(mus, ms[i])).cuda()
            assert torch.equal(got[i][0][k], mu), (k, i, (got[i][0][k] - mu).abs().max().item())
            assert torch.equal(got[i][1][k], Sigma), (k, i, (got[i][1][k] - Sigma).abs().max().item())
    farm.close()


@gpu
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_graph_outputs_equal_lone_predict_calls(model, K):
    run_child("exact", model, str(K), env_extra=EXACT_ENV)


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_parity_with_the_oracle_at_c4_sizes(model):
    """mu and Sigma against the oracle's predict_f / _f_g / _f_g_h on epoch-major pixels and the oracle's velocities,
    within 1e-10 of the terms' scale; the results' lnlike column against the likelihood graph's within 1e-12."""
    from oracle import oracle as orc
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    n_pix = [100, 300] if model == "SB2" else [100]
    chunks = [synthetic.make_chunk(model, 20, n, seed=4100 + n, wl0=5000.0 + n) for n in n_pix]
    ncomp, norb = NCOMP[model], NORB[model]
    p = synthetic.default_params(model)
    ms = [2 * n for n in n_pix]
    grids = [grid_of(ch, m) for ch, m in zip(chunks, ms)]
    farm = ChunkFarm(model, chunks)
    farm.attach_prediction_grids(grids)
    mus = mus_of(model)
    got = farm.predict_components(p[None], mus)
    _, _, res, _ = raw_predict(farm, p[None])
    lnl = np.asarray(farm.chunk_lnlikes(p).cpu().numpy()).reshape(-1)
    assert np.all(np.abs(res[0, :, 0] - lnl) <= 1e-12 * np.abs(lnl)), (res[0, :, 0], lnl)
    amps, ls = p[norb::2], p[norb + 1::2]
    for i, ch in enumerate(chunks):
        vel = orc.get_velocities(model, p[:norb], ch["date1D"])
        lw = orc.replicate_wls(ch["lwl"], vel, ch["mask"])
        if ncomp == 1:
            # the oracle's predict_f takes mu_GP for both the mean and the residual; the farm's residual mean is mu_GP = 1
            mu_r, S_r = orc.predict_f(lw[0], ch["fl"], ch["sigma"], grids[i], amps[0], ls[0], mu_GP=1.0)
            mu_r = mu_r - 1.0 + mus[0]
        elif ncomp == 2:
            mu_r, S_r = orc.predict_f_g(lw[0], lw[1], ch["fl"], ch["sigma"], grids[i], grids[i], mus[0], amps[0], ls[0],
                                        mus[1], amps[1], ls[1])
        else:
            mu_r, S_r = orc.predict_f_g_h(lw[0], lw[1], lw[2], ch["fl"], ch["sigma"], grids[i], grids[i], grids[i],
                                          *mus, amps[0], ls[0], amps[1], ls[1], amps[2], ls[2])
        mu, S = got[i][0][0].cpu().numpy(), got[i][1][0].cpu().numpy()
        scale = float(np.max(amps ** 2))
        assert np.max(np.abs(S - S_r)) <= 1e-10 * scale, np.max(np.abs(S - S_r)) / scale
        assert np.max(np.abs(mu - mu_r)) <= 1e-10 * max(scale, np.max(np.abs(mu_r))), np.max(np.abs(mu - mu_r))
    farm.close()


@gpu
def test_diag_is_the_diagonal_of_full():
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [50, 90, 130], seed=900)
    grids = [grid_of(ch, 60 + 20 * i) for i, ch in enumerate(chunks)]
    P = proposals("SB2", 2, seed=3)
    full = ChunkFarm("SB2", chunks, n_proposals=2)
    full.attach_prediction_grids(grids, sigma="full")
    diag = ChunkFarm("SB2", chunks, n_proposals=2)
    diag.attach_prediction_grids(grids, sigma="diag")
    a, b = full.predict_components(P, [0.5, 0.5]), diag.predict_components(P, [0.5, 0.5])
    for (mu_f, S), (mu_d, v) in zip(a, b):
        assert v.shape == mu_d.shape == (2, S.shape[1])
        assert np.array_equal(mu_f.cpu().numpy(), mu_d.cpu().numpy())
        assert np.array_equal(np.diagonal(S.cpu().numpy(), axis1=1, axis2=2), v.cpu().numpy())
    full.close()
    diag.close()


def _np(outs):
    return [(mu.cpu().numpy(), S.cpu().numpy()) for mu, S in outs]


@gpu
def test_outputs_are_bit_stable_across_calls_branches_and_ranks():
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [40 + 35 * i for i in range(9)], seed=300)   # N = 160 .. 1280
    grids = [grid_of(ch, 50 + 13 * i) for i, ch in enumerate(chunks)]
    K = 2
    P = proposals("SB2", K, seed=9)
    mus = [0.45, 0.55]
    single = ChunkFarm("SB2", chunks, n_proposals=K)
    single.attach_prediction_grids(grids, predict_nbranch=4)
    ref = _np(single.predict_components(P, mus))
    assert all(np.isfinite(mu).all() and np.isfinite(S).all() for mu, S in ref)
    again = _np(single.predict_components(P, mus))
    assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(ref, again))
    other = ChunkFarm("SB2", chunks, n_proposals=K)
    other.attach_prediction_grids(grids, predict_nbranch=16)
    o = _np(other.predict_components(P, mus))
    assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(ref, o))
    other.close()
    for world in (2, 4):
        seen = set()
        for r in range(world):
            f = ChunkFarm("SB2", chunks, n_proposals=K, rank=r, world_size=world)
            f.world_size = 1   # no process group here: take the un-reduced buffers
            f.attach_prediction_grids(grids, predict_nbranch=4)
            outs = _np(f.predict_components(P, mus))
            for i in f.mine:
                assert np.array_equal(outs[i][0], ref[i][0]) and np.array_equal(outs[i][1], ref[i][1])
                seen.add(i)
            for i in set(range(len(chunks))) - set(f.mine):
                assert not outs[i][1].any()   # other ranks' entries are zero before the all-reduce
            f.close()
        assert seen == set(range(len(chunks)))
    single.close()


@gpu
def test_a_bad_proposal_gives_nan_for_that_proposal_only():
    """|v| >= c in proposal 1 and an empty chunk with m = 0: proposal 1's outputs are NaN, the others' the bits of an
    all-valid batch, and predict_components names the proposal."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [50, 90], seed=90)
    empty = synthetic.make_chunk("SB2", 4, 30, seed=99)
    empty["mask"][:] = False
    for key in ("lwl", "fl", "sigma", "epoch"):
        empty[key] = empty[key][:0]
    chunks.insert(1, empty)
    grids = [grid_of(chunks[0], 70), np.zeros(0), grid_of(chunks[2], 40)]
    P = proposals("SB2", 3, seed=2)
    bad = P.copy()
    bad[1, 1] = 4e5
    farm = ChunkFarm("SB2", chunks, n_proposals=3, nbranch=1)
    farm.attach_prediction_grids(grids, predict_nbranch=1)
    dg, sg, rg, off = raw_predict(farm, P)
    db, sb, rb, _ = raw_predict(farm, bad)
    nch = len(farm.mine)
    for k in range(3):
        for c in range(nch):
            if k == 1:
                assert rb[k, c, 0] == -np.inf and rb[k, c, 3] == 0
            else:
                assert np.array_equal(rb[k, c], rg[k, c])
    # per chunk, proposal k's block of delta and Sigma
    for c, i in enumerate(farm.mine):
        M = 2 * (70 if i == 0 else 40)
        for k in range(3):
            it = k * nch + c
            d, s = slice(off[0, it], off[0, it] + M), slice(off[1, it], off[1, it] + M * M)
            if k == 1:
                assert np.isnan(db[d]).all() and np.isnan(sb[s]).all()
            else:
                assert np.isfinite(dg[d]).all() and np.array_equal(db[d], dg[d]) and np.array_equal(sb[s], sg[s])
    with pytest.raises(ValueError, match="proposal 1, chunk 0"):
        farm.predict_components(bad, [0.5, 0.5])
    out = farm.predict_components(P, [0.5, 0.5])
    assert out[1][0].shape == (3, 0) and out[1][1].shape == (3, 0, 0)
    farm.close()


@gpu
def test_the_other_graphs_are_untouched():
    import torch
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [50 + 30 * i for i in range(5)], seed=120)
    P = proposals("SB2", 2, seed=8)
    farm = ChunkFarm("SB2", chunks, n_proposals=2)
    torch.cuda.synchronize()
    mem = torch.cuda.memory_allocated()
    farm.lnprob_many(P)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == mem and farm._pred is None
    launches = farm.launches_per_eval
    lnl = farm.chunk_lnlikes(P).cpu().numpy()
    rows = farm.chunk_lnlike_grads_many(P).cpu().numpy()
    farm.attach_prediction_grids([grid_of(ch, 64) for ch in chunks])
    farm.predict_components(P, [0.5, 0.5])
    assert np.array_equal(farm.chunk_lnlikes(P).cpu().numpy(), lnl)
    assert np.array_equal(farm.chunk_lnlike_grads_many(P).cpu().numpy(), rows)
    L, lib = _lib()
    assert farm.launches_per_eval == launches == lib.psoap_farm_launches_per_eval(farm._farm)
    farm.close()


if __name__ == "__main__":
    if sys.argv[1] == "exact":
        exact_case(sys.argv[2], int(sys.argv[3]))
        print("exact ok")
