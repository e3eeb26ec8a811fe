"""Posterior draws of the prediction graph (psoap_farm_predict_attach_draws / psoap_farm_predict_draws,
ChunkFarm.draw_components): per (proposal, chunk) item X[s] = delta + L z[s], L = chol(Sigma + jitter I), with the
normals from a counter-based Philox4x32-10 that this file restates in numpy.

The references: the restated generator (the same uniforms; Box-Muller through numpy's log / cos / sin), numpy's Cholesky
of the graph's own Sigma output, and the outputs of the prediction graph without draws.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NCOMP = {"SB1": 1, "SB2": 2, "ST3": 3}
gpu = pytest.mark.gpu


def _lib():
    from psoap_b200 import _lib as L
    return L, L.load()


# ---------------------------------------------------------------------------------------------- the generator, restated
M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 on uint64 arrays holding 32-bit words: ctr (4 arrays), key (2 arrays or scalars)."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in ctr]
    k0, k1 = (np.asarray(x, dtype=np.uint64) & M32 for x in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & M32, p0 & M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c


def uniform(hi, lo):
    v = ((hi << np.uint64(32)) | lo) >> np.uint64(11)
    return (v.astype(np.float64) + 0.5) * 2.0 ** -53


def normals(seed, chunk_key, proposal, S, M):
    """Z [S, M]: row a of draw s from counter (a >> 1, s, proposal, chunk_key), key (seed low, seed high)."""
    j = np.arange((M + 1) // 2, dtype=np.uint64)[None, :]
    s = np.arange(S, dtype=np.uint64)[:, None]
    shape = (S, j.shape[1])
    ctr = [np.broadcast_to(j, shape), np.broadcast_to(s, shape), np.full(shape, proposal, np.uint64),
           np.full(shape, chunk_key, np.uint64)]
    x = philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32))
    u1, u2 = uniform(x[0], x[1]), uniform(x[2], x[3])
    r = np.sqrt(-2.0 * np.log(u1))
    z = np.empty((S, 2 * j.shape[1]))
    z[:, 0::2] = r * np.cos(2.0 * np.pi * u2)
    z[:, 1::2] = r * np.sin(2.0 * np.pi * u2)
    return z[:, :M]


# ---------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("ctr,key,out", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_restatement_reproduces_the_known_answers(ctr, key, out):
    assert [int(v) for v in philox4x32_10(ctr, key)] == list(out)


def test_uniforms_stay_inside_the_open_interval():
    hi = np.array([0, 0xFFFFFFFF, 0x80000000], dtype=np.uint64)
    lo = np.array([0, 0xFFFFF7FF, 0], dtype=np.uint64)
    u = uniform(hi, lo)
    assert u[0] == 2.0 ** -54 and 0.0 < u.min() and u.max() < 1.0 and u[2] == 0.5 + 2.0 ** -54


def test_draw_entries_reject_a_null_farm_and_bad_arguments():
    from psoap_b200 import _build
    _build.build_library()
    L, lib = _lib()
    assert lib.psoap_version() >= 106
    m = (ctypes.c_int64 * 2)(10, 20)
    keys = (ctypes.c_int64 * 2)(0, 1)
    off = (ctypes.c_int64 * 12)()
    assert lib.psoap_farm_predict_draws_workspace_bytes(None, 4, m, 0, 8) == 0
    assert lib.psoap_farm_predict_attach_draws(None, 4, m, None, 0, 8, 1e-8, keys, None, 0, off) == -1
    assert b"psoap_farm_predict_attach_draws" in lib.psoap_last_error()
    assert lib.psoap_farm_predict_draws(None, *([None] * 8)) == -1
    assert b"psoap_farm_predict_draws" in lib.psoap_last_error()
    assert lib.psoap_debug_normals(1, -1, 0, 4, 10, None, None) == -1
    assert lib.psoap_debug_normals(1, 0, 0, 0, 10, L.vp(256), None) == -1
    assert lib.psoap_debug_normals(1, 0, 0, 4, 0, L.vp(256), None) == -1
    assert lib.psoap_debug_normals(1, 1 << 32, 0, 4, 10, L.vp(256), None) == -1
    assert b"psoap_debug_normals" in lib.psoap_last_error()
    assert lib.psoap_launch_count() == 0


def _bare_farm():
    """A ChunkFarm with only the host attributes the argument checks read (no device needed)."""
    from psoap_b200.farm import ChunkFarm
    f = ChunkFarm.__new__(ChunkFarm)
    f.model, f.n_chunks, f.n_proposals, f.n_params = "SB2", 2, 2, 11
    f._n_pix, f._pred, f.mine, f._farm = [40, 0], None, [0], None
    return f


def test_draw_arguments_are_checked():
    f = _bare_farm()
    g = np.linspace(8.5, 8.6, 7)
    for bad in (-1, 2.0, True, "3"):
        with pytest.raises(ValueError, match="n_draws"):
            f.attach_prediction_grids([g, []], n_draws=bad)
    for bad in (-1e-9, np.inf, np.nan):
        with pytest.raises(ValueError, match="jitter"):
            f.attach_prediction_grids([g, []], n_draws=4, jitter=bad)
    P = np.zeros((2, 11))
    with pytest.raises(ValueError, match="P must hold"):
        f.draw_components(P[:1], [0.5, 0.5], 1)
    with pytest.raises(ValueError, match="mus"):
        f.draw_components(P, [0.5], 1)
    for bad in (-1, 2 ** 64, 1.5, None):
        with pytest.raises(ValueError, match="seed"):
            f.draw_components(P, [0.5, 0.5], bad)
    with pytest.raises(RuntimeError, match="n_draws > 0"):
        f.draw_components(P, [0.5, 0.5], 1)
    f._pred = {"n_draws": 0}
    with pytest.raises(RuntimeError, match="n_draws > 0"):
        f.draw_components(P, [0.5, 0.5], 1)
    f._pred = {"n_draws": 4}
    with pytest.raises(RuntimeError, match="draw_components"):
        f.predict_components(P, [0.5, 0.5])
    with pytest.raises(RuntimeError, match="already attached"):
        f.attach_prediction_grids([g, []], n_draws=4)


# ---------------------------------------------------------------------------------------------- GPU
def _chunks(model, n_pix, seed, n_epochs=4, **kw):
    from psoap_b200 import synthetic
    return [synthetic.make_chunk(model, n_epochs, n, seed=seed + i, wl0=5000.0 + 3.0 * i, **kw) for i, n in enumerate(n_pix)]


def _empty_chunk(model):
    from psoap_b200 import synthetic
    ch = synthetic.make_chunk(model, 4, 30, seed=99)
    ch["mask"][:] = False
    for key in ("lwl", "fl", "sigma", "epoch"):
        ch[key] = ch[key][:0]
    return ch


def grid_of(ch, m, shift=0.0):
    """m rest-frame ln-wavelength points over the chunk's range (not on the pixels)."""
    lo, hi = ch["lwl"].min(), ch["lwl"].max()
    return lo + (hi - lo) * (np.arange(m) + 0.37) / m + shift


def proposals(model, K, seed):
    from psoap_b200 import synthetic
    p = synthetic.default_params(model)
    rng = np.random.default_rng(seed)
    return np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])


def mus_of(model):
    return np.linspace(0.4, 0.6, NCOMP[model])


def _np(outs):
    return [tuple(t.cpu().numpy() for t in o) for o in outs]


def _same(a, b):
    return all(len(x) == len(y) and all(np.array_equal(u, v, equal_nan=True) for u, v in zip(x, y)) for x, y in zip(a, b))


def raw_predict(farm, P):
    """One psoap_farm_predict call on this rank's items: delta, sigma, results [K, n_mine, 4], offsets."""
    import torch
    L, lib = _lib()
    off = farm._pred["off"]
    p = torch.from_numpy(np.ascontiguousarray(P, dtype=np.float64)).cuda()
    d = torch.full((max(1, int(off[0, -1])),), 7.0, dtype=torch.float64, device="cuda")
    s = torch.full((max(1, int(off[1, -1])),), 7.0, dtype=torch.float64, device="cuda")
    r = torch.empty((farm.n_proposals, len(farm.mine), 4), dtype=torch.float64, device="cuda")
    L.check(lib.psoap_farm_predict(farm._farm, L.ptr(p), L.ptr(d), L.ptr(s), L.ptr(r), L.stream_ptr()))
    return d.cpu().numpy(), s.cpu().numpy(), r.cpu().numpy(), off


def raw_draws(farm, P, seed):
    """One psoap_farm_predict_draws call on this rank's items: delta, sigma, draws, results, sigma results, offsets."""
    import torch
    L, lib = _lib()
    off = farm._pred["off"]
    K, n = farm.n_proposals, len(farm.mine)
    p = torch.from_numpy(np.ascontiguousarray(P, dtype=np.float64)).cuda()
    sd = torch.tensor([seed], dtype=torch.int64, device="cuda")
    bufs = [torch.full((max(1, int(off[r, -1])),), 7.0, dtype=torch.float64, device="cuda") for r in range(3)]
    r = torch.empty((2, K, n, 4), dtype=torch.float64, device="cuda")
    L.check(lib.psoap_farm_predict_draws(farm._farm, L.ptr(p), L.ptr(sd), *[L.ptr(b) for b in bufs], L.ptr(r[0]),
                                         L.ptr(r[1]), L.stream_ptr()))
    return [b.cpu().numpy() for b in bufs] + [r[0].cpu().numpy(), r[1].cpu().numpy(), off]


@gpu
def test_generator_equals_the_restatement():
    import torch
    L, lib = _lib()
    for seed, key, prop, S, M in [(0, 0, 0, 3, 7), (2 ** 64 - 1, 255, 3, 5, 130), (0x0123456789ABCDEF, 17, 1, 64, 601)]:
        out = torch.full((S, M), 7.0, dtype=torch.float64, device="cuda")
        L.check(lib.psoap_debug_normals(seed, key, prop, S, M, L.ptr(out), L.stream_ptr()))
        z = out.cpu().numpy()
        ref = normals(seed, key, prop, S, M)
        assert np.max(np.abs(z - ref)) <= 1e-13, (seed, np.max(np.abs(z - ref)))
    # a different seed, key, proposal or draw gives other normals
    a = normals(5, 1, 0, 2, 8)
    for other in (normals(6, 1, 0, 2, 8), normals(5, 2, 0, 2, 8), normals(5, 1, 1, 2, 8)):
        assert not np.any(a == other)
    assert not np.any(a[0] == a[1])


def _check_product(farm, out, P, seed, tol_of):
    """draws - mu == L Z per item of this farm, L = numpy's Cholesky of the graph's Sigma + jitter I, Z restated;
    returns the largest error relative to the scale max|L| |Z| and the smallest pivot of L."""
    jitter, S = farm._pred["jitter"], farm._pred["n_draws"]
    worst, pivot = 0.0, np.inf
    for i, (mu, Sig, X) in enumerate(out):
        M = mu.shape[1]
        if M == 0:
            continue
        for k in range(P.shape[0]):
            Lc = np.linalg.cholesky(Sig[k] + jitter * np.eye(M))
            pivot = min(pivot, float(np.min(np.diag(Lc)) ** 2))
            Z = normals(seed, i, k, S, M)
            ref = Z @ Lc.T
            err = np.max(np.abs((X[k] - mu[k]) - ref))
            scale = np.max(np.abs(Z) @ np.abs(Lc).T)
            assert err <= tol_of(Sig[k] + jitter * np.eye(M), Lc) * scale, (i, k, err / scale)
            worst = max(worst, err / scale)
    return worst, pivot


@gpu
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_draws_are_delta_plus_l_z_on_a_coarse_grid(model):
    """A coarse grid (spacing about three length scales): Sigma is well conditioned and the product agrees with numpy's
    Cholesky to 1e-12 of its scale.  The chunk without pixels yields empty outputs."""
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks(model, [60, 90], seed=40)
    chunks.insert(1, _empty_chunk(model))
    grids = [grid_of(chunks[0], 12), np.zeros(0), grid_of(chunks[2], 17)]
    K, S = 2, 48
    farm = ChunkFarm(model, chunks, n_proposals=K)
    farm.attach_prediction_grids(grids, n_draws=S)
    P = proposals(model, K, seed=1)
    out = _np(farm.draw_components(P, mus_of(model), seed=1234))
    assert out[1][0].shape == (K, 0) and out[1][1].shape == (K, 0, 0) and out[1][2].shape == (K, S, 0)
    assert out[0][2].shape == (K, S, 12 * NCOMP[model])
    conds = [np.linalg.cond(o[1][k] + 1e-8 * np.eye(o[1].shape[1])) for o in out if o[0].shape[1] for k in range(K)]
    eps = np.finfo(float).eps
    worst, pivot = _check_product(farm, out, P, 1234,
                                  lambda A, Lc: max(1e-12, 4.0 * A.shape[0] * eps * np.linalg.cond(A)))
    print("coarse %s: kappa <= %.3g, max error %.3g of the scale, smallest pivot %.3g" % (model, max(conds), worst, pivot))
    farm.close()


@gpu
def test_draws_on_the_retrieve_grid():
    """The retrieve script's 2x oversampled grid (m = 2 n_pix): Sigma is numerically singular and only the jitter makes
    it definite.  Tolerance from the Cholesky error bound, |L Lhat^T - A| <= c M eps |L||L^T|, which moves L by at most
    about kappa(A) M eps |L| (normwise), with a factor 4 of headroom."""
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [100], seed=4100, n_epochs=20)
    farm = ChunkFarm("SB2", chunks)
    farm.attach_prediction_grids([grid_of(chunks[0], 200)], n_draws=16)
    P = proposals("SB2", 1, seed=0)
    out = _np(farm.draw_components(P, mus_of("SB2"), seed=77))
    eps = np.finfo(float).eps
    worst, pivot = _check_product(farm, out, P, 77, lambda A, Lc: 4.0 * A.shape[0] * eps * np.linalg.cond(A))
    print("retrieve grid: max error %.3g of the scale, smallest pivot %.3g (jitter 1e-8)" % (worst, pivot))
    assert pivot > 0.0
    farm.close()


@gpu
def test_sample_moments_match_the_prediction():
    """S = 20000 draws of one small item: sample mean and covariance within 6 standard errors of (mu, Sigma + jitter I),
    entry by entry (fixed seed)."""
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [50], seed=31)
    farm = ChunkFarm("SB2", chunks)
    S = 20000
    farm.attach_prediction_grids([grid_of(chunks[0], 4)], n_draws=S, jitter=1e-6)
    P = proposals("SB2", 1, seed=0)
    mu, Sig, X = _np(farm.draw_components(P, mus_of("SB2"), seed=2024))[0]
    A = Sig[0] + 1e-6 * np.eye(Sig.shape[1])
    x = X[0]
    se_mean = np.sqrt(np.diag(A) / S)
    assert np.all(np.abs(x.mean(axis=0) - mu[0]) <= 6 * se_mean)
    C = np.cov(x, rowvar=False)
    se_cov = np.sqrt((np.outer(np.diag(A), np.diag(A)) + A ** 2) / S)
    assert np.all(np.abs(C - A) <= 6 * se_cov), np.max(np.abs(C - A) / se_cov)
    farm.close()


def draws_case(path):
    """Child process (launch switches in the environment): draws of a fixed problem saved to path."""
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [40 + 35 * i for i in range(5)], seed=300)
    farm = ChunkFarm("SB2", chunks, n_proposals=2)
    farm.attach_prediction_grids([grid_of(ch, 30 + 13 * i) for i, ch in enumerate(chunks)], n_draws=8, predict_nbranch=4)
    out = _np(farm.draw_components(proposals("SB2", 2, seed=9), [0.45, 0.55], seed=31337))
    np.savez(path, *[a for o in out for a in o])
    farm.close()


@gpu
def test_draws_are_bit_stable_across_calls_seeds_branches_issue_and_ranks(tmp_path):
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [40 + 35 * i for i in range(5)], seed=300)
    grids = [grid_of(ch, 30 + 13 * i) for i, ch in enumerate(chunks)]
    K, P, mus = 2, proposals("SB2", 2, seed=9), [0.45, 0.55]
    single = ChunkFarm("SB2", chunks, n_proposals=K)
    single.attach_prediction_grids(grids, n_draws=8, predict_nbranch=4)
    ref = _np(single.draw_components(P, mus, seed=31337))
    assert all(np.isfinite(a).all() for o in ref for a in o)
    assert _same(ref, _np(single.draw_components(P, mus, seed=31337)))
    other_seed = _np(single.draw_components(P, mus, seed=31338))
    for a, b in zip(ref, other_seed):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and not np.any(a[2] == b[2])
    for nb in (1, 16):
        f = ChunkFarm("SB2", chunks, n_proposals=K)
        f.attach_prediction_grids(grids, n_draws=8, predict_nbranch=nb)
        assert _same(ref, _np(f.draw_components(P, mus, seed=31337))), nb
        f.close()
    path = str(tmp_path / "direct.npz")
    env = dict(os.environ, PSOAP_FARM_DIRECT="1")
    env["PYTHONPATH"] = os.pathsep.join([ROOT] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), "draws", path], env=env, capture_output=True,
                       text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    z = np.load(path)
    flat = [z["arr_%d" % j] for j in range(len(z.files))]
    assert all(np.array_equal(a, b) for a, b in zip(flat, [a for o in ref for a in o]))
    seen = set()
    for rk in range(2):
        f = ChunkFarm("SB2", chunks, n_proposals=K, rank=rk, world_size=2)
        f.world_size = 1   # no process group here: take the un-reduced buffers
        f.attach_prediction_grids(grids, n_draws=8, predict_nbranch=4)
        outs = _np(f.draw_components(P, mus, seed=31337))
        for i in f.mine:
            assert _same([outs[i]], [ref[i]]), (rk, i)
            seen.add(i)
        f.close()
    assert seen == set(range(len(chunks)))
    single.close()


@gpu
@pytest.mark.parametrize("sigma", ["full", "diag"])
def test_prediction_outputs_are_those_of_the_graph_without_draws(sigma):
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("ST3", [50, 80, 120], seed=610)
    chunks.insert(2, _empty_chunk("ST3"))
    grids = [grid_of(ch, 20 + 11 * i) if len(ch["fl"]) else np.zeros(0) for i, ch in enumerate(chunks)]
    P = proposals("ST3", 2, seed=4)
    plain = ChunkFarm("ST3", chunks, n_proposals=2)
    plain.attach_prediction_grids(grids, sigma=sigma)
    d0, s0, r0, off0 = raw_predict(plain, P)
    drawn = ChunkFarm("ST3", chunks, n_proposals=2)
    drawn.attach_prediction_grids(grids, sigma=sigma, n_draws=5)
    d1, s1, x1, r1, rs1, off1 = raw_draws(drawn, P, 3)
    assert np.array_equal(off0, off1[:2])
    assert np.array_equal(d0, d1) and np.array_equal(s0, s1) and np.array_equal(r0, r1)
    assert np.isfinite(x1[:off1[2, -1]]).all() and np.all(rs1[..., 3] == 0) and np.all(rs1[..., 2] == 0)
    # Sigma's record: its log-determinant with the jitter
    if sigma == "full":
        for c, i in enumerate(drawn.mine):
            M = 3 * (20 + 11 * i)
            A = s1[off1[1, c]:off1[1, c] + M * M].reshape(M, M) + 1e-8 * np.eye(M)
            assert abs(rs1[0, c, 1] - np.linalg.slogdet(A)[1]) <= 1e-6 * M
    with pytest.raises(Exception, match="psoap_farm_predict_draws"):
        raw_predict(drawn, P)
    plain.close()
    drawn.close()


@gpu
@pytest.mark.parametrize("how", ["velocity", "gp"])
def test_a_bad_proposal_gives_nan_draws_for_that_proposal_only(how):
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB2", [50, 90], seed=90)
    grids = [grid_of(chunks[0], 30), grid_of(chunks[1], 20)]
    P = proposals("SB2", 3, seed=2)
    bad = P.copy()
    if how == "velocity":
        bad[1, 1] = 4e5
    else:
        bad[1, 7] = -0.1
    farm = ChunkFarm("SB2", chunks, n_proposals=3, nbranch=1)
    farm.attach_prediction_grids(grids, n_draws=6, predict_nbranch=1)
    g = raw_draws(farm, P, 5)
    b = raw_draws(farm, bad, 5)
    off = g[-1]
    for c in range(2):
        for k in range(3):
            it = k * 2 + c
            x = slice(off[2, it], off[2, it] + 6 * 2 * (30 if c == 0 else 20))
            if k == 1:
                assert np.isnan(b[2][x]).all() and b[3][k, c, 0] == -np.inf
            else:
                assert np.isfinite(g[2][x]).all() and np.array_equal(b[2][x], g[2][x])
    with pytest.raises(ValueError, match="proposal 1, chunk 0"):
        farm.draw_components(bad, [0.5, 0.5], 5)
    farm.close()


@gpu
def test_a_sigma_that_is_not_definite_gives_nan_draws_for_that_item_only():
    """A negative C-level jitter of -2 max diag(Sigma) of chunk 0 (grid inside the data: small posterior variance) makes
    that item's Sigma + jitter I indefinite at its first pivot, while chunk 1's grid lies far from its data (Sigma is the
    prior on a coarse grid, eigenvalues near amp^2) and stays definite.  The Python layer refuses a negative jitter, so
    the test attaches through the C entry and then takes draw_components' path."""
    import torch
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    chunks = _chunks("SB1", [60, 60], seed=700)
    grids = [grid_of(chunks[0], 20), grid_of(chunks[1], 6, shift=0.01)]
    P = proposals("SB1", 1, seed=0)
    plain = ChunkFarm("SB1", chunks)
    plain.attach_prediction_grids(grids)
    d0, s0, r0, o0 = raw_predict(plain, P)
    plain.close()
    S0, S1 = s0[o0[1, 0]:o0[1, 1]].reshape(20, 20), s0[o0[1, 1]:o0[1, 2]].reshape(6, 6)
    jitter = -2.0 * float(np.max(np.diag(S0)))
    assert np.linalg.eigvalsh(S1).min() > 10 * abs(jitter)
    farm = ChunkFarm("SB1", chunks)
    farm.attach_prediction_grids(grids, n_draws=4)
    q = farm._pred
    farm.close()
    gr = [torch.from_numpy(np.ascontiguousarray(g)).cuda() for g in grids]
    ptrs = (L.vp * 2)(*[L.ptr(g) for g in gr])
    m = (ctypes.c_int64 * 2)(20, 6)
    keys = (ctypes.c_int64 * 2)(0, 1)
    bad = ChunkFarm("SB1", chunks)
    nbytes = lib.psoap_farm_predict_draws_workspace_bytes(bad._farm, 4, m, 0, 4)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    off = (ctypes.c_int64 * 9)()
    L.check(lib.psoap_farm_predict_attach_draws(bad._farm, 4, m, ptrs, 0, 4, jitter, keys, L.ptr(ws), nbytes, off))
    bad._pred = dict(q, jitter=jitter, ws=ws, grids=gr, off=np.frombuffer(off, dtype=np.int64).reshape(3, 3).copy())
    d, s, x, r, rs, o = raw_draws(bad, P, 11)
    assert rs[0, 0, 3] == 1 and rs[0, 1, 3] == 0
    assert np.array_equal(d, d0) and np.array_equal(s, s0) and np.array_equal(r, r0)
    assert np.isnan(x[o[2, 0]:o[2, 1]]).all() and np.isfinite(x[o[2, 1]:o[2, 2]]).all()
    Lc = np.linalg.cholesky(S1 + jitter * np.eye(6))
    Z = normals(11, 1, 0, 4, 6)
    X1 = x[o[2, 1]:o[2, 2]].reshape(4, 6) - d[o[0, 1]:o[0, 2]]
    assert np.max(np.abs(X1 - Z @ Lc.T)) <= 1e-12 * np.max(np.abs(Z) @ np.abs(Lc).T)
    with pytest.raises(np.linalg.LinAlgError, match="jitter"):
        bad.draw_components(P, [0.5], 11)
    bad.close()


@gpu
def test_the_other_graphs_are_untouched_by_draws():
    from psoap_b200.farm import ChunkFarm
    chunks = _chunks("SB1", [50 + 30 * i for i in range(4)], seed=120)
    P = proposals("SB1", 2, seed=8)
    farm = ChunkFarm("SB1", chunks, n_proposals=2)
    launches = farm.launches_per_eval
    lnl = farm.chunk_lnlikes(P).cpu().numpy()
    rows = farm.chunk_lnlike_grads_many(P).cpu().numpy()
    farm.attach_prediction_grids([grid_of(ch, 40) for ch in chunks], n_draws=3)
    farm.draw_components(P, [0.5], 0)
    assert np.array_equal(farm.chunk_lnlikes(P).cpu().numpy(), lnl)
    assert np.array_equal(farm.chunk_lnlike_grads_many(P).cpu().numpy(), rows)
    L, lib = _lib()
    assert farm.launches_per_eval == launches == lib.psoap_farm_launches_per_eval(farm._farm)
    farm.close()


if __name__ == "__main__":
    if sys.argv[1] == "draws":
        draws_case(sys.argv[2])
        print("draws ok")
