"""The farm's gradient graph (psoap_farm_grad_attach / psoap_farm_lnprob_grad, ChunkFarm.chunk_lnlike_grads_many and
lnprob_and_grad_many): every (proposal, chunk) pair through the steps of psoap_chunk_lnprob_grad in one graph launch.

The sequential path (ChunkFarm.chunk_lnlike_grads, one chunk at a time on the direct API) is the reference: under
launch switches that give both paths the same launch plan the rows must be the same bits; under the defaults they
agree to rounding.
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
gpu = pytest.mark.gpu


def _lib():
    from psoap_b200 import _lib as L
    return L, L.load()


def proposals(model, K, seed):
    """K distinct valid registered vectors around the synthetic defaults."""
    from psoap_b200 import synthetic
    p = synthetic.default_params(model)
    rng = np.random.default_rng(seed)
    return np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])


def seq_rows(farm, P):
    """chunk_lnlike_grads of every proposal: [K, n_chunks, n_params + 1]."""
    return np.stack([farm.chunk_lnlike_grads(p).cpu().numpy() for p in P])


def c4_subset():
    """8 chunks with the sizes of C4's (N = 2000 .. 6000), spread over its range."""
    from psoap_b200 import synthetic
    return [synthetic.make_chunk("SB2", 20, 100 + (200 * i) // 255, seed=4000 + i, wl0=5000.0 + 4.0 * i)
            for i in (0, 36, 73, 109, 146, 182, 219, 255)]


# ---------------------------------------------------------------------------------------------- CPU
def test_farm_grad_entries_reject_a_null_farm():
    from psoap_b200 import _build
    _build.build_library()
    L, lib = _lib()
    assert lib.psoap_version() >= 102
    assert lib.psoap_farm_grad_workspace_bytes(None, 4) == 0
    assert lib.psoap_farm_grad_attach(None, 4, None, 0) == -1 and b"psoap_farm_grad_attach" in lib.psoap_last_error()
    assert lib.psoap_farm_lnprob_grad(None, None, None, None, None) == -1
    assert b"psoap_farm_lnprob_grad" in lib.psoap_last_error()
    assert lib.psoap_launch_count() == 0


def test_grad_nbranch_is_validated():
    from psoap_b200.farm import ChunkFarm
    with pytest.raises(ValueError, match="grad_nbranch"):
        ChunkFarm("SB1", [], grad_nbranch=0)


# ---------------------------------------------------------------------------------------------- GPU
@gpu
def test_attach_arguments_and_workspace_size():
    import torch
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    L, lib = _lib()
    chunks = [synthetic.make_chunk("SB2", 4, 40 + 30 * i, seed=500 + i) for i in range(4)]
    farm = ChunkFarm("SB2", chunks, n_proposals=2)
    f = farm._farm
    sizes = [lib.psoap_farm_grad_workspace_bytes(f, nb) for nb in (1, 2, 4, 8)]
    assert all(a < b for a, b in zip(sizes, sizes[1:])), sizes
    assert lib.psoap_farm_grad_workspace_bytes(f, 0) == 0
    assert lib.psoap_farm_grad_workspace_bytes(f, 64) == sizes[-1]   # capped at the 8 (proposal, chunk) pairs
    P = torch.from_numpy(proposals("SB2", 2, 1)).cuda()
    res = torch.empty((2, 4, 4), dtype=torch.float64, device="cuda")
    g = torch.empty((2, 4, 11), dtype=torch.float64, device="cuda")
    ws = torch.empty(sizes[1] + 512, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    n0 = lib.psoap_launch_count()
    assert lib.psoap_farm_lnprob_grad(f, L.ptr(P), L.ptr(res), L.ptr(g), L.stream_ptr()) == -1   # before attach
    assert lib.psoap_farm_grad_attach(f, 0, L.ptr(ws), sizes[1]) == -1
    assert lib.psoap_farm_grad_attach(f, 2, L.ptr(ws), sizes[1] - 1) == -3
    assert lib.psoap_farm_grad_attach(f, 2, L.vp(ws.data_ptr() + 8), sizes[1]) == -3
    assert lib.psoap_launch_count() == n0
    assert lib.psoap_farm_grad_attach(f, 2, L.ptr(ws), sizes[1]) == 0
    assert lib.psoap_farm_grad_attach(f, 2, L.ptr(ws), sizes[1]) == -1   # one gradient graph per farm
    L.check(lib.psoap_farm_lnprob_grad(f, L.ptr(P), L.ptr(res), L.ptr(g), L.stream_ptr()))
    torch.cuda.synchronize()
    assert lib.psoap_launch_count() > n0
    assert torch.isfinite(res[:, :, 0]).all() and torch.isfinite(g).all()
    farm.close()


def exact_case(model, K):
    """Graph rows == sequential rows, under switches that give both paths the same launch plan (run in a child
    process with PSOAP_POTRF=3 PSOAP_GROUP=4 PSOAP_LOOKAHEAD=0 PSOAP_FARM_LOOKAHEAD=0).  At least 8 (proposal,
    chunk) pairs, so that the farm's chain from psoap_chunk.reserved is 3 as well.  Chunks of 1 to 6 row blocks."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    n_pix = [30, 60, 95, 130, 160, 190, 45, 110]     # x 4 epochs: N = 120 .. 760
    nch = 8 if K == 1 else 3
    chunks = [synthetic.make_chunk(model, 4, n_pix[i], seed=700 + i, mask_frac=0.02) for i in range(nch)]
    assert nch * K >= 8
    blocks = sorted({(len(ch["fl"]) + 127) // 128 for ch in chunks})
    assert blocks[0] == 1 and (K > 1 or blocks[-1] == 6), blocks
    farm = ChunkFarm(model, chunks, n_proposals=K, grad_nbranch=3)
    P = proposals(model, K, seed=K)
    got = farm.chunk_lnlike_grads_many(P).cpu().numpy()
    ref = seq_rows(farm, P)
    assert np.isfinite(ref).all()
    assert np.array_equal(got, ref), np.abs(got - ref).max()
    farm.close()
    return True


EXACT_ENV = {"PSOAP_POTRF": "3", "PSOAP_GROUP": "4", "PSOAP_LOOKAHEAD": "0", "PSOAP_FARM_LOOKAHEAD": "0"}


@gpu
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("model", ["SB1", "SB2", "ST3"])
def test_graph_rows_equal_sequential_rows(model, K):
    env = dict(os.environ, **EXACT_ENV)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), "exact", model, str(K)], env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "exact ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def few_pairs_case():
    """Fewer than 8 (proposal, chunk) pairs: the graph takes look-ahead and chain 7, as the direct API does by
    default, so its rows are the sequential rows' bits without any switch."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 5, 60 + 70 * i, seed=800 + i) for i in range(3)]   # N = 300 .. 1000
    farm = ChunkFarm("SB2", chunks, n_proposals=2)
    P = proposals("SB2", 2, seed=6)
    got = farm.chunk_lnlike_grads_many(P).cpu().numpy()
    ref = seq_rows(farm, P)
    assert np.isfinite(ref).all()
    assert np.array_equal(got, ref), np.abs(got - ref).max()
    farm.close()
    return True


@gpu
@pytest.mark.parametrize("issue", ["graph", "direct"])
def test_few_pairs_take_the_direct_apis_plan(issue):
    if issue == "graph":
        assert few_pairs_case()
        return
    env = dict(os.environ, PSOAP_FARM_DIRECT="1")
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), "few"], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "few ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


@gpu
@pytest.mark.parametrize("K", [1, 2])
def test_graph_rows_match_sequential_rows_c4_sizes(K):
    """Default launch choices: the graph and the sequential path agree in every direction to 1e-10 of the terms'
    scale, and the lnlike column is the likelihood graph's when both graphs have the same branch count."""
    from psoap_b200.farm import ChunkFarm
    farm = ChunkFarm("SB2", c4_subset(), n_proposals=K)
    assert min(farm.grad_nbranch, 8 * K) == min(32, 8 * K)   # both graphs run one branch per pair
    P = proposals("SB2", K, seed=10 + K)
    got = farm.chunk_lnlike_grads_many(P).cpu().numpy()
    ref = seq_rows(farm, P)
    lnl = np.asarray(farm.chunk_lnlikes(P).cpu().numpy()).reshape(K, -1)
    assert np.array_equal(got[:, :, 0], lnl)
    rng = np.random.default_rng(3)
    for k in range(K):
        for _ in range(4):
            u = rng.standard_normal(farm.n_params)
            for gg, gs in zip(got[k, :, 1:], ref[k, :, 1:]):
                assert abs(gg @ u - gs @ u) <= 1e-10 * np.sum(np.abs(gs * u)), (gg @ u, gs @ u)
        lnp, g = farm.lnprob_and_grad_many(P)
        u = rng.standard_normal(farm.n_params)
        gs = ref[k, :, 1:].sum(axis=0)
        assert abs(g[k] @ u - gs @ u) <= 1e-10 * np.sum(np.abs(ref[k, :, 1:] * u))
    farm.close()


STEP_SCALE = {"SB2": np.array([1e-3, 0.1, 1e-3, 0.1, 1e-3, 1e-2, 0.1, 1e-3, 1e-2, 1e-3, 1e-2])}


@gpu
def test_directional_derivatives_of_lnprob_many():
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 6, 70 + 10 * i, seed=60 + i, mask_frac=0.03) for i in range(3)]
    K = 4
    farm = ChunkFarm("SB2", chunks, n_proposals=K)
    P = proposals("SB2", K, seed=4)
    lnp, G = farm.lnprob_and_grad_many(P)
    assert np.array_equal(lnp, farm.lnprob_many(P))
    rng = np.random.default_rng(5)
    for _ in range(3):
        U = rng.standard_normal(P.shape) * STEP_SCALE["SB2"]
        t = 1e-3
        fd = (farm.lnprob_many(P + t * U) - farm.lnprob_many(P - t * U)) / (2 * t)
        for k in range(K):
            scale = np.sum(np.abs(G[k] * U[k]))
            assert abs(fd[k] - G[k] @ U[k]) <= 1e-5 * scale, (k, fd[k], G[k] @ U[k], scale)
    farm.close()


def _bits_chunks():
    from psoap_b200 import synthetic
    return [synthetic.make_chunk("SB2", 4, 40 + 35 * i, seed=300 + i) for i in range(9)]   # N = 160 .. 1280


@gpu
def test_rows_are_bit_stable_across_calls_branches_and_ranks():
    from psoap_b200.farm import ChunkFarm
    chunks = _bits_chunks()
    K = 2
    P = proposals("SB2", K, seed=9)
    single = ChunkFarm("SB2", chunks, n_proposals=K, grad_nbranch=8)
    ref = single.chunk_lnlike_grads_many(P).cpu().numpy()
    assert np.isfinite(ref).all()
    assert np.array_equal(single.chunk_lnlike_grads_many(P).cpu().numpy(), ref)
    ref_lnp, ref_g = single.lnprob_and_grad_many(P)
    other = ChunkFarm("SB2", chunks, n_proposals=K, grad_nbranch=16)
    assert np.array_equal(other.chunk_lnlike_grads_many(P).cpu().numpy(), ref)
    other.close()
    for world in (2, 4):
        total = np.zeros_like(ref)
        for r in range(world):
            f = ChunkFarm("SB2", chunks, n_proposals=K, rank=r, world_size=world)
            f.world_size = 1  # no process group here: take the un-reduced rows
            rows = f.chunk_lnlike_grads_many(P).cpu().numpy()
            for i in f.mine:
                assert np.array_equal(rows[:, i], ref[:, i])
            total = total + rows
            f.close()
        assert np.array_equal(total, ref)
        lnp = np.array([float(np.sum(t[:, 0])) for t in total])
        g = np.stack([np.sum(t[:, 1:], axis=0) for t in total])
        assert np.array_equal(lnp, ref_lnp) and np.array_equal(g, ref_g)
    single.close()


@gpu
def test_a_bad_item_does_not_touch_the_next_one():
    """One workspace for every item (grad_nbranch = 1): a proposal with |v| >= c and one with a negative amplitude
    give -inf and all-NaN rows, and the valid proposals around them the bits they have in an all-valid batch."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 4, 50 + 40 * i, seed=90 + i) for i in range(2)]
    P = proposals("SB2", 4, seed=2)
    good = P.copy()
    bad = P.copy()
    bad[1, 1] = 4e5     # K: |v| >= c
    bad[2, 7] = -0.1    # amp_f < 0
    farm = ChunkFarm("SB2", chunks, n_proposals=4, grad_nbranch=1)
    rb = farm.chunk_lnlike_grads_many(bad).cpu().numpy()
    rg = farm.chunk_lnlike_grads_many(good).cpu().numpy()
    for k in (1, 2):
        assert np.all(rb[k, :, 0] == -np.inf) and np.isnan(rb[k, :, 1:]).all()
    assert np.isfinite(rg).all()
    for k in (0, 3):
        assert np.array_equal(rb[k], rg[k])
    farm.close()


@gpu
def test_the_likelihood_graph_is_untouched():
    import torch
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 4, 50 + 30 * i, seed=120 + i) for i in range(5)]
    P = proposals("SB2", 2, seed=8)
    farm = ChunkFarm("SB2", chunks, n_proposals=2)
    torch.cuda.synchronize()
    mem = torch.cuda.memory_allocated()
    before = farm.chunk_lnlikes(P).cpu().numpy()
    farm.lnprob_many(P)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == mem and farm._grad_farm_ws is None
    launches = farm.launches_per_eval
    farm.chunk_lnlike_grads_many(P)
    assert farm._grad_farm_ws is not None
    after = farm.chunk_lnlikes(P).cpu().numpy()
    assert np.array_equal(before, after)
    L, lib = _lib()
    assert farm.launches_per_eval == launches == lib.psoap_farm_launches_per_eval(farm._farm)
    farm.close()


if __name__ == "__main__":
    if sys.argv[1] == "exact":
        import torch
        assert torch.cuda.is_available()
        exact_case(sys.argv[2], int(sys.argv[3]))
        print("exact ok")
    elif sys.argv[1] == "few":
        few_pairs_case()
        print("few ok")
