"""The factorisation's envelope: pixels in wavelength order leave K exactly zero outside a narrow band of row blocks,
and the likelihood's launches stop at the envelope the device computes from the fill's exact-zero tile flags.

CPU: the host envelope (psoap_b200.envelope) on hand-made flag patterns, its flop model, and the farm's pixel order.
GPU (-m gpu): the device envelope against the host one from the flags of the matrix psoap_debug_fill_lower returns
(sorted C4-size chunks, and an epoch-major chunk whose envelope is the whole matrix); psoap_lnlike on sorted chunks
against the lnlike of the unrestricted gradient elimination (==) under launch switches that give both the same plan;
parity with a scipy Cholesky at the package-default amplitude 0.5.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from psoap_b200 import envelope, synthetic  # noqa: E402

gpu = pytest.mark.gpu
NB = envelope.NB


def c4_chunk(N, seed=11, n_epochs=20):
    """A C4-like SB2 chunk of N = n_epochs * n_pix pixels (epoch-major, as make_chunk returns it)."""
    return synthetic.make_chunk("SB2", n_epochs, N // n_epochs, seed=seed, wl0=5000.0 + 0.37 * seed)


def chunk_z(ch, sort=True):
    p = synthetic.default_params("SB2")
    vel = synthetic.host_velocities("SB2", p[:7], ch["date1D"])
    if sort:
        order, zs = envelope.sorted_chunk_z(ch, vel)
    else:
        order = np.arange(len(ch["fl"]))
        zs = np.array([ch["lwl"] + (-np.asarray(v)[ch["epoch"]]) / synthetic.c_kms for v in vel])
    return zs, np.asarray(ch["fl"])[order], np.asarray(ch["sigma"])[order]


# ---------------------------------------------------------------------------------------------- CPU
def test_tend_banded_pattern():
    T, w = 12, 3
    flags = np.zeros((T, T), dtype=bool)
    for I in range(T):
        flags[I, max(0, I - w):I + 1] = True
    tend = envelope.tend_by_end(flags)
    assert tend[0] == T
    # rows I with I - w >= e are zero in columns < e: tend[e] = min(e + w, T)
    assert list(tend[1:]) == [min(e + w, T) for e in range(1, T + 1)]
    assert np.all(np.diff(tend[1:]) >= 0)


def test_tend_needs_the_suffix_minimum():
    T = 8
    flags = np.eye(T, dtype=bool)
    flags[6, 0] = True   # a late row reaching back to column 0 keeps every earlier group's rows up to it
    tend = envelope.tend_by_end(flags)
    assert tend[1] == 7 and tend[7] == 7 and tend[8] == 8


def test_tend_dense_is_whole_matrix():
    T = 9
    tend = envelope.tend_by_end(np.tril(np.ones((T, T), dtype=bool)))
    assert list(tend) == [T] * (T + 1)


def test_flop_model_dense_equals_full_envelope():
    T = 40
    full = np.full(T + 1, T)
    for G in (1, 2, 4, 8):
        assert envelope.executed_flops(T, G) == envelope.executed_flops(T, G, full)
    band = envelope.tend_by_end(np.tril(np.triu(np.ones((T, T), dtype=bool), -17)))
    assert envelope.executed_flops(T, 8, band) < 0.7 * envelope.executed_flops(T, 8)


def test_sorted_chunk_envelope_is_narrow():
    zs, fl, sg = chunk_z(c4_chunk(6000))
    tend = envelope.tend_by_end(envelope.tile_flags_from_z(zs, [0.1, 0.05], [5.0, 7.0], sg))
    T = envelope.padded_tiles(6000)
    assert tend[8] < T and tend[16] < T
    zs_u, _, sg_u = chunk_z(c4_chunk(6000), sort=False)
    tend_u = envelope.tend_by_end(envelope.tile_flags_from_z(zs_u, [0.1, 0.05], [5.0, 7.0], sg_u))
    assert np.all(tend_u[1:] == T)


# ---------------------------------------------------------------------------------------------- GPU helpers
def _device_envelope_and_fill(zs, fl, sg, amps, ls, mu=1.0):
    """psoap_lnlike on the vectors, then (tend read from its workspace, lnlike, the debug fill's padded matrix)."""
    import torch
    from psoap_b200 import _lib
    lib = _lib.load()
    N = len(fl)
    ncomp = len(zs)
    zd = [torch.tensor(np.ascontiguousarray(z), dtype=torch.float64, device="cuda") for z in zs]
    fd = torch.tensor(fl, dtype=torch.float64, device="cuda")
    sd = torch.tensor(sg, dtype=torch.float64, device="cuda")
    nbytes = lib.psoap_lnlike_workspace_bytes(N)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    wp = (ws.data_ptr() + 255) // 256 * 256
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    ptrs = [z.data_ptr() for z in zd] + [None] * (3 - ncomp)
    _lib.check(lib.psoap_lnlike(ncomp, N, ptrs[0], ptrs[1], ptrs[2], fd.data_ptr(), sd.data_ptr(), _lib.dbl_array(amps),
                                _lib.dbl_array(ls), mu, wp, nbytes, res.data_ptr(), None))
    torch.cuda.synchronize()
    tp, T = _lib.vp(), ctypes.c_int()
    _lib.check(lib.psoap_lnlike_envelope_view(wp, N, ctypes.byref(tp), ctypes.byref(T)))
    T = T.value
    off = tp.value - ws.data_ptr()   # the envelope lives inside the workspace tensor
    tend = ws[off:off + 4 * (T + 1)].view(torch.int32).cpu().numpy().astype(np.int64)
    Np = T * NB
    W = torch.zeros((Np, Np), dtype=torch.float64, device="cuda")   # row-major [col, row]: W(i, j) = W[j, i]
    rvec = torch.empty(Np, dtype=torch.float64, device="cuda")
    _lib.check(lib.psoap_debug_fill_lower(ncomp, N, ptrs[0], ptrs[1], ptrs[2], None, None, 0, fd.data_ptr(), sd.data_ptr(),
                                          _lib.dbl_array(amps), _lib.dbl_array(ls), mu, W.data_ptr(), Np, rvec.data_ptr(),
                                          None))
    K = W.t().cpu().numpy()
    return tend, float(res[0].item()), K


def _scipy_lnlike(zs, fl, sg, amps, ls, mu=1.0):
    from scipy.linalg import cho_factor, cho_solve
    K = np.diag(np.asarray(sg, dtype=np.float64) ** 2)
    for z, a, l in zip(zs, amps, ls):
        p2 = -0.5 * synthetic.c_kms ** 2 / (l * l)
        D = z[None, :] - z[:, None]
        K += a * a * np.exp((p2 * D) * D)
    cf = cho_factor(K, lower=True)
    r = np.asarray(fl, dtype=np.float64) - mu
    return -0.5 * (r @ cho_solve(cf, r) + 2.0 * np.sum(np.log(np.diag(cf[0]))))


# ---------------------------------------------------------------------------------------------- GPU
@gpu
@pytest.mark.parametrize("N,sort", [(2000, True), (4000, True), (5000, True), (6000, True), (6000, False)],
                         ids=["2000", "4000", "5000", "6000", "6000-unsorted"])
def test_device_envelope_matches_fill_flags(N, sort):
    zs, fl, sg = chunk_z(c4_chunk(N, seed=N), sort=sort)
    amps, ls = [0.1, 0.05], [5.0, 7.0]
    tend, lnl, K = _device_envelope_and_fill(zs, fl, sg, amps, ls)
    T = envelope.padded_tiles(N)
    assert len(tend) == T + 1 and tend[0] == T
    want = envelope.tend_by_end(envelope.tile_flags_from_matrix(K))
    assert np.array_equal(tend, want), (tend, want)
    if sort and N >= 4000:
        assert tend[8] < T            # the restriction is active
    if not sort:
        assert np.all(tend == T)      # epoch-major order: every launch in full
    assert abs(lnl - _scipy_lnlike(zs, fl, sg, amps, ls)) <= 1e-10 * abs(lnl)


@gpu
@pytest.mark.parametrize("N", [4000, 6000])
@pytest.mark.parametrize("ncomp", [1, 2])
def test_sorted_parity_default_amplitude(N, ncomp):
    """amp 0.5: a 128 x 128 diagonal block of a sorted chunk holds ~20 near-duplicate pixels per wavelength; its
    condition number rises to ~5e4, which the explicit inverses of the panel chain carry as cond * eps."""
    zs, fl, sg = chunk_z(c4_chunk(N, seed=N + 1))
    amps, ls = [0.5, 0.5][:ncomp], [5.0, 7.0][:ncomp]
    tend, lnl, _ = _device_envelope_and_fill(zs[:ncomp], fl, sg, amps, ls)
    ref = _scipy_lnlike(zs[:ncomp], fl, sg, amps, ls)
    assert abs(lnl - ref) <= 1e-10 * abs(ref), (lnl, ref)


# The gradient elimination runs every launch in full (no envelope), and its lnlike comes from the same kernels; under
# switches that give both the same launch plan (forced group size, so no single-panel tail) the two are the same bits.
SAME_PLAN_ENVS = {"group2-chain7-lookahead": {"PSOAP_GROUP": "2"},
                  "group4-chain7-lookahead": {"PSOAP_GROUP": "4"},
                  "group4-chain3": {"PSOAP_GROUP": "4", "PSOAP_POTRF": "3"},
                  "group8-no-lookahead": {"PSOAP_GROUP": "8", "PSOAP_LOOKAHEAD": "0"},
                  "group2-no-pdl": {"PSOAP_GROUP": "2", "PSOAP_PDL": "0"}}


def _child_same_bits():
    from psoap_b200 import covariance
    for N, ncomp in ((6000, 2), (4500, 1), (6000, 1)):
        zs, fl, sg = chunk_z(c4_chunk(N, seed=N + 7))
        amps, ls = [0.1, 0.05][:ncomp], [5.0, 7.0][:ncomp]
        tend, lnl, _ = _device_envelope_and_fill(zs[:ncomp], fl, sg, amps, ls)
        assert tend[8] < envelope.padded_tiles(N), tend
        g = covariance.lnlike_grad(list(zs[:ncomp]), fl, sg, amps, ls)
        assert lnl == g.lnlike, (N, ncomp, lnl, g.lnlike)
        print("N = %d ncomp = %d lnlike %.17g == %.17g" % (N, ncomp, lnl, g.lnlike))
    print("same bits ok")


@gpu
@pytest.mark.parametrize("cfg", sorted(SAME_PLAN_ENVS))
def test_restricted_lnlike_equals_unrestricted(cfg):
    env = dict(os.environ, **SAME_PLAN_ENVS[cfg])
    env["PYTHONPATH"] = os.pathsep.join([ROOT] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), "same-bits"], env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "same bits ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


if __name__ == "__main__" and sys.argv[1:] == ["same-bits"]:
    _child_same_bits()
