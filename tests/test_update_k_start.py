"""Each update tile starts its k loop at the first panel its row block can hold a non-zero.

The envelope kernel stores the row profile F (the suffix minimum of every row block's first non-zero block column) next
to tend, and every trailing-update tile of row block I, in the group update, its look-ahead parts and the in-group
column updates, starts at panel max(a, F[I]) of its group [a, e) (gemm.cuh SyrkSrc::kfirst).  The panels it skips are
exact zeros in row block I of L, so the result keeps its bits.

CPU: the host replay of the tile k ranges (psoap_debug_syrk_tile_k), driven with launch_factor's plan for groups of 1,
2, 4 and 8 and for a lone matrix's groups that end in single panels, on constructed exact-zero patterns (test_envelope_patterns): every skipped panel is zero in row block I of
the exact L from numpy's Cholesky, every tile runs at least one stage, and a column update whose row block is zero in
all its panels occurs and keeps one stage.  The host flop model with the profile.
GPU (-m gpu): the profile the device stores equals the host's suffix minimum, also on a pattern whose first non-zero
columns are far from monotone; the restricted likelihood against the closed form and the unrestricted gradient
elimination on every pattern, with groups of 8 (k start) and of 2 (none); and the same bits as the unrestricted
gradient elimination under the farm's plan (groups of 8, chain 3, no look-ahead).
"""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from psoap_b200 import envelope  # noqa: E402
import test_envelope_patterns as tp  # noqa: E402

gpu = pytest.mark.gpu
NB = envelope.NB
BK = 16
# the farm's plan: groups of 8, chain 3, no look-ahead
FARM_PLAN = {"PSOAP_POTRF": "3", "PSOAP_GROUP": "8", "PSOAP_LOOKAHEAD": "0"}


@pytest.fixture(scope="module")
def lib():
    from psoap_b200 import _build, _lib
    _build.build_library()
    return _lib.load()


def _reach_back(N):
    """band1, and every fifth row tile also reaches back to a column tile 3 .. 9 tiles before it (varying): the first
    non-zero columns f jump down and up again, so the suffix minimum F lies below f on many rows."""
    T, pad = tp.geometry(N)
    lab = tp._band1(N)
    for I in range(5, T, 5):
        back = 3 + (I * 7) % 7
        J = max(0, I - back)
        src = max(J * NB - pad, 0) + 1
        lab[I * NB - pad + 2] = lab[min(src, N - 1)]
    return lab


PATTERNS = {"band1": tp._band1, "band3": tp._band3, "widening": tp._widening, "gapped": tp._gapped,
            "out_of_order": tp._out_of_order, "group_edges": tp._group_edges, "pad_only": tp._pad_only,
            "reach_back": _reach_back}


def _labels_case(name, N, ncomp=1):
    case = tp.make_case("band1", N, ncomp)
    lab = np.asarray(PATTERNS[name](N), dtype=np.int64)
    case.update(name=name, labels=[lab] * ncomp, zs=[tp.Z0 + tp.DZ * lab for _ in range(ncomp)])
    return case


def _replay(lib, R, part, ncol1, sh, row0, kbeg, kend, prof, panel0):
    cap = sh * sh * (R + 1) * (R + 1) + 16
    bufs = [(ctypes.c_int * cap)() for _ in range(4)]
    pa = (ctypes.c_int * len(prof))(*[int(x) for x in prof])
    n = lib.psoap_debug_syrk_tile_k(R, part, ncol1, sh, row0, kbeg, kend, pa, len(prof), panel0, *bufs, cap)
    assert n >= 0
    return [np.array(b[:n]) for b in bufs]


SINGLE_ROWS = 24   # api.cu launch_factor: a lone chain-7 matrix ends in single-panel groups over its last 24 row blocks


def _group_starts(T, G, lone):
    """launch_factor's group boundaries: uniform groups of G, or (lone) single panels once T - a <= SINGLE_ROWS."""
    gs, a = [], 0
    while a < T:
        gs.append(a)
        a += min(1 if lone and T - a <= SINGLE_ROWS else G, T - a)
    return gs + [T]


def _launches(T, G, lone, pad, tend):
    """launch_factor's update launches for the groups of _group_starts, with the envelope: (group start a, row0, R,
    kbeg, kend, part, ncol1, shapes).  Parts 1 and 2 with ncol1 = 2 x the next group's size are the look-ahead split;
    part 1 takes both tile shapes (SH = 2 with chain 7)."""
    gs = _group_starts(T, G, lone)
    out = []
    for q in range(len(gs) - 1):
        a, e = gs[q], gs[q + 1]
        end = int(tend[e])
        kbeg = (pad // BK) * BK if q == 0 else 0
        for g in range(1, e - a):
            kb = a + g
            out.append((a, kb, end - kb, kbeg, NB * g, 1, 2, (1, 2)))
        if end > e:
            out.append((a, e, end - e, kbeg, NB * (e - a), 0, 2, (1,)))
            if q + 2 < len(gs):
                ncol1 = 2 * (gs[q + 2] - gs[q + 1])
                out.append((a, e, end - e, kbeg, NB * (e - a), 1, ncol1, (1, 2)))
                out.append((a, e, end - e, kbeg, NB * (e - a), 2, ncol1, (1,)))
    return out


@pytest.mark.parametrize("name", list(PATTERNS))
def test_update_tiles_skip_only_zero_panels(lib, name):
    """Every tile of every update launch: its k range ends at kend, starts at the group's kbeg or later on a 16-column
    boundary, runs at least one stage, and every panel it skips is exactly zero in its row block of L.  Tiles skip on
    every pattern but gapped, and there some in-group column update has a row block that is zero in all its panels and
    keeps one stage."""
    N = 6000
    case = _labels_case(name, N)
    T, pad = tp.geometry(N)
    K = tp.exact_K(case)
    L = np.linalg.cholesky(K)
    zero = ~np.any(L.reshape(T, NB, T, NB) != 0.0, axis=(1, 3))      # zero[I, k]: block (I, k) of L is exactly zero
    flags = tp.cluster_flags(case["labels"], N)
    assert np.array_equal(envelope.tile_flags_from_matrix(K), flags)
    prof = envelope.row_profile(flags)
    tend = envelope.tend_by_end(flags)
    for I in range(T):
        assert zero[I, :prof[I]].all(), (I, prof[I])
    skipped = all_zero_kept = 0
    for G, lone in ((1, False), (2, False), (4, False), (8, False), (2, True), (4, True)):
        for a, row0, R, kbeg, kend, part, ncol1, shapes in _launches(T, G, lone, pad, tend):
            for sh in shapes:
                rows, _, kb, kt = _replay(lib, R, part, ncol1, sh, row0, kbeg, kend, prof, a)
                assert np.all(kt >= 1) and np.all(kb + BK * kt == kend), (G, part, sh)
                for I, k0 in zip(rows // sh, kb):
                    assert k0 == min(max(kbeg, NB * (prof[I] - a)), kend - BK), (name, G, part, sh, I, k0)
                    if k0 > kbeg:
                        skipped += 1
                        # every panel of the group that holds a skipped column
                        for p in range(kbeg // NB, (k0 - 1) // NB + 1):
                            assert zero[I, a + p], (name, G, part, sh, I, a + p)
                    if part == 1 and ncol1 == 2 and row0 > a and prof[I] >= row0:
                        # a column update's row block that is zero in every panel: one stage, in a zero panel
                        assert zero[I, a:row0].all() and k0 == kend - BK
                        all_zero_kept += 1
    if name == "gapped":   # every row tile reaches back to tile 0 (F = 0): nothing may be skipped
        assert skipped == 0
    else:
        assert skipped > 0 and all_zero_kept > 0, (name, skipped, all_zero_kept)


def test_replay_without_profile_runs_the_full_range(lib):
    """A null profile (the gradient, Schur and prediction paths) keeps the launch's k range for every tile."""
    for part, ncol1 in ((0, 2), (1, 2), (1, 6), (2, 6)):
        for sh in (1, 2):
            bufs = [(ctypes.c_int * 4096)() for _ in range(4)]
            n = lib.psoap_debug_syrk_tile_k(9, part, ncol1, sh, 3, 112, 1024, None, 0, 0, *bufs, 4096)
            assert n > 0
            assert all(bufs[2][t] == 112 and bufs[3][t] == (1024 - 112) // BK for t in range(n))


def test_replay_rejects_bad_arguments(lib):
    bufs = [(ctypes.c_int * 16)() for _ in range(4)]
    prof = (ctypes.c_int * 4)(0, 0, 1, 2)
    assert lib.psoap_debug_syrk_tile_k(2, 0, 2, 3, 0, 0, 128, None, 0, 0, *bufs, 16) == -1      # no such shape
    assert lib.psoap_debug_syrk_tile_k(2, 0, 2, 1, 0, 128, 128, None, 0, 0, *bufs, 16) == -1    # empty k range
    assert lib.psoap_debug_syrk_tile_k(9, 0, 2, 1, 0, 0, 128, None, 0, 0, *bufs, 16) == -1      # cap too small
    assert lib.psoap_debug_syrk_tile_k(2, 0, 2, 1, 2, 0, 128, prof, 4, 0, *bufs, 16) > 0        # rows 2, 3 of 4
    assert lib.psoap_debug_syrk_tile_k(2, 0, 2, 1, 3, 0, 128, prof, 4, 0, *bufs, 16) == -1      # row 4 of 4


def test_flop_model_with_profile():
    """The host model: the profile never adds flops, changes nothing when every row reaches back to column 0, and
    removes the zero panels of a band."""
    for T in (1, 9, 47):
        for G in (1, 2, 4, 8):
            tend = np.full(T + 1, T)
            assert envelope.executed_flops(T, G, tend, np.zeros(T, dtype=int)) == envelope.executed_flops(T, G, tend)
            flags = tp.cluster_flags([tp._band3(T * NB - 5)], T * NB - 5)
            tend, prof = envelope.tend_by_end(flags), envelope.row_profile(flags)
            assert envelope.executed_flops(T, G, tend, prof) <= envelope.executed_flops(T, G, tend)
            if T == 47 and G == 8:
                assert envelope.executed_flops(T, G, tend, prof) < 0.9 * envelope.executed_flops(T, G, tend)


# ---------------------------------------------------------------------------------------------- GPU
def _device_profile(case):
    """psoap_lnlike on the case's pixels as given: (profile read from the workspace, [lnlike, logdet, quad, info])."""
    import torch
    from psoap_b200 import _lib
    lib = _lib.load()
    N, ncomp = len(case["fl"]), len(case["zs"])
    zd = [torch.tensor(np.ascontiguousarray(z), dtype=torch.float64, device="cuda") for z in case["zs"]]
    fd = torch.tensor(case["fl"], dtype=torch.float64, device="cuda")
    sd = torch.tensor(case["sigma"], dtype=torch.float64, device="cuda")
    nbytes = lib.psoap_lnlike_workspace_bytes(N)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    wp = (ws.data_ptr() + 255) // 256 * 256
    res = torch.full((4,), 7.0, dtype=torch.float64, device="cuda")
    ptrs = [z.data_ptr() for z in zd] + [None] * (3 - ncomp)
    _lib.check(lib.psoap_lnlike(ncomp, N, ptrs[0], ptrs[1], ptrs[2], fd.data_ptr(), sd.data_ptr(),
                                _lib.dbl_array(case["amps"]), _lib.dbl_array(case["ls"]), tp.MU, wp, nbytes,
                                res.data_ptr(), _lib.stream_ptr()))
    torch.cuda.synchronize()
    pp, T = _lib.vp(), ctypes.c_int()
    _lib.check(lib.psoap_lnlike_profile_view(wp, N, ctypes.byref(pp), ctypes.byref(T)))
    off = pp.value - ws.data_ptr()
    prof = ws[off:off + 4 * T.value].view(torch.int32).cpu().numpy().astype(np.int64)
    return prof, res.cpu().numpy()


def _child_profile():
    """The profile the update tiles read is F, the suffix minimum of the first non-zero columns (not f itself, which
    differs from it on the out-of-order and reach-back patterns); the likelihood stays within the closed form's
    tolerance and equals the unrestricted gradient elimination's."""
    from psoap_b200 import covariance
    for name in PATTERNS:
        for N in (1000, 2049, 6000):
            for ncomp in (1, 3):
                case = _labels_case(name, N, ncomp)
                prof, res = _device_profile(case)
                flags = tp.cluster_flags(case["labels"], N)
                want = envelope.row_profile(flags)
                assert np.array_equal(prof, want), (name, N, prof, want)
                if name in ("out_of_order", "reach_back") and N >= 2049:
                    assert not np.array_equal(want, tp.first_cols(flags))
                tp.check_against_closed_form(case, res, (name, N, ncomp))
                g = covariance.lnlike_grad(case["zs"], case["fl"], case["sigma"], case["amps"], case["ls"], tp.MU)
                assert res[0] == g.lnlike, (name, N, ncomp, res[0], g.lnlike)
    print("profile ok")


def _run_child(args, env_extra):
    """This file as a script in a child process: the launch switches are read once per process."""
    import subprocess
    env = dict(os.environ, **env_extra)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, HERE] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    return subprocess.run([sys.executable, "-s"] + args, env=env, capture_output=True, text=True, timeout=900)


# groups of 8 take the profile's k start, groups of 2 (the direct API's own plan at these sizes) do not
PROFILE_PLANS = {"groups-of-8": FARM_PLAN, "groups-of-2": {"PSOAP_GROUP": "2"}}


@gpu
@pytest.mark.parametrize("plan", sorted(PROFILE_PLANS))
def test_device_profile_is_the_suffix_minimum(plan):
    r = _run_child([os.path.abspath(__file__), "profile"], PROFILE_PLANS[plan])
    assert r.returncode == 0 and "profile ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


@gpu
def test_same_bits_under_the_farm_plan():
    """psoap_lnlike == the unrestricted gradient elimination's lnlike on C4-like chunks and on every constructed
    pattern, under the farm's plan (groups of 8, chain 3, no look-ahead), where the k start skips the most."""
    for script in ("test_envelope.py", "test_envelope_patterns.py"):
        r = _run_child([os.path.join(HERE, script), "same-bits"], FARM_PLAN)
        assert r.returncode == 0 and "same bits ok" in r.stdout, (script, r.stdout[-2000:] + r.stderr[-4000:])


if __name__ == "__main__" and sys.argv[1:] == ["profile"]:
    _child_profile()
