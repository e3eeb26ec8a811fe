"""The blocked Cholesky / Schur complement (psoap_schur, csrc/api.cu launch_factor) on matrices with an EXACT answer,
through every launch path the library can take.

Covariance matrices of the likelihood hide tile-level errors: most trailing-update tiles of a single-epoch chunk are
below 1e-13 max|A|, and a tile that misses part of its update can leave lnlike unchanged to 1e-10.  Here the input is

    Lfull = [[L11, 0], [L21, L22]]      integer lower triangle: off-diagonal entries uniform in [-3, 3], diagonal
                                        c + U[0, c], c = ceil(2 sqrt(n + m)) (kappa(A11) ~ 30), times 2^-e (max|A| ~ 1)
    A = Lfull Lfull^T                   exact in FP64 whatever the summation order: every partial sum is an integer
                                        (times 4^-e) below 2^53

so the factorisation of the leading n x n block A11 and the Schur complement of the border are known exactly:

    S      = A22 - A21 A11^-1 A12 = L22 L22^T
    r      = L11 z (z small integers):  residual rows -A21 A11^-1 r = -L21 z,  quad = r^T A11^-1 r = z^T z
    logdet = 2 sum log diag(L11)

Every wrong tile, dropped k-range or misplaced store moves these by orders of magnitude more than the tolerances,
which sit at least 10x above what LAPACK (scipy) achieves on the same inputs (test_harness_* check both on the CPU).
"""
import functools
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NB = 128
# Tolerances.  S: per entry, |got - S_ij| <= S_RTOL sqrt(S_ii S_jj).  Residual rows: per row, relative to
# |L21_i| |z| (the size of the terms summed).  logdet: absolute, relative to sum |log L_jj| + n (logdet itself can be
# near 0).  quad and lnlike: relative.
S_RTOL = 1e-12
RES_RTOL = 1e-12
LOGDET_RTOL = 1e-12
QUAD_RTOL = 1e-12
# Stored where no kernel may write: the strict upper triangle outside the 32 x 32 diagonal sub-blocks (warp tiles that
# straddle the diagonal compute their whole sub-block, api.cu / gemm.cuh), and the rows between Nt and ld.
SENTINEL = -1234.5


def _pad(n):
    return (n + NB - 1) // NB * NB


# ---------------------------------------------------------------------------------------------- inputs
def lfull_int(t, seed):
    """[t, t] int16 lower triangle: off-diagonal uniform in [-3, 3], diagonal c + U[0, c] with c = ceil(2 sqrt t).
    Any partial sum of A = L L^T is at most max_i |L_i|^2 <= (2c)^2 + 9 (t - 1) in magnitude (Cauchy-Schwarz)."""
    rng = np.random.default_rng(seed)
    L = np.tril(rng.integers(-3, 4, size=(t, t), dtype=np.int8), -1).astype(np.int16)
    c = int(math.ceil(2.0 * math.sqrt(t)))
    assert (2 * c) ** 2 + 9 * (t - 1) < 2 ** 53
    L[np.diag_indices(t)] = c + rng.integers(0, c + 1, size=t)
    return L


def scale_exponent(L):
    """e such that 2^-e max diag(L) is in (1/2, 1]: max|A| ~ 1."""
    return int(math.ceil(math.log2(int(np.diagonal(L).max()))))


@functools.lru_cache(maxsize=4)
def make_case(n, m, seed=None):
    """Host inputs of one case: A (float64, exact), r = L11 z, and the exact answers (read only: cached)."""
    t = n + m
    seed = n + 7 * m if seed is None else seed
    Li = lfull_int(t, seed)
    s = 2.0 ** -scale_exponent(Li)
    L = Li.astype(np.float64) * s
    A = L @ L.T                                           # exact (every partial sum an integer < 2^53, times s^2)
    z = np.random.default_rng(seed + 1).integers(-4, 5, size=n).astype(np.float64)
    return dict(n=n, m=m, A=A, r=L[:n, :n] @ z, **exact_answers(L, n, m, z))


def exact_answers(L, n, m, z):
    d = np.diagonal(L)[:n]
    return dict(S=L[n:, n:] @ L[n:, n:].T, resid=-(L[n:, :n] @ z), quad=float(z @ z), Ldiag=d.copy(),
                logdet=2.0 * math.fsum(np.log(d)), logdet_scale=2.0 * (math.fsum(np.abs(np.log(d))) + n),
                res_scale=np.sqrt((L[n:, :n] ** 2).sum(axis=1)) * math.sqrt(float(z @ z)))


# ---------------------------------------------------------------------------------------------- comparison
def errors(case, got):
    """Each observable's error in units of its tolerance (<= 1 passes)."""
    n, m = case["n"], case["m"]
    out = {}
    if m:
        S = case["S"]
        dS = np.sqrt(np.diagonal(S))
        low = np.tril_indices(m)
        e = np.abs(got["S"][low] - S[low]) / (dS[low[0]] * dS[low[1]])
        out["S"] = float(e.max()) / S_RTOL
        out["resid"] = float((np.abs(got["resid"] - case["resid"]) / case["res_scale"]).max()) / RES_RTOL
    out["logdet"] = abs(got["logdet"] - case["logdet"]) / case["logdet_scale"] / LOGDET_RTOL
    out["quad"] = abs(got["quad"] - case["quad"]) / case["quad"] / QUAD_RTOL
    lnl = -0.5 * (case["quad"] + case["logdet"])
    out["lnlike"] = abs(got["lnlike"] - lnl) / (0.5 * (case["quad"] + case["logdet_scale"])) / QUAD_RTOL
    return out


def blocked_schur(A, r, n, defect=None):
    """numpy right-looking blocked Cholesky of the leading n x n block on the padded layout the library uses (identity
    front padding, 128-wide panels, trailing update in 128 x 64 tiles).  defect = (step, row tile, 64-column tile, k0):
    that tile of that step's trailing update misses its k-columns k0..127 (a scheduling or pipeline bug)."""
    import scipy.linalg as sl
    t = A.shape[0]
    m = t - n
    Nn, Nt = _pad(n), _pad(n) + _pad(m)
    pad = Nn - n
    W = np.eye(Nt)
    idx = np.r_[pad:Nn, Nn:Nn + m]
    W[np.ix_(idx, idx)] = A
    rv = np.zeros(Nt)
    rv[pad:Nn] = r
    logdet = quad = 0.0
    for k in range(Nn // NB):
        s, rest = slice(NB * k, NB * (k + 1)), slice(NB * (k + 1), Nt)
        L = np.linalg.cholesky(W[s, s])
        logdet += 2.0 * np.log(np.diagonal(L)).sum()      # the identity padding adds log 1 = 0
        y = sl.solve_triangular(L, rv[s], lower=True)
        quad += y @ y
        P = sl.solve_triangular(L, W[rest, s].T, lower=True).T
        rv[rest] -= P @ y
        U = P @ P.T
        if defect is not None and defect[0] == k:
            _, I, J, k0 = defect
            rs, cs = slice(NB * I, NB * (I + 1)), slice(64 * J, 64 * (J + 1))
            U[rs, cs] -= P[rs, k0:] @ P[cs, k0:].T
        W[rest, rest] -= U
    return dict(S=W[Nn:Nn + m, Nn:Nn + m], resid=rv[Nn:Nn + m], logdet=logdet, quad=quad,
                lnlike=-0.5 * (quad + logdet))


def lapack_schur(case):
    import scipy.linalg as sl
    n, A = case["n"], case["A"]
    c = sl.cho_factor(A[:n, :n], lower=True)
    logdet = 2.0 * np.log(np.diagonal(c[0])).sum()
    quad = float(case["r"] @ sl.cho_solve(c, case["r"]))
    out = dict(logdet=logdet, quad=quad, lnlike=-0.5 * (quad + logdet))
    if case["m"]:
        X = sl.cho_solve(c, A[:n, n:])
        out["S"] = A[n:, n:] - A[n:, :n] @ X
        out["resid"] = -(A[n:, :n] @ sl.cho_solve(c, case["r"]))
    return out


# ---------------------------------------------------------------------------------------------- launch plan
def direct_plan(n, m, nsm, env=None):
    """What launch_factor (csrc/api.cu) does for psoap_schur(n, m) on a device with nsm SMs under the environment
    switches `env`: the group boundaries and the trailing updates (R row tiles, part, ncol1, tiles, how dealt out)."""
    env = env or {}
    Nn = _pad(n)
    Nt = Nn + _pad(m)
    Te, Tt = Nn // NB, Nt // NB
    lookahead = int(env.get("PSOAP_LOOKAHEAD", 1)) != 0
    g = int(env.get("PSOAP_GROUP", 0))
    g_group = 8 if g >= 8 else 4 if g >= 4 else 2 if g >= 2 else 1 if g == 1 else 0
    potrf = 7 if int(env.get("PSOAP_POTRF", 7)) == 7 else 3
    slots = 2 * nsm                                       # CTAS_PER_SM (gemm.cuh)
    yl = int(env.get("PSOAP_YIELD_LOOKAHEAD", 0))
    yield_mode = yl if yl in (1, 2) else (1 if Tt >= 96 else 2)
    tail = int(env.get("PSOAP_TAIL", 0)) != 0
    G = g_group or (4 if Tt >= 96 else 2)
    chain = 3 if Tt >= 192 else potrf
    lone = lookahead and chain == 7 and g_group == 0
    groups, a = [], 0
    while a < Te:
        size = min(1 if (lone and Tt - a <= 24) else G, Te - a)   # SINGLE_ROWS = 24
        groups.append((a, size))
        a += size
    updates = []
    for q, (a, size) in enumerate(groups):
        R = Tt - a - size
        nxt = q + 1 < len(groups)
        parts = [(0, 2)] if (not nxt or not lookahead) else [(1, 2 * groups[q + 1][1]), (2, 2 * groups[q + 1][1])]
        for part, ncol1 in parts:
            h = ncol1 // 2
            ntiles = R * (R + 1) if part == 0 else (R * (R + 1) if R <= h else h * (h + 1) + (R - h) * ncol1) \
                if part == 1 else ((R - h) * (R - h + 1) if R > h else 0)
            rem = ntiles % slots
            quarters = 4 * rem if (tail and part != 1 and rem > 0 and 4 * rem <= 3 * slots) else 0
            updates.append(dict(R=R, part=part, ncol1=ncol1, ntiles=ntiles, quarters=quarters,
                                persistent_rounds=(ntiles - quarters // 4) // slots))
    return dict(Te=Te, Tt=Tt, pad=Nn - n, G=G, chain=chain, groups=groups, yield_mode=yield_mode, updates=updates,
                slots=slots)


# Shapes (n, m) and what each exercises on a 148-SM B200 (default configuration; checked by test_shape_arithmetic):
SHAPES = [
    (1, 0),        # one block, front padding 127, T_elim = T_total = 1
    (1, 1),        # one data block (pad 127) under a one-block border: T_elim 1 of 2
    (128, 0),      # padding 0, T = 1
    (129, 0),      # padding 127, T = 2
    (127, 130),    # T_elim = 1 under a two-block border (pad 1, T_total 3, 126 dead border rows)
    (1000, 257),   # both ragged: pad 24, T_elim 8 of 11, 127 dead rows; single panels only (11 <= 24 rows)
    (3000, 200),   # pad 72, T_elim 24 of 26: one group of 2 (26 > 24 rows left), then single panels
    (4000, 0),     # C1's shape: pad 96, T = 32: groups of 2 at blocks 0, 2, 4, 6, then single panels
    (6000, 300),   # pad 16, T_elim 47 of 50: first bulk update 46 x 47 = 2162 tiles on 147 persistent CTAs
                   # (yield mode 2), ~15 tiles each; PSOAP_TAIL=1: 7 rounds of 296 + 90 tiles as 360 quarters
]
LARGE_SHAPES = [
    (12200, 300),  # pad 88, T_elim 96 of 99: G = 4 automatically, yield mode 1 (one tile per CTA), chain 7
    (24500, 0),    # pad 76, T = 192: chain 3 (potrf_diag3 + trsm3) on the direct path, G = 4
]
SHAPE_IDS = ["1x0-pad127", "1x1-border1", "128x0-pad0", "129x0-T2", "127x130-Telim1of3", "1000x257-ragged",
             "3000x200-group2-then-single", "4000x0-C1", "6000x300-persistent"]
LARGE_IDS = ["12200x300-G4-yield1", "24500x0-chain3"]

# Environment switches (read once per process, so each runs in a child process) and what they select.
CONFIGS = {
    "inverse-chain": {"PSOAP_POTRF": "3"},
    "group1": {"PSOAP_GROUP": "1"},
    "group4": {"PSOAP_GROUP": "4"},
    "group8": {"PSOAP_GROUP": "8"},
    "farm-sequence": {"PSOAP_LOOKAHEAD": "0", "PSOAP_POTRF": "3", "PSOAP_GROUP": "8", "PSOAP_PDL": "0"},
    "quarter-tail": {"PSOAP_TAIL": "1"},
    "yield1": {"PSOAP_YIELD_LOOKAHEAD": "1"},
    "yield2": {"PSOAP_YIELD_LOOKAHEAD": "2"},
    "no-pdl": {"PSOAP_PDL": "0"},
    "pdl-everywhere": {"PSOAP_PDL": "100000"},
    # uniform groups of 2 to the end (no single panels): the plan below 96 blocks without the single-panel tail
    "group2": {"PSOAP_GROUP": "2"},
    # chain 7 without the side stream: part-0 updates only, small tiles in the in-group column updates
    "no-lookahead": {"PSOAP_LOOKAHEAD": "0"},
    # the graph farm's sequence with rank-512 updates (ChunkFarm below 64 (proposal, chunk) pairs)
    "farm-sequence-rank512": {"PSOAP_LOOKAHEAD": "0", "PSOAP_POTRF": "3", "PSOAP_GROUP": "4", "PSOAP_PDL": "0"},
    # a captured look-ahead farm (fewer than 8 branches) that was given chain 3: side stream, no PDL
    "lookahead-farm-sequence": {"PSOAP_POTRF": "3", "PSOAP_PDL": "0"},
    # the direct plan from 192 blocks on (chain 3, G = 4, one tile per CTA in the bulk update)
    "plan-from-192-blocks": {"PSOAP_POTRF": "3", "PSOAP_GROUP": "4", "PSOAP_YIELD_LOOKAHEAD": "1"},
    # the direct plan from 96 blocks on without its single-panel end (chain 7, G = 4, one tile per CTA)
    "group4-yield1": {"PSOAP_GROUP": "4", "PSOAP_YIELD_LOOKAHEAD": "1"},
}
# the pivot-failure cases run under both chains: potrf_diag7 + trsm7 (default below 192 blocks) and potrf_diag3 + trsm3
PIVOT_CONFIGS = ("inverse-chain", "farm-sequence")


def pivot_rows(n):
    """Data rows whose pivot is made exactly -L_jj^2 (shape (4000, 0): pad 96, groups of 2 at the start)."""
    pad = _pad(n) - n
    return [0, NB - pad - 1, NB - pad, 3 * NB - pad + 50, n - 1]   # block 3 = second panel of the second group


# ---------------------------------------------------------------------------------------------- CPU self-test
def test_harness_construction_is_exact():
    """float64 BLAS product == int64 product, for the inputs as built, and the partial-sum bound holds at every size
    the GPU tests use."""
    Li = lfull_int(700, 5)
    s = 2.0 ** -scale_exponent(Li)
    L = Li.astype(np.float64) * s
    A = L @ L.T
    Ai = Li.astype(np.int64) @ Li.astype(np.int64).T
    assert np.array_equal(A, Ai.astype(np.float64) * (s * s))
    assert 0.25 < np.abs(A).max() < 4.0
    z = np.random.default_rng(6).integers(-4, 5, size=700)
    assert np.array_equal(L @ z.astype(np.float64), (Li.astype(np.int64) @ z) * s)
    for n, m in SHAPES + LARGE_SHAPES:          # the Cauchy-Schwarz bound of every size used (lfull_int asserts it)
        c = int(math.ceil(2.0 * math.sqrt(n + m)))
        assert (2 * c) ** 2 + 9 * (n + m - 1) < 2 ** 53


@pytest.mark.parametrize("n,m", [(1000, 257), (3000, 200)])
def test_harness_condition_number(n, m):
    ev = np.linalg.eigvalsh(make_case(n, m)["A"][:n, :n])
    assert ev[0] > 0 and ev[-1] / ev[0] <= 1e4, ev[-1] / ev[0]


@pytest.mark.parametrize("n,m", [(127, 130), (1000, 257), (3000, 200), (1000, 0)])
def test_harness_lapack_headroom(n, m):
    """scipy's LAPACK Cholesky meets every tolerance with at least 10x to spare."""
    case = make_case(n, m)
    err = errors(case, lapack_schur(case))
    assert max(err.values()) <= 0.1, err


@pytest.mark.parametrize("n,m,defect", [(1000, 257, (0, 9, 3, 112)), (1000, 257, (0, 4, 5, 112)),
                                        (1000, 257, (3, 2, 5, 112)), (1000, 257, (7, 2, 4, 112)),
                                        (1000, 0, (2, 4, 1, 112))],
                         ids=["cross-tile-step0", "data-tile-step0", "diagonal-tile-step3", "schur-diagonal-tile-step7",
                              "m0-data-tile-step2"])
def test_harness_detects_dropped_k_columns(n, m, defect):
    """The correct numpy blocked Cholesky passes; with ONE 128 x 64 tile of one step's trailing update missing its last
    16 k-columns it fails by at least 100x, also where only logdet / quad / lnlike are observed (m = 0).  Tiles are
    relative to the step's trailing matrix (row tile, 64-column tile)."""
    case = make_case(n, m)
    good = errors(case, blocked_schur(case["A"], case["r"], n))
    assert max(good.values()) <= 0.1, good
    bad = errors(case, blocked_schur(case["A"], case["r"], n, defect))
    assert max(bad.values()) >= 100.0, bad


def test_shape_arithmetic():
    """The launch decisions each shape is meant to exercise (SHAPES comments), on a 148-SM B200."""
    p = {s: direct_plan(*s, nsm=148) for s in SHAPES + LARGE_SHAPES}
    assert [(p[s]["Te"], p[s]["Tt"], p[s]["pad"]) for s in SHAPES[:5]] == \
        [(1, 1, 127), (1, 2, 127), (1, 1, 0), (2, 2, 127), (1, 3, 1)]
    assert p[(1000, 257)]["groups"] == [(a, 1) for a in range(8)] and p[(1000, 257)]["Tt"] == 11
    assert p[(3000, 200)]["groups"] == [(0, 2)] + [(a, 1) for a in range(2, 24)]
    assert p[(4000, 0)]["groups"][:5] == [(0, 2), (2, 2), (4, 2), (6, 2), (8, 1)] and p[(4000, 0)]["pad"] == 96
    six = p[(6000, 300)]
    assert (six["Te"], six["Tt"], six["yield_mode"], six["updates"][1]["ntiles"]) == (47, 50, 2, 2162)
    assert six["updates"][1]["ntiles"] // 147 >= 14                  # each persistent CTA loops over many tiles
    big = p[(12200, 300)]
    assert (big["Te"], big["Tt"], big["G"], big["yield_mode"], big["chain"]) == (96, 99, 4, 1, 7)
    assert p[(24500, 0)]["chain"] == 3 and p[(24500, 0)]["Tt"] == 192
    # under PSOAP_TAIL=1 the 6000 x 300 bulk update is 7 persistent rounds of 296 tiles + 90 tiles as 360 quarters
    t = direct_plan(6000, 300, 148, CONFIGS["quarter-tail"])["updates"][1]
    assert (t["persistent_rounds"], t["quarters"]) == (7, 360)


def test_pivot_rows_land_where_meant():
    rows = pivot_rows(4000)
    pad = _pad(4000) - 4000
    blocks = [(j + pad) // NB for j in rows]
    assert blocks == [0, 0, 1, 3, 31] and (rows[1] + pad) % NB == NB - 1 and (rows[2] + pad) % NB == 0
    assert direct_plan(4000, 0, 148)["groups"][1] == (2, 2)          # block 3 is the second panel of its group
    assert direct_plan(4000, 0, 148, CONFIGS["inverse-chain"])["groups"][1] == (2, 2)


# ---------------------------------------------------------------------------------------------- GPU harness
def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def bordered(n, m, A, ld_extra=0):
    """S laid out as covariance._Bordered does (identity front padding, border from row padded(n), unit diagonal on
    the dead rows), with SENTINEL where no kernel may write.  Returns the row-major tensor St [Nt, Nt + ld_extra],
    S(i, j) = St[j, i], and the mask of the sentinel entries.  A: [n + m, n + m] (numpy or CUDA tensor)."""
    torch = _torch()
    from psoap_b200.covariance import _Bordered
    B = _Bordered(n, m)
    Ad = A if isinstance(A, torch.Tensor) else torch.from_numpy(A).cuda()
    B.data_block().copy_(Ad[:n, :n])
    if m:
        B.cross_block(0, m).copy_(Ad[n:, :n].T)
        B.border_block(0, m).copy_(Ad[n:, n:])
    Nt = B.Nt
    ar = torch.arange(Nt, device="cuda")
    # St[j, i] with i < j (upper triangle of S), outside the 32 x 32 diagonal sub-blocks
    mask = (ar[None, :] < ar[:, None]) & ((ar[None, :] // 32) != (ar[:, None] // 32))
    St = torch.full((Nt, Nt + ld_extra), SENTINEL, dtype=torch.float64, device="cuda")
    St[:, :Nt] = B.St.masked_fill_(mask, SENTINEL)
    del B
    return St, mask


def run_schur(n, m, St, r, key="exact"):
    """psoap_schur on St (leading dimension St.shape[1]) with the residual r [n] (device); returns the observables.
    The workspace is the same buffer on every call with the same key."""
    import ctypes
    torch = _torch()
    from psoap_b200 import _lib
    lib = _lib.load()
    Nn, Nt = _pad(n), _pad(n) + _pad(m)
    nbytes = lib.psoap_schur_workspace_bytes(n, m)
    ws = _lib.workspace(nbytes + 256, key)
    rv, acc, info = _lib.vp(), _lib.vp(), _lib.vp()
    _lib.check(lib.psoap_schur_views(_lib.ptr(ws), n, m, ctypes.byref(rv), ctypes.byref(acc), ctypes.byref(info)))
    base = ws.data_ptr()
    r_view = ws[rv.value - base: rv.value - base + Nt * 8].view(torch.float64)
    r_view.zero_()
    r_view[Nn - n:Nn] = r
    ws[acc.value - base: acc.value - base + 64].zero_()
    ws[info.value - base: info.value - base + 8].zero_()
    res = torch.full((4,), 7.0, dtype=torch.float64, device="cuda")
    rc = lib.psoap_schur(_lib.ptr(St), St.shape[1], n, m, _lib.ptr(ws), nbytes, _lib.ptr(res), _lib.stream_ptr())
    torch.cuda.synchronize()
    out = res.cpu().numpy()
    return dict(rc=rc, lnlike=float(out[0]), logdet=float(out[1]), quad=float(out[2]), info=float(out[3]),
                r_tail=r_view[Nn:].cpu().numpy())


def check_case(name, n, m, A, r, exact, ld_extra=0):
    """One psoap_schur call against the exact answers; raises AssertionError with the case name."""
    Nn, Nt = _pad(n), _pad(n) + _pad(m)
    St, mask = bordered(n, m, A, ld_extra)
    got = run_schur(n, m, St, r)
    assert got["rc"] == 0, (name, got["rc"])
    assert got["info"] == 0.0, (name, got["info"])
    # trailing block: S(Nn + a, Nn + b) = St[Nn + b, Nn + a]; lower triangle = upper triangle of St's block
    T = St[Nn:Nt, Nn:Nt].T.cpu().numpy()
    got["S"] = T[:m, :m]
    got["resid"] = got["r_tail"][:m]
    err = errors(exact, got)
    assert max(err.values()) <= 1.0, (name, err)
    dead = np.tril(T)[m:, :]
    assert np.array_equal(dead, np.tril(np.eye(Nt - Nn))[m:, :]), (name, "dead border rows")
    assert not got["r_tail"][m:].any(), (name, "residual of dead rows")
    # nothing stored above the diagonal (outside the 32 x 32 diagonal sub-blocks) nor between Nt and ld
    assert not bool(((St[:, :Nt] != SENTINEL) & mask).any()), (name, "store above the diagonal")
    if ld_extra:
        assert bool((St[:, Nt:] == SENTINEL).all()), (name, "store between Nt and ld")
    return err


def check_pivot_failure(name, n, A, r, exact, j):
    """A_jj - 2 L_jj^2 makes pivot j exactly -L_jj^2: info = j + 1 (1-based data row), lnlike = -inf, return code 0;
    then the valid matrix on the same workspace must be exact again."""
    torch = _torch()
    Ad = A.clone() if isinstance(A, torch.Tensor) else torch.from_numpy(A).cuda()
    Ljj = float(exact["Ldiag"][j])
    Ad[j, j] -= 2.0 * Ljj * Ljj
    St, _ = bordered(n, 0, Ad)
    got = run_schur(n, 0, St, r)
    assert got["rc"] == 0 and got["info"] == j + 1 and got["lnlike"] == -np.inf, (name, j, got["info"], got["lnlike"])
    check_case(name + "-after", n, 0, A, r, exact)


def _load_case(path):
    with np.load(path) as f:
        case = {k: f[k] for k in f.files}
    for k in ("n", "m"):
        case[k] = int(case[k])
    for k in ("quad", "logdet", "logdet_scale"):
        case[k] = float(case[k])
    return case


def run_stored_cases(case_dir, names):
    """Runs the named cases stored by the parent in case_dir (also the entry of the child processes).  Names:
    '<n>x<m>' (ld = Nt), '<n>x<m>-ld' (ld = Nt + 2), '<n>x<m>-pivot<j>'."""
    torch = _torch()
    done = []
    for name in names:
        base, _, variant = name.partition("-")
        case = _load_case(os.path.join(case_dir, base + ".npz"))
        n, m = case["n"], case["m"]
        r = torch.from_numpy(case["r"]).cuda()
        if variant.startswith("pivot"):
            check_pivot_failure(name, n, case["A"], r, case, int(variant[5:]))
        else:
            check_case(name, n, m, case["A"], r, case, ld_extra=2 if variant == "ld" else 0)
        done.append(name)
    return done


def store_case(case_dir, n, m):
    np.savez(os.path.join(case_dir, f"{n}x{m}.npz"), **make_case(n, m))


@pytest.fixture(scope="module")
def case_dir(tmp_path_factory):
    """The host-built inputs of SHAPES, written once and read by this process and by the child processes."""
    d = tmp_path_factory.mktemp("exact_cases")
    for n, m in SHAPES:
        store_case(str(d), n, m)
    return str(d)


def _names(pivots):
    names = [f"{n}x{m}" for n, m in SHAPES] + ["1000x257-ld", "4000x0-ld"]
    if pivots:
        names += [f"4000x0-pivot{j}" for j in pivot_rows(4000)]
    return names


# ---------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_schur_exact_default(shape, case_dir):
    n, m = shape
    run_stored_cases(case_dir, [f"{n}x{m}"])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1000, 257), (4000, 0)], ids=["1000x257", "4000x0"])
def test_schur_exact_leading_dimension(shape, case_dir):
    """ld = Nt + 2: the two rows between Nt and ld of every column are never written."""
    n, m = shape
    run_stored_cases(case_dir, [f"{n}x{m}-ld"])


@pytest.mark.gpu
@pytest.mark.parametrize("j", pivot_rows(4000), ids=["row0", "last-of-block0", "first-of-block1",
                                                     "second-panel-of-group", "last-row"])
def test_pivot_failure_reports_lapack_index(j, case_dir):
    """Chain 7 (the default below 192 blocks); chain 3 in test_schur_exact_launch_paths."""
    run_stored_cases(case_dir, [f"4000x0-pivot{j}"])


def _gpu_case(n, m, seed):
    """A large case built on the GPU (torch FP64 matmul of the integer factor: exact as on the host), with some rows
    checked against an int64 product on the host."""
    torch = _torch()
    t = n + m
    Li = lfull_int(t, seed)
    e = scale_exponent(Li)
    s = 2.0 ** -e
    L = torch.from_numpy(Li).cuda().to(torch.float64).mul_(s)
    A = L @ L.T
    rows = [0, n - 1, t - 1, t // 3]
    for i in rows:
        want = np.zeros(t, dtype=np.int64)
        li = Li[i, :i + 1].astype(np.int64)
        for k0 in range(0, i + 1, 4096):
            k1 = min(i + 1, k0 + 4096)
            want += Li[:, k0:k1].astype(np.int64) @ li[k0:k1]
        assert np.array_equal(A[i].cpu().numpy(), want.astype(np.float64) * (s * s)), ("row", i)
    z = torch.from_numpy(np.random.default_rng(seed + 1).integers(-4, 5, size=n).astype(np.float64)).cuda()
    r = L[:n, :n] @ z
    d = np.diagonal(Li)[:n] * s
    exact = dict(n=n, m=m, quad=float((z @ z).item()), logdet=2.0 * math.fsum(np.log(d)), Ldiag=d,
                 logdet_scale=2.0 * (math.fsum(np.abs(np.log(d))) + n))
    if m:
        L22, L21 = L[n:, n:], L[n:, :n]
        exact["S"] = (L22 @ L22.T).cpu().numpy()
        exact["resid"] = (-(L21 @ z)).cpu().numpy()
        exact["res_scale"] = (torch.sqrt((L21 ** 2).sum(dim=1)) * math.sqrt(exact["quad"])).cpu().numpy()
    del L
    return A, r, exact


@pytest.mark.gpu
@pytest.mark.parametrize("shape", LARGE_SHAPES, ids=LARGE_IDS)
def test_schur_exact_large(shape):
    torch = _torch()
    n, m = shape
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    plan = direct_plan(n, m, nsm)
    assert plan["chain"] == (3 if plan["Tt"] >= 192 else 7)
    A, r, exact = _gpu_case(n, m, seed=n + 7 * m)
    check_case(f"{n}x{m}", n, m, A, r, exact)
    del A
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS), ids=list(CONFIGS))
def test_schur_exact_launch_paths(config, case_dir):
    """Every shape up to 6000 (+ the ld = Nt + 2 cases, + the pivot failures under chain 3) in a child process with
    the environment switch set: they are read once per process."""
    torch = _torch()
    env = CONFIGS[config]
    if config == "quarter-tail":
        nsm = torch.cuda.get_device_properties(0).multi_processor_count
        ups = [u for s in SHAPES for u in direct_plan(*s, nsm=nsm, env=env)["updates"]]
        assert any(u["quarters"] and u["persistent_rounds"] >= 1 for u in ups), "no shape reaches the quarter-tile tail"
    names = _names(pivots=config in PIVOT_CONFIGS)
    child_env = dict(os.environ, **env)
    code = ("import sys, json; sys.path.insert(0, %r); import test_factor_exact as t; "
            "print('DONE', json.dumps(t.run_stored_cases(%r, %r)))") % (os.path.dirname(__file__), case_dir, names)
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=child_env, capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    done = json.loads(out.stdout.split("DONE", 1)[1])
    assert done == names


@pytest.mark.gpu
def test_farm_rank1024_graph_vs_oracle(oracle):
    """The farm's shipped configuration (chain 3, rank-1024 updates with G = 8, graph replay), which ChunkFarm picks
    for 64 (proposal, chunk) pairs or more: 16 multi-epoch SB2 chunks of N = 960 .. 1360 (a full 8-panel group, and a
    partial one from N = 1025) x 4 proposals, each pair against the CPU oracle."""
    from psoap_b200 import synthetic
    from psoap_b200.farm import ChunkFarm
    chunks = [synthetic.make_chunk("SB2", 8, 120 + (50 * i) // 15, seed=1200 + i) for i in range(16)]
    assert [c["N"] for c in chunks][::15] == [960, 1360]
    p = synthetic.default_params("SB2")
    P = np.stack([p * (1.0 + 0.02 * k * np.array([0, 1, 0, 0, 0, 0, 0, 1, -1, 0, 1])) for k in range(4)])
    farm = ChunkFarm("SB2", chunks, n_proposals=4)
    assert farm.n_chunks * farm.n_proposals == 64
    per = farm.chunk_lnlikes(P).cpu().numpy().copy()
    farm.close()
    for k in range(4):
        _, ref = oracle.farm_lnprob("SB2", P[k], chunks)
        assert np.all(np.abs(per[k] - ref) <= 1e-10 * np.abs(ref)), (k, per[k], ref)

