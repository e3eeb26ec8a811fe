"""Every kernel that writes covariance entries, against a correctly rounded exponential, at ulp tolerance.

An entry is sum_c amp_c^2 exp_neg((p2_c r) r), r = z_j - z_i, p2 = -0.5 c^2 / l^2 (common.cuh se_term), and exp_neg is
the project's own table-driven exponential.  The host reproduces the device's rounded arguments bit for bit in plain
float64 numpy (numpy does not contract into FMA): amp2 = amp * amp, p2 = (-0.5 c^2) / (l * l), r = zj - zi,
x = (p2 * r) * r, and for the fused Doppler path z = lwl + (-v) / c.  The reference is the exact exponential AT THE
REALISED x, so the error measured is exp_neg's (and the sum's), never the rounding of its argument.  Exact values are
long double (64-bit significand: numpy's exp is the C library's expl) where the host has it, otherwise mpmath at 40
digits on a fixed subsample of 2^16 entries; the edge points are checked with mpmath everywhere.  numpy's float64 exp
is not a reference here: it is not correctly rounded everywhere.

Errors are in units of ulp(RN(exact)), where a subnormal or zero RN(exact) has ulp 2^-1074.  The bounds:

  single term, amp = 1 (amp2 = 1, so the entry IS exp_neg(x)):
      |got - e| <= SINGLE_ULP = 1.5 ulp,  got == 0 iff RN(e) == 0,  NaN in -> NaN out.
      (exp_neg reaches 1.27 ulp on a host copy of it, 34754 of 2e7 uniform samples above 1 ulp: 1 ulp is not its bound.)
  full entry S = sum_c amp2_c e_c, summed in component order, every amp <= 1 (see full_bound):
      |got - S| <= (2 + (ncomp - 1) / 2) 2^-52 S + 2 ncomp 2^-1074.
  diagonals bit-exact with the host: sum amp2 (fill_full), sum amp2 + sigma^2 (fill_lower), + nugget (predict mode 1).

The 1e-12 relative tolerances of test_gpu_parity.py are the parity contract with the reference CPU code; they are
about 4500 ulp wide and their 1e-300 floor accepts anything for x in [-745, -690].  This file holds the kernels to what
exp_neg actually promises, at the points where a table-driven exponential goes wrong: the exact-zero threshold
(x = ln 2^-1075), the normal/subnormal boundary (ln 2^-1022), the table-interval edges k ln2 / 64, the -750 clamp,
x = -0 and tiny x, far pairs, and a uniform sweep over [-760, 0].

CPU: the harness itself (named points hit exactly, the ulp helper on hand-worked cases, the long-double reference
against mpmath at the edge points).
GPU (-m gpu): fill_v12_kernel (psoap_fill_v12 / psoap_fill_v12n, ncomp 1 to 3, ragged shapes, ld > N, a NaN column),
fill_full_kernel (psoap_fill_v11), fill_lower_kernel (psoap_debug_fill_lower, pre-shifted and fused Doppler path, with
and without front padding), the prediction's border fill (psoap_predict modes 0 and 1, and the farm's
predict_border_farm_kernel through ChunkFarm.predict_components) with data so far from the grid that Sigma is the
border block itself; the same entries from all of them compared with ==; and the exact-zero threshold end to end, through
the likelihood's envelope and the Fisher information's tile flags.
"""
import ctypes
import functools
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from psoap_b200 import envelope  # noqa: E402

gpu = pytest.mark.gpu
C_KMS = 2.99792458e5
TINY = np.ldexp(1.0, -1074)               # the least subnormal: ulp of every subnormal and of 0
MIN_NORMAL = np.ldexp(1.0, -1022)
SINGLE_ULP = 1.5
LD = np.finfo(np.longdouble).nmant >= 63  # x86 80-bit long double; some aarch64 hosts have only float64
SUBSAMPLE = 1 << 16                       # entries per check evaluated by mpmath when long double is not wide enough
SENTINEL = -7.0                           # what the buffers hold where a kernel must not write
L0 = 5.0                                  # the length scale the named points are aimed with (km/s)
X_SWEEP = -760.0                          # the uniform sweep runs over [X_SWEEP, 0]: past the clamp at -750


# ---------------------------------------------------------------------------------------------- realised arguments
def p2_of(l):
    """p2 = -0.5 c^2 / l^2 as gp_coeffs rounds it: (-0.5 * C_KMS2) / (l * l)."""
    return (-0.5 * (C_KMS * C_KMS)) / (l * l)


def realised_x(zr, zc, l):
    """x[i, j] = (p2 r) r with r = zc[j] - zr[i], rounded as se_term rounds it."""
    p2 = p2_of(l)
    r = np.asarray(zc, dtype=np.float64)[None, :] - np.asarray(zr, dtype=np.float64)[:, None]
    return (p2 * r) * r


def shifted(lwl, vel_c, epoch):
    """z_at's fused Doppler shift: lwl + (-v) / c, per pixel."""
    return np.asarray(lwl) + (-np.asarray(vel_c)[np.asarray(epoch)]) / C_KMS


# ---------------------------------------------------------------------------------------------- exact values
def _mp():
    import mpmath
    return mpmath


def mp_rn(v):
    """RN(v) to float64 for an mpmath number v >= 0 (subnormals rounded on the 2^-1074 grid, ties to even)."""
    mpmath = _mp()
    if mpmath.isnan(v):
        return np.nan
    if v == 0:
        return 0.0
    if v < MIN_NORMAL:
        with mpmath.workprec(200):
            k = int(mpmath.nint(v * mpmath.mpf(2) ** 1074))   # nint: ties to even
        return float(np.ldexp(float(k), -1074))
    with mpmath.workprec(53):
        return float(+v)


def mp_exp(x):
    """exp(x) at 40 digits for a float64 x (exact arithmetic on the double's value)."""
    mpmath = _mp()
    with mpmath.workdps(40):
        return mpmath.exp(mpmath.mpf(float(x)))


def rn_of(k_ln2, div=1):
    """RN(-k ln 2 / div) from 200-bit arithmetic."""
    mpmath = _mp()
    with mpmath.workprec(200):
        v = -mpmath.mpf(k_ln2) * mpmath.log(2) / div
    with mpmath.workprec(53):
        return float(+v)


def exp_hp(x):
    """exp(x), elementwise, in high precision: long double, or (fallback) an object array of 40-digit mpmath numbers."""
    x = np.asarray(x, dtype=np.float64)
    if LD:
        return np.exp(x.astype(np.longdouble))
    return np.array([mp_exp(v) for v in x.ravel()], dtype=object).reshape(x.shape)


def rn(S):
    """RN(S) to float64 for a high-precision array."""
    if S.dtype == object:
        return np.array([mp_rn(v) for v in S.ravel()], dtype=np.float64).reshape(S.shape)
    return S.astype(np.float64)


def ulp(y):
    """ulp of a float64 y: the spacing above |y|; 2^-1074 for subnormals and zero."""
    return np.spacing(np.abs(np.asarray(y, dtype=np.float64)))


def ulp_err(got, S):
    """|got - S| in units of ulp(RN(S)), as float64 (got float64, S high precision)."""
    got = np.asarray(got, dtype=np.float64)
    d = np.abs((got.astype(object) if S.dtype == object else got.astype(np.longdouble)) - S)
    return np.asarray(d / ulp(rn(S)), dtype=np.float64)


def full_bound(S, ncomp):
    """|got - S| allowed for a full entry S = sum_c amp2_c e_c (every amp2_c <= 1), summed in component order:
         exp_neg:      |y_c - e_c| <= 1.5 ulp(RN(e_c)) <= 1.5 (2^-52 e_c + 2^-1074)  (ulp = 2^-1074 when RN(e_c) is subnormal)
         product:      t_c = RN(amp2_c y_c): + 0.5 ulp, <= 2^-53 amp2_c y_c + 2^-1075
         so a term:    |t_c - amp2_c e_c| <= 2 2^-52 amp2_c e_c + 2 2^-1074           (amp2_c <= 1; first order in 2^-52)
         ncomp - 1 additions of non-negative terms: each <= 2^-53 of a partial sum <= S (subnormal sums are exact)
       total (2 + (ncomp - 1) / 2) 2^-52 S + 2 ncomp 2^-1074."""
    tiny = np.longdouble(TINY) if S.dtype != object else TINY
    return (2.0 + (ncomp - 1) / 2.0) * 2.0 ** -52 * S + 2 * ncomp * tiny


# ---------------------------------------------------------------------------------------------- bound checks
STATS = {}


def _record(kind, kernel, ncomp, err, R, zero_mismatch):
    """kind "single": exp_neg's own error (one live term, amp = 1); "full": a whole entry's, in ulps of RN(S)."""
    s = STATS.setdefault((kernel, ncomp, kind), dict(n=0, max=0.0, max_sub=0.0, zero_mismatch=0))
    s["n"] += err.size
    if err.size:
        s["max"] = max(s["max"], float(err.max()))
        sub = R < MIN_NORMAL
        if sub.any():
            s["max_sub"] = max(s["max_sub"], float(err[sub].max()))
    s["zero_mismatch"] += int(zero_mismatch)


def report(kernel):
    for (k, nc, kind), s in sorted(STATS.items()):
        if k == kernel:
            print("%-20s ncomp %d %-6s entries %9d  max %.4f ulp  subnormal band max %.4f ulp  zero-set mismatches %s"
                  % (k, nc, kind, s["n"], s["max"], s["max_sub"], s["zero_mismatch"] if kind == "single" else "-"))


def _subsample(n):
    return slice(None) if LD or n <= SUBSAMPLE else np.linspace(0, n - 1, SUBSAMPLE).astype(np.int64)


def check_single(got, x, kernel, ncomp, tag=""):
    """One live term with amp = 1: |got - exp(x)| <= 1.5 ulp, got == 0 iff RN(exp x) == 0, NaN iff x is NaN."""
    got, x = np.asarray(got, dtype=np.float64).ravel(), np.asarray(x, dtype=np.float64).ravel()
    assert np.array_equal(np.isnan(got), np.isnan(x)), (kernel, ncomp, tag, "NaN in, NaN out")
    keep = ~np.isnan(x)
    got, x = got[keep], x[keep]
    idx = _subsample(got.size)
    got, x = got[idx], x[idx]
    e = exp_hp(x)
    R = rn(e)
    err = ulp_err(got, e)
    zm = np.count_nonzero((got == 0.0) != (R == 0.0))
    _record("single", kernel, ncomp, err, R, zm)
    assert zm == 0, (kernel, ncomp, tag, "zero set", x[(got == 0.0) != (R == 0.0)][:8])
    bad = err > SINGLE_ULP
    assert not bad.any(), (kernel, ncomp, tag, float(err.max()), x[bad][:8], got[bad][:8])


def check_full(got, xs, amps, kernel, tag=""):
    """Full entries sum_c amp_c^2 exp(x_c) within full_bound of the exact sum."""
    ncomp = len(xs)
    assert all(0.0 <= a <= 1.0 for a in amps)
    got = np.asarray(got, dtype=np.float64).ravel()
    xs = [np.asarray(x, dtype=np.float64).ravel() for x in xs]
    assert not np.isnan(got).any(), (kernel, ncomp, tag)
    idx = _subsample(got.size)
    got, xs = got[idx], [x[idx] for x in xs]
    S = 0
    for x, a in zip(xs, amps):
        S = S + (a * a) * exp_hp(x)           # amp2 = RN(a * a), as gp_coeffs; the product with e in high precision
    S = np.asarray(S)
    if S.dtype != object:
        S = S.astype(np.longdouble)
    dev = np.abs((got.astype(object) if S.dtype == object else got.astype(np.longdouble)) - S)
    ok = np.asarray(dev <= full_bound(S, ncomp), dtype=bool)
    _record("full", kernel, ncomp, ulp_err(got, S), rn(S), 0)
    assert ok.all(), (kernel, ncomp, tag, np.flatnonzero(~ok)[:8], got[~ok][:8])


def check_matrix_full(got, zr, zc, amps, ls, kernel, mask=None, tag=""):
    """check_full over a matrix, given the rows' and columns' z per component; mask picks the entries checked."""
    xs = [realised_x(r, c, l) for r, c, l in zip(zr, zc, ls)]
    if mask is None:
        check_full(got, xs, amps, kernel, tag)
    else:
        check_full(got[mask], [x[mask] for x in xs], amps, kernel, tag)


# ---------------------------------------------------------------------------------------------- argument generator
def _neighbours(x, k):
    """x and its k float64 neighbours on each side, ascending."""
    lo, hi = [x], [x]
    for _ in range(k):
        lo.insert(0, np.nextafter(lo[0], -np.inf))
        hi.append(np.nextafter(hi[-1], np.inf))
    return lo[:-1] + hi


X_ZERO = rn_of(1075)                       # RN(ln 2^-1075) = -745.1332191019412: RN(exp x) is 0 at and below it
X_SUBNORMAL = rn_of(1022)                  # RN(ln 2^-1022) = -708.3964185322641: the normal/subnormal boundary
TABLE_K = [k for k in list(range(1, 65)) + [64 * e + j for e in (7, 200, 1000, 1022, 1050, 1074) for j in range(64)]
           if k <= 68806]                  # every table index j at seven exponents, up to the zero threshold


def named_targets():
    """name -> the realised arguments x the generator must hit exactly."""
    t = {"zero_threshold": _neighbours(X_ZERO, 3),
         "subnormal_boundary": _neighbours(X_SUBNORMAL, 3),
         "table_edges": [y for k in TABLE_K for y in _neighbours(rn_of(k, 64), 1)],
         "clamp": _neighbours(-750.0, 2),
         "tiny": [-1e-300],
         "far": [-9e4]}
    return {k: np.array(v, dtype=np.float64) for k, v in t.items()}


def aim(targets, l0=L0, lsteps=16, rsteps=6):
    """(l, r) per target x with (p2(l) r) r == x exactly: r within rsteps ulps of sqrt(x / p2), l from l0 and its next
    doubles up (one r lattice reaches about every other double x; neighbouring p2 shift it).  NaN where nothing hits."""
    t = np.asarray(targets, dtype=np.float64)
    L, R = np.full(t.size, np.nan), np.full(t.size, np.nan)
    l = l0
    for _ in range(lsteps):
        todo = np.flatnonzero(np.isnan(L))
        if not todo.size:
            break
        p2 = p2_of(l)
        r0 = np.sqrt(t[todo] / p2)
        for direction in (np.inf, -np.inf):
            r = r0.copy()
            for _ in range(rsteps):
                hit = ((p2 * r) * r == t[todo]) & np.isnan(L[todo])
                L[todo[hit]], R[todo[hit]] = l, r[hit]
                r = np.nextafter(r, direction)
        l = np.nextafter(l, np.inf)
    return L, R


@functools.lru_cache(maxsize=None)
def named_points(l0=L0):
    """name -> (l, r, x target) arrays, aimed from l0; x = -0 comes from r = 0."""
    out = {}
    for name, t in named_targets().items():
        L, R = aim(t, l0)
        out[name] = (L, R, t)
    out["zero"] = (np.array([l0]), np.array([0.0]), np.array([-0.0]))
    return out


def sweep_r(n, l, rng, x_lo=X_SWEEP):
    """n values of r, random sign, whose x = p2(l) r^2 is uniform over [x_lo, 0]."""
    x = rng.uniform(x_lo, 0.0, n)
    return np.sqrt(x / p2_of(l)) * rng.choice([-1.0, 1.0], n)


def v12_vectors(M, N, l, rng):
    """rows: z = 0 first (r is then the column value exactly), then z near 8.5 (the subtraction is exercised); columns
    alternate between r values of a uniform x sweep (against the z = 0 row) and 8.5 + r (against the 8.5 rows), so that
    every row meets the whole sweep and the pairs across the two groups are far (x ~ -1e11, exactly 0)."""
    R = np.sqrt(X_SWEEP / p2_of(l))
    rows = np.concatenate([[0.0], 8.5 + rng.uniform(-0.02 * R, 0.02 * R, M - 1)])
    r = sweep_r(N, l, rng)
    cols = np.where(np.arange(N) % 2 == 0, r, 8.5 + r)
    return rows, cols


def sym_vector(N, l, rng):
    """One ln-wavelength vector for the symmetric fills: z = 0, aimed r values hit with l (against that z = 0 pixel), and
    a jittered 8.5 + run whose neighbours out to ~40 pixels cover x in [-800, 0]."""
    aimed = np.concatenate([R[L == l] for L, R, _ in named_points(l).values()])
    aimed = aimed[rng.permutation(aimed.size)]
    n1 = min(max(N - 1, 0), N // 4)
    aimed = np.concatenate([aimed, sweep_r(n1, l, rng)])
    R = np.sqrt(-800.0 / p2_of(l))
    run = 8.5 + np.arange(N) * (R / 40.0) + rng.uniform(0.0, R / 80.0, N)
    z = run.copy()
    if N:
        z[0] = 0.0
        z[1:1 + n1] = aimed[:n1] * rng.choice([-1.0, 1.0], n1)
    return z


# ---------------------------------------------------------------------------------------------- CPU
def test_named_points_are_hit():
    """Every named argument is realised exactly by an (l, r) pair, with few distinct l; x = -0 has its sign."""
    pts = named_points()
    assert set(pts) == {"zero_threshold", "subnormal_boundary", "table_edges", "clamp", "tiny", "far", "zero"}
    ls = set()
    for name, (L, R, t) in pts.items():
        assert not np.isnan(L).any(), (name, t[np.isnan(L)])
        for l in np.unique(L):
            sel = L == l
            x = (p2_of(l) * R[sel]) * R[sel]
            assert np.array_equal(x, t[sel]) and np.array_equal(np.signbit(x), np.signbit(t[sel])), name
            ls.add(float(l))
    assert len(ls) <= 16, sorted(ls)
    assert X_ZERO == -745.1332191019412 and X_SUBNORMAL == -708.3964185322641
    assert len(pts["zero_threshold"][2]) == 7 and len(set(pts["zero_threshold"][2])) == 7
    # the table edges cover every table index j at the far end and inside the subnormal band
    ks = np.array(TABLE_K)
    assert set(ks % 64) == set(range(64)) and (-ks * np.log(2) / 64 <= X_SUBNORMAL).sum() >= 3 * 64
    rng = np.random.default_rng(0)
    x = realised_x([0.0], sweep_r(1 << 14, L0, rng), L0)
    assert x.min() >= X_SWEEP * (1 + 1e-12) and (x < -750.0).any() and ((x < X_SUBNORMAL) & (x > X_ZERO)).sum() > 200


def test_ulp_helper_by_hand():
    """ulp of 1, of a subnormal, of 0; RN(exp x) switches from 0 to 2^-1074 between X_ZERO and the double above it, and
    to the normal range at X_SUBNORMAL; errors of hand-picked values in ulps."""
    assert ulp(1.0) == 2.0 ** -52 and ulp(0.0) == TINY and ulp(3 * TINY) == TINY and ulp(MIN_NORMAL) == TINY
    assert ulp(np.nextafter(1.0, 0.0)) == 2.0 ** -53
    up = np.nextafter(X_ZERO, 0.0)
    e = exp_hp(np.array([X_ZERO, up]))
    assert np.array_equal(rn(e), [0.0, TINY])
    assert mp_rn(mp_exp(X_ZERO)) == 0.0 and mp_rn(mp_exp(up)) == TINY
    # the tie 2^-1075 rounds to even (0); just above it rounds up
    mpmath = _mp()
    with mpmath.workprec(200):
        half = mpmath.mpf(2) ** -1075
        assert mp_rn(half) == 0.0 and mp_rn(half * (1 + mpmath.mpf(2) ** -100)) == TINY
        assert mp_rn(3 * half) == 2 * TINY                  # 1.5 ulp ties to the even 2 ulp
    s = exp_hp(np.array([np.nextafter(X_SUBNORMAL, -np.inf), X_SUBNORMAL]))    # X_SUBNORMAL lies above ln 2^-1022
    r = rn(s)
    assert r[0] < MIN_NORMAL <= r[1] and ulp(r[0]) == ulp(r[1]) == TINY
    one = exp_hp(np.array([0.0]))
    assert ulp_err(np.array([1.0]), one)[0] == 0.0
    assert ulp_err(np.array([np.nextafter(1.0, 2.0)]), one)[0] == 1.0
    e_up = exp_hp(np.array([up]))                           # 2^-1075 (1 + 1.1e-13)
    assert ulp_err(np.array([TINY]), e_up)[0] == pytest.approx(0.5, abs=1e-9)
    assert ulp_err(np.array([2 * TINY]), e_up)[0] == pytest.approx(1.5, abs=1e-9)
    assert ulp_err(np.array([0.0]), exp_hp(np.array([X_ZERO])))[0] < 0.5


def test_long_double_reference_matches_mpmath_at_edges():
    """The vectorised reference agrees with 40-digit mpmath on every named point: the same RN(exp x), and (long double)
    the value within 4e-3 ulp (a few units of the 64-bit significand): the reference's own error is far below the
    bounds it checks."""
    mpmath = _mp()
    x = np.concatenate([t for _, _, t in named_points().values()])
    e = exp_hp(x)
    r = rn(e)
    for xi, ei, ri in zip(x, e, r):
        m = mp_exp(xi)
        assert mp_rn(m) == ri, xi
        if LD:
            k = 1100 if ei < 1e-300 else 0                      # scaled clear of the double's subnormals, exactly
            sc = ei * np.longdouble(2) ** k
            hi = float(sc)
            with mpmath.workdps(40):
                exact = (mpmath.mpf(hi) + mpmath.mpf(float(sc - np.longdouble(hi)))) * mpmath.mpf(2) ** -k
                assert abs((exact - m) / float(ulp(ri))) < 4e-3, xi


def test_vectors_reach_the_bands():
    """The vectors the symmetric fills and the bit-equality test use put entries, for three components summed too, in
    the subnormal band, at RN = 0 next to a non-zero, and across [-750, 0]."""
    rng = np.random.default_rng(700 + 3)
    zs = [sym_vector(300, LS[c], rng) for c in range(3)]
    xs = [realised_x(z, z, l) for z, l in zip(zs, LS)]
    S = 0
    for x, a in zip(xs, AMPS):
        S = S + (a * a) * exp_hp(x)
    R = rn(np.asarray(S))
    assert np.count_nonzero((R > 0) & (R < MIN_NORMAL)) > 10
    x0 = xs[0]
    assert np.count_nonzero((x0 > X_ZERO) & (x0 < X_SUBNORMAL)) > 50 and np.count_nonzero((x0 < X_ZERO) & (x0 > -750)) > 5
    assert set(np.floor(x0[x0 > -750] / 50)) >= set(range(-15, 0))


def test_bounds_reject_the_known_regressions():
    """The checks fail on host copies of the regressions the issue names: a result 2 ulp off, flush-to-zero in the
    subnormal band, a relative error of 1e-14; and pass on RN(exp) itself."""
    x = np.concatenate([np.linspace(-745.0, -1.0, 4001), named_points()["zero_threshold"][2]])
    good = rn(exp_hp(x))
    check_single(good, x, "host", 1)
    two = good + 2 * ulp(good)
    with pytest.raises(AssertionError):
        check_single(two, x, "host", 1)
    ftz = np.where(x < -708.4, 0.0, good)
    with pytest.raises(AssertionError):
        check_single(ftz, x, "host", 1)
    with pytest.raises(AssertionError):
        check_full(good * (1 + 1e-14), [x], [1.0], "host")
    check_full(good, [x], [1.0], "host")
    for key in [k for k in STATS if k[0] == "host"]:
        STATS.pop(key)


# ---------------------------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _L():
    from psoap_b200 import _lib as L
    return L, L.load()


def dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def run_v12(rows, cols, amps, ls, ld=None):
    """fill_v12_kernel into an [M + 1, ld] buffer of SENTINEL: psoap_fill_v12 for one component, psoap_fill_v12n
    otherwise.  Checks that nothing outside [M, N] is written; returns the [M, N] entries."""
    torch = _torch()
    L, lib = _L()
    M, N, n = len(rows[0]), len(cols[0]), len(rows)
    ld = N if ld is None else ld
    buf = torch.full((M + 1, ld), SENTINEL, dtype=torch.float64, device="cuda")
    rd, cd = [dev(r) for r in rows], [dev(c) for c in cols]
    if n == 1:
        L.check(lib.psoap_fill_v12(L.ptr(buf), ld, M, N, L.ptr(rd[0]), L.ptr(cd[0]), float(amps[0]), float(ls[0]),
                                   L.stream_ptr()))
    else:
        rp = (L.vp * n)(*[v.data_ptr() for v in rd])
        cp = (L.vp * n)(*[v.data_ptr() for v in cd])
        L.check(lib.psoap_fill_v12n(n, L.ptr(buf), ld, M, N, ctypes.cast(rp, ctypes.POINTER(L.vp)),
                                    ctypes.cast(cp, ctypes.POINTER(L.vp)), L.dbl_array(amps), L.dbl_array(ls),
                                    L.stream_ptr()))
    out = buf.cpu().numpy()
    assert (out[:M, N:] == SENTINEL).all() and (out[M] == SENTINEL).all(), "fill_v12 wrote outside the matrix"
    return out[:M, :N]


def run_v11(zs, amps, ls, ld=None):
    """fill_full_kernel (psoap_fill_v11) into an [N + 1, ld] buffer of SENTINEL; returns the [N, N] matrix."""
    torch = _torch()
    L, lib = _L()
    N = len(zs[0])
    ld = N if ld is None else ld
    buf = torch.full((N + 1, ld), SENTINEL, dtype=torch.float64, device="cuda")
    zd = [dev(z) for z in zs]
    p = [L.ptr(z) for z in zd] + [L.vp(None)] * (3 - len(zd))
    L.check(lib.psoap_fill_v11(len(zd), L.ptr(buf), ld, N, p[0], p[1], p[2], L.dbl_array(amps), L.dbl_array(ls),
                               L.stream_ptr()))
    out = buf.cpu().numpy()
    assert (out[:N, N:] == SENTINEL).all() and (out[N] == SENTINEL).all(), "fill_v11 wrote outside the matrix"
    return out[:N, :N]


def run_lower(zs, sigma, amps, ls, fused=None):
    """fill_lower_kernel (psoap_debug_fill_lower): the [N, N] data block of the padded matrix, entry (i, j) for i >= j
    (the upper triangle as the buffer held it).  fused = (lwl, epoch, vel [ncomp, n_epochs]) takes the fused Doppler
    path; zs is then ignored."""
    torch = _torch()
    L, lib = _L()
    N, ncomp = len(sigma), len(amps)
    Np = envelope.padded_tiles(N) * envelope.NB
    pad = Np - N
    W = torch.full((Np, Np), SENTINEL, dtype=torch.float64, device="cuda")
    rvec = torch.full((Np,), SENTINEL, dtype=torch.float64, device="cuda")
    fl, sg = dev(np.ones(N)), dev(sigma)
    if fused is None:
        zd = [dev(z) for z in zs] + [None] * (3 - ncomp)
        ep = vd = None
        ne = 0
    else:
        lwl, epoch, vel = fused
        zd = [dev(lwl), None, None]
        ep = torch.from_numpy(np.ascontiguousarray(epoch, dtype=np.int32)).cuda()
        vd = dev(vel)
        ne = vel.shape[1]
    L.check(lib.psoap_debug_fill_lower(ncomp, N, L.ptr(zd[0]), L.ptr(zd[1]), L.ptr(zd[2]), L.ptr(ep), L.ptr(vd), ne,
                                       L.ptr(fl), L.ptr(sg), L.dbl_array(amps), L.dbl_array(ls), 1.0, L.ptr(W), Np,
                                       L.ptr(rvec), L.stream_ptr()))
    full = W.cpu().numpy().T                                        # [row, col]: the buffer is column-major
    return full[pad:, pad:], full


# ---------------------------------------------------------------------------------------------- GPU: fill_v12
AMPS = (1.0, 0.5, 0.75)
LS = (5.0, 7.0, 6.0)


def _onehot(ncomp, c):
    return [1.0 if k == c else 0.0 for k in range(ncomp)]


@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_fill_v12_named_points(ncomp):
    """Every named point through the row z = 0, in each component slot in turn (that component amp = 1, the others 0,
    so the entry is that component's exp_neg): 1.5 ulp, the exact zero set, x = -0 -> 1."""
    pts = named_points()
    L_all = np.concatenate([L for L, _, _ in pts.values()])
    R_all = np.concatenate([R for _, R, _ in pts.values()])
    calls = 0
    for live in range(ncomp):
        for l in np.unique(L_all):
            r = R_all[L_all == l]
            cols = np.concatenate([r, -r])
            ls = [LS[c] if c != live else l for c in range(ncomp)]
            got = run_v12([np.zeros(1)] * ncomp, [cols] * ncomp, _onehot(ncomp, live), ls)
            check_single(got, realised_x([0.0], cols, l), "fill_v12", ncomp, ("named", live, l))
            calls += 1
    got = run_v12([np.zeros(1)] * ncomp, [np.array([0.0, -0.0])] * ncomp, _onehot(ncomp, ncomp - 1), LS[:ncomp])
    assert np.array_equal(got, [[1.0, 1.0]])
    report("fill_v12")


@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_fill_v12_dense_sweep(ncomp):
    """One dense call of 2^24 entries (4097 x 4097) with the last component live at amp = 1: the uniform sweep through
    the z = 0 row and through the 8.5 rows, at 1.5 ulp with the exact zero set; then every component live
    (amps 1, 0.5, 0.75) within full_bound."""
    rng = np.random.default_rng(100 + ncomp)
    n = 4097
    vecs = [v12_vectors(n, n, LS[c], rng) for c in range(ncomp)]
    rows, cols = [v[0] for v in vecs], [v[1] for v in vecs]
    got = run_v12(rows, cols, _onehot(ncomp, ncomp - 1), LS[:ncomp])
    for i0 in range(0, n, 512):
        sl = slice(i0, min(n, i0 + 512))
        check_single(got[sl], realised_x(rows[-1][sl], cols[-1], LS[ncomp - 1]), "fill_v12", ncomp, ("dense", i0))
    m = 1025
    rows, cols = [r[:m] for r in rows], [c[:m] for c in cols]
    got = run_v12(rows, cols, AMPS[:ncomp], LS[:ncomp])
    check_matrix_full(got, rows, cols, AMPS[:ncomp], LS[:ncomp], "fill_v12", tag="all live")
    report("fill_v12")


@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_fill_v12_ragged_shapes(ncomp):
    """M, N in {1, 63, 64, 65, 4097} (not both 4097), ld = N + 3: full_bound inside, nothing written outside."""
    rng = np.random.default_rng(200 + ncomp)
    sizes = [1, 63, 64, 65, 4097]
    for M in sizes:
        for N in sizes:
            if M == N == 4097:
                continue
            vecs = [v12_vectors(M, N, LS[c], rng) for c in range(ncomp)]
            rows, cols = [v[0] for v in vecs], [v[1] for v in vecs]
            got = run_v12(rows, cols, AMPS[:ncomp], LS[:ncomp], ld=N + 3)
            check_matrix_full(got, rows, cols, AMPS[:ncomp], LS[:ncomp], "fill_v12", tag=(M, N))
    report("fill_v12")


@gpu
@pytest.mark.parametrize("ncomp", [1, 3])
def test_fill_v12_nan_column(ncomp):
    """A NaN column (in the last component) gives a NaN column and nothing else; an infinite column (in the first)
    gives x = -inf, an exact 0 term."""
    rng = np.random.default_rng(300 + ncomp)
    vecs = [v12_vectors(70, 130, LS[c], rng) for c in range(ncomp)]
    rows, cols = [v[0] for v in vecs], [v[1] for v in vecs]
    cols[ncomp - 1][5] = np.nan
    cols[0][66] = np.inf
    got = run_v12(rows, cols, AMPS[:ncomp], LS[:ncomp])
    assert np.isnan(got[:, 5]).all() and np.count_nonzero(np.isnan(got)) == got.shape[0]
    assert (realised_x(rows[0], cols[0], LS[0])[:, 66] == -np.inf).all()
    if ncomp == 1:
        assert (got[:, 66] == 0.0).all()
        check_single(got, realised_x(rows[0], cols[0], LS[0]), "fill_v12", 1, "nan")
    keep = np.ones(got.shape, dtype=bool)
    keep[:, 5] = False
    check_matrix_full(got, rows, cols, AMPS[:ncomp], LS[:ncomp], "fill_v12", mask=keep, tag="nan")


# ---------------------------------------------------------------------------------------------- GPU: fill_full
@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_fill_v11_bounds_and_symmetry(ncomp):
    """psoap_fill_v11 at N across the 64-row tiles, ld = N + 5: off-diagonal entries within full_bound (and at 1.5 ulp
    with the exact zero set when only the last component is live), the diagonal == sum amp2 bit for bit, mat == mat.T
    bit for bit, nothing written outside."""
    for N in (1, 2, 63, 64, 65, 127, 129, 1000):
        rng = np.random.default_rng(400 + 10 * N + ncomp)
        zs = [sym_vector(N, LS[c], rng) for c in range(ncomp)]
        off = ~np.eye(N, dtype=bool)
        got = run_v11(zs, AMPS[:ncomp], LS[:ncomp], ld=N + 5)
        assert np.array_equal(got, got.T), N
        d = AMPS[0] * AMPS[0]
        for a in AMPS[1:ncomp]:
            d = d + a * a
        assert (np.diag(got) == d).all(), N
        check_matrix_full(got, zs, zs, AMPS[:ncomp], LS[:ncomp], "fill_v11", mask=off, tag=N)
        got = run_v11(zs, _onehot(ncomp, ncomp - 1), LS[:ncomp], ld=N + 5)
        x = realised_x(zs[-1], zs[-1], LS[ncomp - 1])
        check_single(got[off], x[off], "fill_v11", ncomp, N)
        assert (np.diag(got) == 1.0).all()
    report("fill_v11")


# ---------------------------------------------------------------------------------------------- GPU: fill_lower
def lower_case(N, ncomp, seed):
    """Base ln-wavelengths, epochs and a velocity table for the fused path, and the host-shifted z per component."""
    rng = np.random.default_rng(seed)
    lwl = sym_vector(N, LS[0], rng)
    epoch = (np.arange(N) % 3).astype(np.int32)
    vel = np.array([[-12.3, 4.56, 27.1], [3.3, -40.2, 0.0], [-0.7, 15.5, -8.25]])[:ncomp]
    zs = [shifted(lwl, vel[c], epoch) for c in range(ncomp)]
    sigma = rng.integers(1, 4, N).astype(np.float64) * 0.125
    return lwl, epoch, vel, zs, sigma


@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
@pytest.mark.parametrize("N", [1000, 1024])
def test_fill_lower_bounds_and_fused_shift(N, ncomp):
    """psoap_debug_fill_lower with front padding (N = 1000) and without (N = 1024): the fused Doppler path writes the
    same bits as the pre-shifted path fed with the host-shifted z; the strict lower triangle within full_bound of the
    exact sum at the host-shifted z; the diagonal == sum amp2 + sigma^2 bit for bit."""
    lwl, epoch, vel, zs, sigma = lower_case(N, ncomp, 500 + N + ncomp)
    amps, ls = AMPS[:ncomp], LS[:ncomp]
    pre, pre_all = run_lower(zs, sigma, amps, ls)
    fus, fus_all = run_lower(None, sigma, amps, ls, fused=(lwl, epoch, vel))
    assert np.array_equal(pre_all, fus_all)
    low = np.tril(np.ones((N, N), dtype=bool), -1)
    check_matrix_full(pre, zs, zs, amps, ls, "fill_lower", mask=low, tag=N)
    d = amps[0] * amps[0]
    for a in amps[1:]:
        d = d + a * a
    assert np.array_equal(np.diag(pre), d + sigma * sigma)
    pre1, _ = run_lower(zs, sigma, _onehot(ncomp, ncomp - 1), ls)
    x = realised_x(zs[-1], zs[-1], ls[-1])
    check_single(pre1[low], x[low], "fill_lower", ncomp, N)
    report("fill_lower")


# ---------------------------------------------------------------------------------------------- GPU: predict border
def far_data(n, ncomp):
    """Data pixels in clusters of 5 identical z near 9.5 (the data block is positive definite with integer sigma), every
    one of them > 0.9 from every grid point near 0 or 8.5: each data-grid argument is below -1e9, C is exactly 0."""
    z = 9.5 + 1e-2 * (np.arange(n) // 5)
    rng = np.random.default_rng(n)
    return [z] * ncomp, 1.0 + rng.integers(-32, 33, n) / 64.0, rng.integers(1, 4, n).astype(np.float64)


def run_predict(mode, grids, amps, ls, nugget=0.0, n=70):
    """psoap_predict on far data: (Sigma [M, M], delta [M]) as numpy."""
    from psoap_b200 import covariance
    ncomp = len(grids)
    zd, fl, sg = far_data(n, ncomp)
    Sigma, delta = covariance._predict_device(mode, [dev(z) for z in zd], dev(fl), dev(sg), [dev(g) for g in grids],
                                              list(amps), list(ls), 1.0, nugget)
    return Sigma.cpu().numpy(), delta.cpu().numpy()


@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_predict_border_is_sigma(ncomp):
    """With C exactly 0, Sigma = A bit for bit.  Mode 0: blockdiag(K_c(grid_c)), off-component blocks exactly 0, each
    block within full_bound (one component) with the diagonal == amp_c^2.  Mode 1: sum_c K_c within full_bound, the
    diagonal == sum amp2 + nugget bit for bit.  delta is exactly 0 in both."""
    m = 150                                     # mode 0: M = ncomp m crosses 128-row tiles
    rng = np.random.default_rng(600 + ncomp)
    grids = [sym_vector(m, LS[c], rng) for c in range(ncomp)]
    amps, ls = AMPS[:ncomp], LS[:ncomp]
    S0, d0 = run_predict(0, grids, amps, ls)
    assert not d0.any()
    off = ~np.eye(m, dtype=bool)
    for a in range(ncomp):
        for b in range(ncomp):
            blk = S0[a * m:(a + 1) * m, b * m:(b + 1) * m]
            if a != b:
                assert not blk.any(), (a, b)
                continue
            assert (np.diag(blk) == amps[a] * amps[a]).all()
            check_matrix_full(blk, [grids[a]], [grids[a]], [amps[a]], [ls[a]], "predict_border", mask=off, tag=a)
    nugget = 1e-8
    S1, d1 = run_predict(1, grids, amps, ls, nugget=nugget)
    assert not d1.any()
    d = amps[0] * amps[0]
    for x in amps[1:]:
        d = d + x * x
    assert (np.diag(S1) == d + nugget).all()
    check_matrix_full(S1, grids, grids, amps, ls, "predict_border", mask=off, tag="mode 1")
    S1, _ = run_predict(1, grids, _onehot(ncomp, ncomp - 1), ls)
    x = realised_x(grids[-1], grids[-1], ls[-1])
    check_single(S1[off], x[off], "predict_border", ncomp)
    report("predict_border")


# ---------------------------------------------------------------------------------------------- GPU: cross-kernel bits
@gpu
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_kernels_agree_bit_for_bit(ncomp):
    """The same (z, amp, l) through every kernel that writes an entry: fill_v11's matrix == fill_v12n(rows = z,
    cols = z) everywhere == predict mode 1 (no nugget) == fill_lower's strict lower triangle; predict mode 0's block c
    == fill_v11 of component c alone == fill_v12 of component c alone.  Pre-shifted z at N = 300 (front padding 84)."""
    N = 300
    rng = np.random.default_rng(700 + ncomp)
    zs = [sym_vector(N, LS[c], rng) for c in range(ncomp)]
    amps, ls = AMPS[:ncomp], LS[:ncomp]
    v11 = run_v11(zs, amps, ls)
    v12 = run_v12(zs, zs, amps, ls)
    assert np.array_equal(v12, v11)
    low = np.tril(np.ones((N, N), dtype=bool), -1)
    lower, _ = run_lower(zs, np.ones(N), amps, ls)
    assert np.array_equal(lower[low], v11[low])
    S1, _ = run_predict(1, zs, amps, ls)
    assert np.array_equal(S1, v11)
    S0, _ = run_predict(0, zs, amps, ls)
    for c in range(ncomp):
        one = run_v11([zs[c]], [amps[c]], [ls[c]])
        assert np.array_equal(S0[c * N:(c + 1) * N, c * N:(c + 1) * N], one), c
        assert np.array_equal(run_v12([zs[c]], [zs[c]], [amps[c]], [ls[c]]), one), c


# ---------------------------------------------------------------------------------------------- GPU: farm border fill
FARM_ORBITS = {"SB2": [0.2, 0.0, 0.2, 10.0, 10.0, 0.0, 0.0],
               "ST3": [0.4, 0.0, 0.2, 10.0, 10.0, 0.0, 0.2, 0.0, 0.2, 80.0, 100.0, 3.0, 0.0]}


@gpu
@pytest.mark.parametrize("model", ["SB2", "ST3"])
def test_farm_predict_border_is_sigma(model):
    """predict_border_farm_kernel through ChunkFarm.predict_components with zero orbital velocities (K = 0, gamma = 0:
    the shifted z are the pixels' own bits) and pixels far from every grid point: each item's Sigma is
    blockdiag(K_c(grid_c)) bit for bit, == psoap_fill_v11 of component c alone, within full_bound, the off-component
    blocks exactly 0, and mu == the component means exactly."""
    from psoap_b200.farm import ChunkFarm
    ncomp = {"SB2": 2, "ST3": 3}[model]
    rng = np.random.default_rng(800 + ncomp)
    chunks, grids, ms = [], [], (90, 140)
    for i, m in enumerate(ms):
        n = 60 + 50 * i
        zd, fl, sg = far_data(n, 1)
        chunks.append(dict(lwl=zd[0], fl=fl, sigma=sg, epoch=(np.arange(n) % 3).astype(np.int32),
                           date1D=np.array([0.5, 1.5, 2.5])))
        grids.append(np.stack([sym_vector(m, LS[c], rng) for c in range(ncomp)]))
    K = 2
    gps = [[(AMPS[c], LS[c]) for c in range(ncomp)], [(AMPS[(c + 1) % 3] * 0.5, LS[(c + 2) % 3]) for c in range(ncomp)]]
    P = np.array([FARM_ORBITS[model] + [v for a_l in gp for v in a_l] for gp in gps])
    mus = np.linspace(0.4, 0.6, ncomp)
    farm = ChunkFarm(model, chunks, n_proposals=K)
    farm.attach_prediction_grids(grids, predict_nbranch=2)
    out = farm.predict_components(P, mus)
    for i, m in enumerate(ms):
        mu, Sig = out[i][0].cpu().numpy(), out[i][1].cpu().numpy()
        for k in range(K):
            assert np.array_equal(mu[k], np.repeat(mus, m)), (i, k)
            off = ~np.eye(m, dtype=bool)
            for a in range(ncomp):
                for b in range(ncomp):
                    blk = Sig[k, a * m:(a + 1) * m, b * m:(b + 1) * m]
                    if a != b:
                        assert not blk.any(), (i, k, a, b)
                        continue
                    amp, l = gps[k][a]
                    assert np.array_equal(blk, run_v11([grids[i][a]], [amp], [l])), (i, k, a)
                    check_matrix_full(blk, [grids[i][a]], [grids[i][a]], [amp], [l], "predict_border_farm",
                                      mask=off, tag=(i, k, a))
    farm.close()
    report("predict_border_farm")


# ---------------------------------------------------------------------------------------------- GPU: exact-zero threshold
def threshold_case(x_target, amp, N=512, a=5, b=300):
    """N = 512 pixels (4 row blocks, no front padding, so the likelihood's tiles and the Fisher's data-order tiles
    coincide) in clusters of 32 identical z inside row blocks, cluster centres 1e-2 apart (x <= -1.6e5 between clusters).
    Pixel a (block 0) and pixel b (block 2) are clusters of their own, b placed so that its pair with a has the
    realised x closest to x_target: tile (2, 0) holds that one pair and nothing else above -1.6e5."""
    from test_envelope_patterns import DZ, MU, Z0
    labels = np.arange(N) // 32
    labels[a], labels[b] = labels.max() + 1, labels.max() + 2
    z = Z0 + DZ * labels
    r = np.sqrt(x_target / p2_of(L0))
    z[b] = z[a] + r
    x = realised_x([z[a]], [z[b]], L0)[0, 0]
    assert abs(x - x_target) < 1e-6
    rng = np.random.default_rng(int(-x_target * 10) + int(amp * 8))
    fl = MU + rng.integers(-32, 33, N) / 64.0
    sigma = rng.integers(1, 4, N).astype(np.float64)
    # the correctly rounded K entry of the pair, from 40-digit mpmath (== the long-double reference)
    k_rn = mp_rn((amp * amp) * mp_exp(x))
    e_rn = mp_rn(mp_exp(x))
    if LD:
        assert k_rn == float(np.longdouble(amp * amp) * exp_hp(np.array([x]))[0]) and e_rn == rn(exp_hp(np.array([x])))[0]
    T = N // envelope.NB
    flags = np.eye(T, dtype=bool)
    if k_rn != 0.0:
        flags[b // envelope.NB, a // envelope.NB] = True
    case = dict(N=N, labels=[labels], zs=[z], fl=fl, sigma=sigma, amps=[amp], ls=[L0], A=amp * amp)
    return case, x, k_rn, e_rn, flags


THRESHOLD_CASES = {"x=-744.4 amp=1": (-744.4, 1.0, True, True),
                   "x=-745.9 amp=1": (-745.9, 1.0, False, False),
                   "x=-744.4 amp=0.5": (-744.4, 0.5, False, True)}


@gpu
@pytest.mark.parametrize("name", sorted(THRESHOLD_CASES))
def test_exact_zero_threshold_end_to_end(name):
    """One pair near the zero threshold decides tile (2, 0).  The likelihood's envelope (psoap_lnlike_envelope_view)
    == tend_by_end of the flags of the correctly rounded K; the Fisher's flags (psoap_chunk_fisher_views, one SB1
    orbit with K = 0 and gamma = 0) mark the tile exactly when RN(exp x) != 0, with amp = 0.5 too, where the K entry
    rounds to 0 and the likelihood's tile is empty: the Fisher flags mark non-zero exponentials, not entries.  The
    lnlike against the closed form of test_envelope_patterns (the pair's entry, at most 2^-1074, is below its
    resolution)."""
    from test_envelope_patterns import MU, check_against_closed_form, device_lnlike
    from test_fisher import chunk_fisher
    x_target, amp, k_nonzero, e_nonzero = THRESHOLD_CASES[name]
    case, x, k_rn, e_rn, flags = threshold_case(x_target, amp)
    assert (k_rn != 0.0) == k_nonzero and (e_rn != 0.0) == e_nonzero, (x, k_rn, e_rn)
    tend, res = device_lnlike(case)
    want = envelope.tend_by_end(np.tril(flags))
    assert np.array_equal(tend, want), (name, tend, want)
    T = flags.shape[0]
    assert tend[1] == (3 if k_nonzero else 1)                            # the tile keeps row block 2 in panel 1's updates
    check_against_closed_form(case, res, name)
    ch = dict(lwl=case["zs"][0], fl=case["fl"], sigma=case["sigma"], date1D=np.array([0.5, 1.5, 2.5]),
              epoch=(np.arange(case["N"]) % 3).astype(np.int32))
    p = np.array([0.0, 0.2, 10.0, 10.0, 0.0, 0.0, amp, L0])
    (fres, _, F), fflags, krange = chunk_fisher("SB1", ch, p, mu=MU, views=True)
    assert fres[3] == 0.0 and np.isfinite(F).all()
    want_f = np.eye(T, dtype=bool)
    if e_nonzero:
        want_f[2, 0] = want_f[0, 2] = True
    assert np.array_equal(fflags.astype(bool), want_f), (name, fflags)
    want_k = np.array([[J, J] for J in range(T)])
    if e_nonzero:
        want_k[0] = want_k[2] = (0, 2)
    assert np.array_equal(krange, want_k), (name, krange)
