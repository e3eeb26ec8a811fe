"""Drop-in for the likelihood / prediction part of psoap.covariance (psoap/covariance.py:25-379).

Same names, positional/keyword signatures, defaults and return types as the reference.  Vectors may be numpy
float64 arrays (uploaded: O(N) bytes) or float64 CUDA tensors (used in place).  `V11` stays in the `lnlike_*`
signatures for compatibility; it is scratch the caller never reads (sample_parallel.py:161-163), so it is not
filled unless `MATERIALIZE_V11` is set (debug: reproduces the side effect K + sigma^2 I at N^2 PCIe cost).

Everything runs in the CUDA library (csrc/): fill + blocked FP64 Cholesky with the solve, log-determinant and
quadratic form fused in.  predict_* build the bordered matrix [[K + s^2 I, C^T], [C, A]] on the device and take
its Schur complement with the same factorisation kernels (A - C K^-1 C^T, and mu from the carried residual).
"""
import collections
import ctypes

import numpy as np

from . import _lib
from . import matrix_functions

MATERIALIZE_V11 = False
NB = 128


def _pad(n):
    return (n + NB - 1) // NB * NB


# --------------------------------------------------------------------------------------------------
# lnlike_* (covariance.py:299-379)
# --------------------------------------------------------------------------------------------------
def _lnlike(V11, lwls, fl, sigma, amps, ls, mu_GP):
    lib = _lib.load()
    torch = _lib.torch_cuda()
    if any(a < 0.0 for a in amps) or any(l < 0.0 for l in ls):  # covariance.py:317-318,:339-340,:362-363
        return -np.inf
    vecs = [_lib.dev_f64(v) for v in lwls]
    fl_d, sg_d = _lib.dev_f64(fl), _lib.dev_f64(sigma)
    N = fl_d.numel()
    for v in vecs + [sg_d]:
        if v.dim() != 1 or v.numel() != N:
            raise ValueError("wavelength, flux and sigma vectors must be 1-D with the same length")
    if N == 0:  # the reference's sums run over nothing: -0.5 * (0 + 0)
        return -0.0
    nbytes = lib.psoap_lnlike_workspace_bytes(N)
    ws = _lib.workspace(nbytes + 256, "lnlike")
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    ptrs = [_lib.ptr(v) for v in vecs] + [_lib.vp(None)] * (3 - len(vecs))
    _lib.check(lib.psoap_lnlike(len(vecs), N, ptrs[0], ptrs[1], ptrs[2], _lib.ptr(fl_d), _lib.ptr(sg_d),
                                _lib.dbl_array(amps), _lib.dbl_array(ls), float(mu_GP), _lib.ptr(ws), nbytes,
                                _lib.ptr(res), _lib.stream_ptr()))
    if MATERIALIZE_V11 and V11 is not None:
        matrix_functions._fill_v11(V11, lwls, amps, ls)
        if isinstance(V11, np.ndarray):
            V11[np.diag_indices_from(V11)] += np.asarray(sigma) ** 2
        else:
            V11.diagonal().add_(sg_d ** 2)
    return float(res[0].item())


def lnlike_f(V11, wl_f, fl, sigma, amp_f, l_f, mu_GP=1.):
    """covariance.py:299-331"""
    return _lnlike(V11, [wl_f], fl, sigma, [amp_f], [l_f], mu_GP)


def lnlike_f_g(V11, wl_f, wl_g, fl, sigma, amp_f, l_f, amp_g, l_g, mu_GP=1.):
    """covariance.py:333-354"""
    return _lnlike(V11, [wl_f, wl_g], fl, sigma, [amp_f, amp_g], [l_f, l_g], mu_GP)


def lnlike_f_g_h(V11, wl_f, wl_g, wl_h, fl, sigma, amp_f, l_f, amp_g, l_g, amp_h, l_h, mu_GP=1.):
    """covariance.py:356-376"""
    return _lnlike(V11, [wl_f, wl_g, wl_h], fl, sigma, [amp_f, amp_g, amp_h], [l_f, l_g, l_h], mu_GP)


# covariance.py:379
lnlike = {"SB1": lnlike_f, "SB2": lnlike_f_g, "ST1": lnlike_f, "ST2": lnlike_f_g, "ST3": lnlike_f_g_h}


def lnlike_host(lwls, fl, sigma, amps, ls, mu_GP=1.):
    """The C ABI's host-buffer entry (psoap_lnlike_host): numpy in, float out, no torch involved."""
    lib = _lib.load()
    vecs = [np.ascontiguousarray(v, dtype=np.float64) for v in lwls]
    fl, sigma = np.ascontiguousarray(fl, dtype=np.float64), np.ascontiguousarray(sigma, dtype=np.float64)
    p = [v.ctypes.data_as(_lib.c_double_p) for v in vecs] + [None] * (3 - len(vecs))
    res = _lib.PsoapResult()
    _lib.check(lib.psoap_lnlike_host(len(vecs), len(fl), p[0], p[1], p[2], fl.ctypes.data_as(_lib.c_double_p),
                                     sigma.ctypes.data_as(_lib.c_double_p), _lib.dbl_array(amps), _lib.dbl_array(ls),
                                     float(mu_GP), ctypes.byref(res)))
    return res.lnlike


LnlikeGrad = collections.namedtuple("LnlikeGrad", ["lnlike", "amp", "l", "mu_GP", "lwl"])


def lnlike_grad(lwls, fl, sigma, amps, ls, mu_GP=1.0):
    """The log-likelihood of `_lnlike` and its exact gradient (psoap_lnlike_grad): returns
    LnlikeGrad(lnlike, amp [ncomp], l [ncomp], mu_GP, lwl [ncomp, N]) with d lnlike / d(amp_c, l_c, mu_GP) as numpy
    arrays / float and d lnlike / d lwls[c][i] as numpy or CUDA tensor like `fl`.  Inputs as in lnlike_f / _f_g / _f_g_h.
    When lnlike is -inf (negative hyper-parameters, K not positive definite) every gradient entry is NaN."""
    lib = _lib.load()
    torch = _lib.torch_cuda()
    on_dev = _is_dev(fl)
    vecs = [_lib.dev_f64(v) for v in lwls]
    fl_d, sg_d = _lib.dev_f64(fl), _lib.dev_f64(sigma)
    ncomp, N = len(vecs), fl_d.numel()
    if not 1 <= ncomp <= 3 or len(amps) != ncomp or len(ls) != ncomp:
        raise ValueError("lnlike_grad takes 1 to 3 components, one amp and one l each")
    for v in vecs + [sg_d]:
        if v.dim() != 1 or v.numel() != N:
            raise ValueError("wavelength, flux and sigma vectors must be 1-D with the same length")
    nbytes = lib.psoap_lnlike_grad_workspace_bytes(ncomp, N)
    ws = _lib.workspace(nbytes + 256, "lnlike_grad")
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    g_hyp = torch.empty(2 * ncomp + 1, dtype=torch.float64, device="cuda")
    g_lwl = torch.empty((ncomp, N), dtype=torch.float64, device="cuda")
    ptrs = [_lib.ptr(v) for v in vecs] + [_lib.vp(None)] * (3 - ncomp)
    _lib.check(lib.psoap_lnlike_grad(ncomp, N, ptrs[0], ptrs[1], ptrs[2], _lib.ptr(fl_d), _lib.ptr(sg_d),
                                     _lib.dbl_array(amps), _lib.dbl_array(ls), float(mu_GP), _lib.ptr(ws), nbytes,
                                     _lib.ptr(res), _lib.ptr(g_hyp), _lib.ptr(g_lwl) if N else _lib.vp(None),
                                     _lib.stream_ptr()))
    h = g_hyp.cpu().numpy()
    if N == 0:
        g_lwl.zero_()
    return LnlikeGrad(float(res[0].item()), h[0:2 * ncomp:2].copy(), h[1:2 * ncomp:2].copy(), float(h[-1]),
                      _out(g_lwl, on_dev))


# --------------------------------------------------------------------------------------------------
# Schur-complement machinery for predict_*
# --------------------------------------------------------------------------------------------------
class _Bordered:
    """Column-major bordered matrix S [Nt, Nt] on the device, held as the row-major tensor St with
    S(i, j) = St[j, i].  Physical layout: [0, pad) identity, [pad, Nn) data block, [Nn, Nn + m) border."""

    def __init__(self, n, m):
        torch = _lib.torch_cuda()
        self.n, self.m = n, m
        self.Nn, self.Nt = _pad(n), _pad(n) + _pad(m)
        self.pad = self.Nn - n
        self.St = torch.zeros((self.Nt, self.Nt), dtype=torch.float64, device="cuda")
        if self.pad:
            self.St.diagonal()[:self.pad] = 1.0
        # dead padding rows of the border get a unit diagonal so nothing degenerate is ever touched
        if self.Nn + m < self.Nt:
            self.St.diagonal()[self.Nn + m:] = 1.0

    def data_block(self):
        return self.St[self.pad:self.Nn, self.pad:self.Nn]

    def cross_block(self, a0, a1):
        """St rows = data pixels, cols = border entries a0..a1  (S(border a, data j) = St[pad + j, Nn + a])."""
        return self.St[self.pad:self.Nn, self.Nn + a0:self.Nn + a1]

    def border_block(self, a0, a1):
        return self.St[self.Nn + a0:self.Nn + a1, self.Nn + a0:self.Nn + a1]

    def schur(self, resid):
        """Eliminate the data block.  resid: [n] device vector (fl - mu).  Returns (Sigma [m, m], delta [m])
        with delta = C K^-1 resid; raises LinAlgError like cho_factor (covariance.py:113 has no try)."""
        lib = _lib.load()
        torch = _lib.torch_cuda()
        nbytes = lib.psoap_schur_workspace_bytes(self.n, self.m)
        ws = _lib.workspace(nbytes + 256, "schur")
        rv, acc, info = _lib.vp(), _lib.vp(), _lib.vp()
        _lib.check(lib.psoap_schur_views(_lib.ptr(ws), self.n, self.m, ctypes.byref(rv), ctypes.byref(acc),
                                         ctypes.byref(info)))
        base = ws.data_ptr()
        r_view = ws[rv.value - base: rv.value - base + self.Nt * 8].view(torch.float64)
        acc_view = ws[acc.value - base: acc.value - base + 64].view(torch.float64)
        info_view = ws[info.value - base: info.value - base + 8].view(torch.int32)
        r_view.zero_()
        r_view[self.pad:self.Nn] = resid
        acc_view.zero_()
        info_view.zero_()
        res = torch.empty(4, dtype=torch.float64, device="cuda")
        _lib.check(lib.psoap_schur(_lib.ptr(self.St), self.Nt, self.n, self.m, _lib.ptr(ws), nbytes, _lib.ptr(res),
                                   _lib.stream_ptr()))
        if float(res[3].item()) != 0.0:
            raise np.linalg.LinAlgError("%d-th leading minor of the array is not positive definite" % int(res[3].item()))
        U = self.St[self.Nn:self.Nn + self.m, self.Nn:self.Nn + self.m]  # upper triangle of St = lower of S
        Sigma = torch.triu(U) + torch.triu(U, 1).T
        delta = -r_view[self.Nn:self.Nn + self.m].clone()
        return Sigma, delta


def _is_dev(x):
    torch = _lib.torch_cuda()
    return isinstance(x, torch.Tensor) and x.is_cuda


def _out(t, on_dev):
    return t if on_dev else t.cpu().numpy()


def _predict_device(mode, lwls, fl_d, sg_d, lwls_predict, amps, ls, resid_mu, nugget=0.0, get_Sigma=True):
    """One psoap_predict call (include/psoap_b200.h): returns (Sigma [M, M] or None, delta [M]) on the device;
    raises LinAlgError when the data block is not positive definite, like cho_factor (covariance.py:113 has no try)."""
    lib = _lib.load()
    torch = _lib.torch_cuda()
    ncomp, n, m = len(lwls), fl_d.numel(), lwls_predict[0].numel()
    M = ncomp * m if mode == 0 else m
    nbytes = lib.psoap_predict_workspace_bytes(ncomp, mode, n, m)
    if nbytes == 0:
        raise ValueError("psoap_predict: unsupported sizes (ncomp=%d mode=%d n=%d m=%d)" % (ncomp, mode, n, m))
    ws = _lib.workspace(nbytes + 256, "predict")
    delta = torch.empty(M, dtype=torch.float64, device="cuda")
    Sigma = torch.empty((M, M), dtype=torch.float64, device="cuda") if get_Sigma else None
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    dptr = (_lib.vp * ncomp)(*[_lib.vp(v.data_ptr()) for v in lwls])
    pptr = (_lib.vp * ncomp)(*[_lib.vp(v.data_ptr()) for v in lwls_predict])
    _lib.check(lib.psoap_predict(ncomp, mode, n, m, dptr, _lib.ptr(fl_d), _lib.ptr(sg_d), pptr, _lib.dbl_array(amps),
                                 _lib.dbl_array(ls), float(resid_mu), float(nugget), _lib.ptr(delta), _lib.ptr(Sigma),
                                 _lib.ptr(ws), nbytes, _lib.ptr(res), _lib.stream_ptr()))
    info = float(res[3].item())
    if info != 0.0:
        raise np.linalg.LinAlgError("%d-th leading minor of the array is not positive definite" % int(info))
    return Sigma, delta


def _fill_data_block(B, lwls, amps, ls, sigma_d):
    matrix_functions._fill_v11(B.data_block(), lwls, amps, ls)
    B.data_block().diagonal().add_(sigma_d * sigma_d)  # covariance.py:110 (sigma**2 on the diagonal)


def _predict_components(lwls, fl, sigma, lwls_predict, mus, amps, ls, get_Sigma=True):
    """predict_f_g (covariance.py:81-148) / predict_f_g_h (:190-251): joint prediction of the components."""
    torch = _lib.torch_cuda()
    on_dev = _is_dev(fl)
    ncomp = len(lwls)
    lw = [_lib.dev_f64(v) for v in lwls]
    lp = [_lib.dev_f64(v) for v in lwls_predict]
    fl_d, sg_d = _lib.dev_f64(fl), _lib.dev_f64(sigma)
    mp = lp[0].numel()
    # A = blockdiag(K_c(predict_c)); C = [K_c(predict_c, data_c)]  (covariance.py:117-136); the hard-coded 1.0 of
    # covariance.py:140,:248 is the residual mean
    Sigma, delta = _predict_device(0, lw, fl_d, sg_d, lp, amps, ls, 1.0, 0.0, get_Sigma)
    mu_cat = torch.cat([torch.full((mp,), float(m), dtype=torch.float64, device="cuda") for m in mus])
    mu = mu_cat + delta
    if get_Sigma:
        return _out(mu, on_dev), _out(Sigma, on_dev)
    return _out(mu, on_dev)


def predict_f_g(lwl_f, lwl_g, fl_fg, sigma_fg, lwl_f_predict, lwl_g_predict, mu_f, amp_f, l_f, mu_g, amp_g, l_g,
                get_Sigma=True):
    """covariance.py:81-148"""
    assert len(lwl_f) == len(lwl_g), "Input wavelengths must be the same length."
    assert len(lwl_f_predict) == len(lwl_g_predict), "Prediction wavelengths must be the same length."
    return _predict_components([lwl_f, lwl_g], fl_fg, sigma_fg, [lwl_f_predict, lwl_g_predict], [mu_f, mu_g],
                               [amp_f, amp_g], [l_f, l_g], get_Sigma)


def predict_f_g_h(lwl_f, lwl_g, lwl_h, fl_fgh, sigma_fgh, lwl_f_predict, lwl_g_predict, lwl_h_predict, mu_f, mu_g,
                  mu_h, amp_f, l_f, amp_g, l_g, amp_h, l_h):
    """covariance.py:190-251"""
    assert len(lwl_f) == len(lwl_g), "Input wavelengths must be the same length."
    assert len(lwl_f) == len(lwl_h), "Input wavelengths must be the same length."
    assert len(lwl_f_predict) == len(lwl_g_predict), "Prediction wavelengths must be the same length."
    assert len(lwl_f_predict) == len(lwl_h_predict), "Prediction wavelengths must be the same length."
    return _predict_components([lwl_f, lwl_g, lwl_h], fl_fgh, sigma_fgh,
                               [lwl_f_predict, lwl_g_predict, lwl_h_predict], [mu_f, mu_g, mu_h],
                               [amp_f, amp_g, amp_h], [l_f, l_g, l_h], True)


def _predict_sum(lwls, fl, sigma, lwls_predict, amps, ls, nugget, resid_mu, transpose_mean):
    torch = _lib.torch_cuda()
    on_dev = _is_dev(fl)
    lw = [_lib.dev_f64(v) for v in lwls]
    lp = [_lib.dev_f64(v) for v in lwls_predict]
    fl_d, sg_d = _lib.dev_f64(fl), _lib.dev_f64(sigma)
    n, mp = fl_d.numel(), lp[0].numel()

    def run(transposed, want_Sigma=True):
        # V11 = sum_c K_c(predict_c) (+ nugget, covariance.py:165); border = V12, or V12^T for the quirk of :294
        return _predict_device(2 if transposed else 1, lw, fl_d, sg_d, lp, amps, ls, resid_mu, nugget, want_Sigma)

    Sigma, delta = run(False)
    if transpose_mean:
        # covariance.py:294 multiplies by V12.T, which only has the right shape when M == N
        if mp != n:
            raise ValueError("shapes (%d,%d) and (%d,) not aligned: predict_f_g_h_sum needs M == N "
                             "(covariance.py:294 uses V12.T)" % (n, mp, n))
        _, delta = run(True, False)
    return Sigma, delta, on_dev


def predict_f_g_sum(lwl_f, lwl_g, fl_fg, sigma_fg, lwl_f_predict, lwl_g_predict, mu_fg, amp_f, l_f, amp_g, l_g):
    """covariance.py:151-187 (nugget 1e-8 on V11, mean from fl - 1.0)"""
    assert len(lwl_f) == len(lwl_g), "Input wavelengths must be the same length."
    Sigma, delta, on_dev = _predict_sum([lwl_f, lwl_g], fl_fg, sigma_fg, [lwl_f_predict, lwl_g_predict],
                                        [amp_f, amp_g], [l_f, l_g], 1e-8, 1.0, False)
    return _out(mu_fg + delta, on_dev), _out(Sigma, on_dev)


def predict_f_g_h_sum(lwl_f, lwl_g, lwl_h, fl_fgh, sigma_fgh, lwl_f_predict, lwl_g_predict, lwl_h_predict, mu_fgh,
                      amp_f, l_f, amp_g, l_g, amp_h, l_h):
    """covariance.py:253-297 (no nugget; mean from fl - mu_fgh through V12.T, reference quirk kept)"""
    assert len(lwl_f) == len(lwl_g), "Input wavelengths must be the same length."
    Sigma, delta, on_dev = _predict_sum([lwl_f, lwl_g, lwl_h], fl_fgh, sigma_fgh,
                                        [lwl_f_predict, lwl_g_predict, lwl_h_predict], [amp_f, amp_g, amp_h],
                                        [l_f, l_g, l_h], 0.0, float(mu_fgh), True)
    return _out(mu_fgh + delta, on_dev), _out(Sigma, on_dev)


def predict_f(lwl_known, fl_known, sigma_known, lwl_predict, amp_f, l_f, mu_GP=1.0):
    """covariance.py:25-54.  The reference body raises NameError (`wl_predict`, :38); this implements the evident
    intent: mu = mu_GP + V12^T V11^-1 (fl - mu_GP), Sigma = V22 - V12^T V11^-1 V12."""
    on_dev = _is_dev(fl_known)
    lw, lp = _lib.dev_f64(lwl_known), _lib.dev_f64(lwl_predict)
    fl_d, sg_d = _lib.dev_f64(fl_known), _lib.dev_f64(sigma_known)
    Sigma, delta = _predict_device(0, [lw], fl_d, sg_d, [lp], [amp_f], [l_f], float(mu_GP))
    return _out(mu_GP + delta, on_dev), _out(Sigma, on_dev)


# --------------------------------------------------------------------------------------------------
# Callers of the hot path that live in psoap.covariance: GP hyper-parameter fit and flux calibration
# (covariance.py:408-424, :560-732).  Host logic as in the reference (scipy Nelder-Mead, numpy Chebyshev);
# every O(N^3) piece goes through the same device kernels (lnlike_f, Schur complements).
# --------------------------------------------------------------------------------------------------
def optimize_GP_f(wl_known, fl_known, sigma_known, amp_f, l_f, mu_GP=1.0):
    """covariance.py:408-424: Nelder-Mead on -lnlike_f, starting from (amp_f, l_f)."""
    from scipy.optimize import minimize
    lw, fl, sg = _lib.dev_f64(wl_known), _lib.dev_f64(fl_known), _lib.dev_f64(sigma_known)  # uploaded once

    def func(x):
        a, l = x
        return -lnlike_f(None, lw, fl, sg, a, l, mu_GP)

    return minimize(func, np.array([amp_f, l_f]), method="Nelder-Mead")["x"]


def _chebyshev_design(x0, x1, x, fl_cal, order):
    """D = fl_cal[:, None] * T^T with T_k the Chebyshev polynomials on [x0, x1] (covariance.py:584-593)."""
    from numpy.polynomial import Chebyshev as Ch
    x = np.asarray(x, dtype=np.float64)
    T = np.array([Ch([0] * k + [1], domain=[x0, x1])(x) for k in range(order + 1)])
    return np.asarray(fl_cal, dtype=np.float64)[:, np.newaxis] * T.T


def _calibrate(fill_blocks, n_cal, n_fixed, resid_fixed, D, mu_GP):
    """Common core of optimize_calibration / optimize_calibration_static (covariance.py:598-624, :686-711):
    fl' = mu + C B^-1 (fl_fixed - mu), C' = A - C B^-1 C^T (first Schur complement); then the least squares
    X = (D^T C'^-1 D)^-1 D^T C'^-1 fl' through a second Schur complement with border D^T."""
    from scipy.linalg import cho_factor, cho_solve
    torch = _lib.torch_cuda()
    B1 = _Bordered(n_fixed, n_cal)
    fill_blocks(B1)
    C_prime, delta = B1.schur(resid_fixed)
    fl_prime = delta + float(mu_GP)
    k = D.shape[1]
    B2 = _Bordered(n_cal, k)
    B2.data_block().copy_(C_prime)
    B2.cross_block(0, k).copy_(torch.from_numpy(np.ascontiguousarray(D)).cuda())
    S2, right = B2.schur(fl_prime)
    left = (-S2).cpu().numpy()
    X = cho_solve(cho_factor(left), right.cpu().numpy())
    return np.dot(D, X), X


def optimize_calibration(lwl0, lwl1, lwl_cal, fl_cal, fl_fixed, A, B, C, order=1, mu_GP=1.0):
    """covariance.py:560-624.  A, B, C are the caller-filled covariance blocks (sigma^2 already on the diagonals of
    A and B), numpy arrays or CUDA tensors."""
    fl_cal = np.asarray(fl_cal, dtype=np.float64)
    D = _chebyshev_design(lwl0, lwl1, lwl_cal, fl_cal, order)
    A_d, B_d, C_d = _lib.dev_f64(A), _lib.dev_f64(B), _lib.dev_f64(C)
    n_cal, n_fixed = A_d.shape[0], B_d.shape[0]

    def fill(Bd):
        Bd.data_block().copy_(B_d)
        Bd.border_block(0, n_cal).copy_(A_d)
        Bd.cross_block(0, n_cal).copy_(C_d.T)  # S(border a, data j) = C[a, j]

    resid = _lib.dev_f64(np.asarray(fl_fixed, dtype=np.float64).flatten()) - float(mu_GP)
    return _calibrate(fill, n_cal, n_fixed, resid, D, mu_GP)


def optimize_calibration_static(wl0, wl1, wl_cal, fl_cal, sigma_cal, wl_fixed, fl_fixed, sigma_fixed, amp, l_f, order=1,
                                mu_GP=1.0):
    """covariance.py:627-711: fills A, B, C itself (zero relative velocity between the epochs)."""
    fl_cal = np.asarray(fl_cal, dtype=np.float64)
    D = _chebyshev_design(wl0, wl1, wl_cal, fl_cal, order)
    lc, lf = _lib.dev_f64(wl_cal), _lib.dev_f64(wl_fixed)
    sc, sf = _lib.dev_f64(sigma_cal), _lib.dev_f64(sigma_fixed)
    n_cal, n_fixed = lc.numel(), lf.numel()

    def fill(Bd):
        _fill_data_block(Bd, [lf], [amp], [l_f], sf)
        matrix_functions._fill_v11(Bd.border_block(0, n_cal), [lc], [amp], [l_f])
        Bd.border_block(0, n_cal).diagonal().add_(sc * sc)
        matrix_functions.fill_V12_sum(Bd.cross_block(0, n_cal), [lf], [lc], [amp], [l_f])

    resid = _lib.dev_f64(np.asarray(fl_fixed, dtype=np.float64).flatten()) - float(mu_GP)
    return _calibrate(fill, n_cal, n_fixed, resid, D, mu_GP)


def cycle_calibration(wl, fl, sigma, amp_f, l_f, ncycles, order=1, limit_array=3, mu_GP=1.0, soften=1.0):
    """covariance.py:714-748.  The reference calls optimize_calibration with the argument list of
    optimize_calibration_static (a stale call that raises TypeError); the evident intent is implemented."""
    wl, fl = np.asarray(wl, dtype=np.float64), np.asarray(fl, dtype=np.float64)
    wl0, wl1 = np.min(wl), np.max(wl)
    fl_out = np.copy(fl)
    sigma = soften * np.asarray(sigma, dtype=np.float64)
    for _ in range(ncycles):
        for i in range(len(wl)):
            wl_remain = np.delete(wl, i, axis=0)[0:limit_array]
            fl_remain = np.delete(fl_out, i, axis=0)[0:limit_array]
            sigma_remain = np.delete(sigma, i, axis=0)[0:limit_array]
            fl_cor, _ = optimize_calibration_static(wl0, wl1, wl[i], fl_out[i], sigma[i], wl_remain.flatten(),
                                                    fl_remain.flatten(), sigma_remain.flatten(), amp_f, l_f,
                                                    order=order, mu_GP=mu_GP)
            fl_out[i] = fl_cor
    return fl_out
