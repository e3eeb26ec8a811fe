"""ctypes binding of the C ABI in include/psoap_b200.h (csrc/libpsoap_b200.so) and device plumbing.

PyTorch is used only for device memory, streams and torch.distributed.  There is no CPU fallback: every
compute entry raises when the library or a CUDA device is missing.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libpsoap_b200.so")

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)
c_i64_p = ctypes.POINTER(ctypes.c_int64)
c_i32_p = ctypes.POINTER(ctypes.c_int32)
vp = ctypes.c_void_p

MODELS = {"SB1": 1, "SB2": 2, "ST1": 3, "ST2": 4, "ST3": 5}
NCOMP = {"SB1": 1, "SB2": 2, "ST1": 1, "ST2": 2, "ST3": 3}
N_ORB = {"SB1": 6, "SB2": 7, "ST1": 11, "ST2": 12, "ST3": 13}  # psoap/utils.py:14


class PsoapResult(ctypes.Structure):
    _fields_ = [("lnlike", ctypes.c_double), ("logdet", ctypes.c_double), ("quad", ctypes.c_double),
                ("info", ctypes.c_double)]


class PsoapChunk(ctypes.Structure):
    _fields_ = [("N", ctypes.c_int64), ("n_epochs", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("lwl", vp), ("epoch", vp), ("fl", vp), ("sigma", vp), ("dates", vp)]


# name -> (restype, argtypes); every symbol include/psoap_b200.h declares
SIGNATURES = {
    "psoap_last_error": (ctypes.c_char_p, []),
    "psoap_version": (ctypes.c_int, []),
    "psoap_device_count": (ctypes.c_int, []),
    "psoap_fill_v11": (ctypes.c_int, [ctypes.c_int, vp, ctypes.c_int64, ctypes.c_int64, vp, vp, vp, c_double_p,
                                      c_double_p, vp]),
    "psoap_fill_v11_host": (ctypes.c_int, [ctypes.c_int, c_double_p, ctypes.c_int64, ctypes.c_int64, c_double_p, c_double_p,
                                           c_double_p, c_double_p, c_double_p]),
    "psoap_fill_v12": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, vp, vp, ctypes.c_double,
                                      ctypes.c_double, vp]),
    "psoap_fill_v12n": (ctypes.c_int, [ctypes.c_int, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                       ctypes.POINTER(vp), ctypes.POINTER(vp), c_double_p, c_double_p, vp]),
    "psoap_replicate_wls": (ctypes.c_int, [vp, vp, vp, ctypes.c_int64, vp, ctypes.c_int, ctypes.c_int, vp]),
    "psoap_orbit_velocities": (ctypes.c_int, [ctypes.c_int, vp, vp, ctypes.c_int, vp, vp, vp]),
    "psoap_model_ncomp": (ctypes.c_int, [ctypes.c_int]),
    "psoap_model_norb": (ctypes.c_int, [ctypes.c_int]),
    "psoap_lnlike_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64]),
    "psoap_lnlike": (ctypes.c_int, [ctypes.c_int, ctypes.c_int64, vp, vp, vp, vp, vp, c_double_p, c_double_p,
                                    ctypes.c_double, vp, ctypes.c_size_t, vp, vp]),
    "psoap_lnlike_host": (ctypes.c_int, [ctypes.c_int, ctypes.c_int64, c_double_p, c_double_p, c_double_p, c_double_p,
                                         c_double_p, c_double_p, c_double_p, ctypes.c_double,
                                         ctypes.POINTER(PsoapResult)]),
    "psoap_schur_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int64]),
    "psoap_schur": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, vp, ctypes.c_size_t, vp, vp]),
    "psoap_schur_views": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(vp), ctypes.POINTER(vp),
                                         ctypes.POINTER(vp)]),
    "psoap_lnlike_grad_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int64]),
    "psoap_lnlike_grad": (ctypes.c_int, [ctypes.c_int, ctypes.c_int64, vp, vp, vp, vp, vp, c_double_p, c_double_p,
                                         ctypes.c_double, vp, ctypes.c_size_t, vp, vp, vp, vp]),
    "psoap_lnlike_grad_views": (ctypes.c_int, [vp, ctypes.c_int64, ctypes.POINTER(vp), c_i64_p, ctypes.POINTER(vp)]),
    "psoap_chunk_lnprob_grad_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int64, ctypes.c_int32]),
    "psoap_chunk_lnprob_grad": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(PsoapChunk), vp, ctypes.c_double, vp,
                                               ctypes.c_size_t, vp, vp, vp]),
    "psoap_orbit_jacobian": (ctypes.c_int, [ctypes.c_int, vp, vp, ctypes.c_int, vp, vp]),
    "psoap_predict_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64]),
    "psoap_predict": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(vp), vp,
                                     vp, ctypes.POINTER(vp), c_double_p, c_double_p, ctypes.c_double, ctypes.c_double,
                                     vp, vp, vp, ctypes.c_size_t, vp, vp]),
    "psoap_predict_host": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                          ctypes.POINTER(c_double_p), c_double_p, c_double_p,
                                          ctypes.POINTER(c_double_p), c_double_p, c_double_p, ctypes.c_double,
                                          ctypes.c_double, c_double_p, c_double_p, ctypes.POINTER(PsoapResult)]),
    "psoap_farm_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, c_i64_p, c_i32_p, ctypes.c_int]),
    "psoap_farm_create": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, ctypes.POINTER(PsoapChunk),
                                         ctypes.c_int, ctypes.c_double, vp, ctypes.c_size_t]),
    "psoap_farm_workspace_bytes_batched": (ctypes.c_size_t, [ctypes.c_int, c_i64_p, c_i32_p, ctypes.c_int,
                                                             ctypes.c_int]),
    "psoap_farm_create_batched": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int,
                                                 ctypes.POINTER(PsoapChunk), ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_double, vp, ctypes.c_size_t]),
    "psoap_farm_lnprob": (ctypes.c_int, [vp, vp, vp, vp]),
    "psoap_farm_launches_per_eval": (ctypes.c_int, [vp]),
    "psoap_farm_destroy": (ctypes.c_int, [vp]),
    "psoap_fp64_peak_tflops": (ctypes.c_int, [c_double_p]),
    "psoap_bench_syrk": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, c_double_p, c_double_p]),
    "psoap_bench_syrk_split": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_double_p, c_double_p]),
    "psoap_debug_fill_lower": (ctypes.c_int, [ctypes.c_int, ctypes.c_int64, vp, vp, vp, vp, vp, ctypes.c_int, vp, vp,
                                              c_double_p, c_double_p, ctypes.c_double, vp, ctypes.c_int64, vp, vp]),
    "psoap_bench_fill": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int64, vp, vp, vp, c_double_p, c_double_p,
                                        ctypes.c_int, c_double_p]),
    "psoap_debug_syrk_tiles": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, c_int_p, c_int_p, ctypes.c_int]),
    "psoap_launch_count": (ctypes.c_int64, []),
}

_lib = None


def load():
    """Load libpsoap_b200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m psoap_b200._build` (nvcc, sm_100a). "
                "psoap_b200 has no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


class PsoapError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = load().psoap_last_error()
        raise PsoapError(f"psoap_b200 error {rc}: {msg.decode() if msg else ''}")


def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("psoap_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def dev_f64(x, device=None):
    """numpy array / sequence / torch tensor -> contiguous float64 CUDA tensor (uploads host data)."""
    torch = torch_cuda()
    if isinstance(x, torch.Tensor):
        t = x
        if t.dtype != torch.float64:
            raise ValueError("expected a float64 tensor")
        if not t.is_cuda:
            t = t.cuda(device)
        return t.contiguous()
    a = np.ascontiguousarray(x, dtype=np.float64)
    return torch.from_numpy(a).cuda(device)


def ptr(t):
    return vp(t.data_ptr()) if t is not None else vp(None)


def stream_ptr():
    torch = torch_cuda()
    return vp(torch.cuda.current_stream().cuda_stream)


def dbl_array(vals):
    return (ctypes.c_double * len(vals))(*[float(v) for v in vals])


_workspaces = {}


def workspace(nbytes, key="default"):
    """Grow-only per-device byte workspace (torch allocations are >= 512-byte aligned)."""
    torch = torch_cuda()
    k = (torch.cuda.current_device(), key)
    buf = _workspaces.get(k)
    if buf is None or buf.numel() < nbytes:
        _workspaces.pop(k, None)
        buf = torch.empty(int(nbytes), dtype=torch.uint8, device="cuda")
        _workspaces[k] = buf
    return buf
