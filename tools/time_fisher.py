"""Time the expected Fisher information (psoap_chunk_fisher, ChunkFarm.fisher), one GPU.

  1. one wavelength-sorted SB2 chunk (20 epochs) at N = 2000, 4000 and 6000: psoap_chunk_fisher against
     psoap_chunk_lnprob_grad, with the GEMM flops the k ranges leave (counted from the ranges the device returns) and
     the rate they run at over the whole call;
  2. C4 (256 SB2 chunks, N = 2000 .. 6000): ChunkFarm.fisher, against lnprob and 2 P x lnprob_and_grad_many (what
     central differences of the gradient would cost).
Chunk times are the median of CUDA-event timed calls after one warm-up call; the C4 figures are host wall times of
calls that end in a device synchronise.  Writes the report to --out (default profiles/time_fisher.txt), with the card
name and power limit read in the same run.
"""
import argparse
import ctypes
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from psoap_b200 import _lib, synthetic  # noqa: E402
from psoap_b200.farm import ChunkFarm  # noqa: E402


def sorted_chunk(n_pix, seed):
    ch = synthetic.make_chunk("SB2", 20, n_pix, seed=seed)
    order = np.argsort(ch["lwl"], kind="stable")
    for k in ("lwl", "fl", "sigma", "epoch"):
        ch[k] = np.ascontiguousarray(ch[k][order])
    return ch


def chunk_times(ch, p, reps):
    """(fisher ms, gradient ms, executed GEMM flops, dense GEMM flops) of one chunk on the direct API."""
    lib = _lib.load()
    m = _lib.MODELS["SB2"]
    t = {k: torch.from_numpy(np.ascontiguousarray(ch[k])).cuda() for k in ("lwl", "fl", "sigma", "date1D", "epoch")}
    d = _lib.PsoapChunk()
    d.N, d.n_epochs = len(ch["fl"]), len(ch["date1D"])
    d.lwl, d.epoch, d.fl = t["lwl"].data_ptr(), t["epoch"].data_ptr(), t["fl"].data_ptr()
    d.sigma, d.dates = t["sigma"].data_ptr(), t["date1D"].data_ptr()
    nb = lib.psoap_chunk_fisher_workspace_bytes(m, d.N, d.n_epochs)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    P = len(p)
    p_d = torch.from_numpy(p.copy()).cuda()
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    g = torch.empty(P, dtype=torch.float64, device="cuda")
    F = torch.empty((P, P), dtype=torch.float64, device="cuda")
    st = _lib.stream_ptr()
    calls = {
        "fisher": lambda: _lib.check(lib.psoap_chunk_fisher(m, ctypes.byref(d), _lib.ptr(p_d), 1.0, _lib.ptr(ws), nb,
                                                            _lib.ptr(res), _lib.ptr(g), _lib.ptr(F), st)),
        "grad": lambda: _lib.check(lib.psoap_chunk_lnprob_grad(m, ctypes.byref(d), _lib.ptr(p_d), 1.0, _lib.ptr(ws), nb,
                                                               _lib.ptr(res), _lib.ptr(g), st)),
    }
    out = {}
    for name, fn in calls.items():
        fn()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        out[name] = float(np.median(ts))
    calls["fisher"]()
    kr, Tb = _lib.vp(), ctypes.c_int()
    _lib.check(lib.psoap_chunk_fisher_views(_lib.ptr(ws), m, d.N, d.n_epochs, None, ctypes.byref(kr), ctypes.byref(Tb)))
    T = Tb.value
    off = kr.value - ws.data_ptr()
    krange = ws[off:off + 8 * T].cpu().numpy().view(np.int32).reshape(T, 2)
    Nn = 128 * T
    executed = 2.0 * P * Nn * 128 * float(np.sum(128 * (krange[:, 1] - krange[:, 0] + 1)))
    dense = 2.0 * P * float(Nn) ** 3
    assert np.isfinite(F.cpu().numpy()).all()
    return out["fisher"], out["grad"], executed, dense


def wall(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def main(out_path, reps):
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say("card: %s (name, power limit, max SM clock; read in this run)" % (smi[0] if smi else "unknown"))
    p = synthetic.default_params("SB2")
    P = len(p)
    say()
    say("1. one SB2 chunk (20 epochs, pixels in ln-wavelength order), P = %d; median of %d CUDA-event timed calls" % (P, reps))
    say("   %6s %12s %16s %10s %14s %14s %12s" % ("N", "fisher ms", "lnprob_grad ms", "ratio", "GEMM TFLOP", "dense TFLOP",
                                                  "TFLOP/s"))
    for N in (2000, 4000, 6000):
        tf, tg, ex, dense = chunk_times(sorted_chunk(N // 20, seed=N), p, reps)
        say("   %6d %12.2f %16.2f %10.1f %14.3f %14.3f %12.1f" % (N, tf, tg, tf / tg, ex * 1e-12, dense * 1e-12,
                                                                   ex / (tf * 1e-3) * 1e-12))
        torch.cuda.empty_cache()
    say("   (TFLOP/s: executed GEMM flops over the whole psoap_chunk_fisher call, gradient steps included)")

    say()
    model, chunks = synthetic.config_chunks("C4")
    say("2. C4 (%d SB2 chunks, N = %d .. %d); median host wall time of %d calls after one warm-up call"
        % (len(chunks), min(len(c["fl"]) for c in chunks), max(len(c["fl"]) for c in chunks), max(1, reps // 3)))
    farm = ChunkFarm(model, chunks)
    t_fisher = wall(lambda: farm.fisher(p), max(1, reps // 3))
    t_lnp = wall(lambda: farm.lnprob(p), reps)
    t_many = wall(lambda: farm.lnprob_and_grad_many(p[None, :]), reps)
    F = farm.fisher(p)
    say("   %-40s %12.1f ms" % ("ChunkFarm.fisher", t_fisher))
    say("   %-40s %12.1f ms" % ("lnprob", t_lnp))
    say("   %-40s %12.1f ms   (one call %.1f ms)" % ("2 P x lnprob_and_grad_many", 2 * P * t_many, t_many))
    say("   F symmetric (==): %s; finite: %s; diagonal: %s" % (np.array_equal(F, F.T), np.isfinite(F).all(),
                                                                " ".join("%.3e" % v for v in np.diag(F))))
    farm.close()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "time_fisher.txt"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    main(a.out, a.reps)
