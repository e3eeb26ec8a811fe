"""Time the log-likelihood gradient against the likelihood (device-resident inputs, CUDA events after warm-up).

  1. psoap_lnlike against psoap_lnlike_grad, SB2 (two components), N = 2000, 4000, 6000, 9000;
  2. the contraction kernel (lnlike_grad_kernel) alone, from a torch.profiler pass of its own, in Gexp/s and GB/s;
  3. ChunkFarm.lnprob_and_grad against ChunkFarm.lnprob on the C4 chunk set, one GPU, with the forward-difference
     alternative (n_params + 1 lnprob calls) beside it.
Writes the report to --out (default profiles/time_grad.txt), with the card name and power limit read in the same run.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from psoap_b200 import _lib, synthetic  # noqa: E402
from psoap_b200.farm import ChunkFarm  # noqa: E402

C_KMS = 2.99792458e5


def problem(N, seed=1):
    rng = np.random.default_rng(seed)
    dpix = 2.8 / C_KMS
    base = np.log(5000.0) + np.arange(N) * dpix
    lw = [torch.from_numpy(base - v / C_KMS).cuda() for v in (0.0, 17.0)]
    fl = torch.from_numpy(1.0 + 0.1 * rng.standard_normal(N)).cuda()
    sg = torch.from_numpy(np.full(N, 0.03)).cuda()
    return lw, fl, sg


def event_ms(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), float(min(times))


def main(out_path):
    lib = _lib.load()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say("card: %s (name, power limit, max SM clock; read in this run)" % (smi[0] if smi else "unknown"))
    amps, ls = _lib.dbl_array([0.1, 0.07]), _lib.dbl_array([5.0, 6.0])
    say("")
    say("1. single problem, SB2 (2 components), median of 10 CUDA-event timings after 2 warm-up calls")
    say("%6s %12s %12s %8s" % ("N", "lnlike ms", "grad ms", "ratio"))
    contraction = []
    for N in (2000, 4000, 6000, 9000):
        lw, fl, sg = problem(N)
        nb1 = lib.psoap_lnlike_workspace_bytes(N)
        ws1 = torch.empty(nb1 + 256, dtype=torch.uint8, device="cuda")
        nb2 = lib.psoap_lnlike_grad_workspace_bytes(2, N)
        ws2 = torch.empty(nb2 + 256, dtype=torch.uint8, device="cuda")
        res = torch.empty(4, dtype=torch.float64, device="cuda")
        gh = torch.empty(5, dtype=torch.float64, device="cuda")
        gl = torch.empty((2, N), dtype=torch.float64, device="cuda")

        def f1():
            _lib.check(lib.psoap_lnlike(2, N, _lib.ptr(lw[0]), _lib.ptr(lw[1]), None, _lib.ptr(fl), _lib.ptr(sg), amps, ls,
                                        1.0, _lib.ptr(ws1), nb1, _lib.ptr(res), _lib.stream_ptr()))

        def f2():
            _lib.check(lib.psoap_lnlike_grad(2, N, _lib.ptr(lw[0]), _lib.ptr(lw[1]), None, _lib.ptr(fl), _lib.ptr(sg), amps,
                                             ls, 1.0, _lib.ptr(ws2), nb2, _lib.ptr(res), _lib.ptr(gh), _lib.ptr(gl),
                                             _lib.stream_ptr()))
        t1, _ = event_ms(f1, 10)
        t2, _ = event_ms(f2, 10)
        say("%6d %12.3f %12.3f %8.2f" % (N, t1, t2, t2 / t1))
        # the contraction kernel alone: a profiler pass of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                f2()
            torch.cuda.synchronize()
        ev = [e for e in prof.events() if "lnlike_grad_kernel" in e.name]
        allk = [e for e in prof.events() if e.device_type.name == "CUDA"]
        if ev:
            us = sum(e.device_time for e in ev) / len(ev)
            tot = sum(e.device_time for e in allk) / 3
            contraction.append((N, us, tot))
        del ws1, ws2
        torch.cuda.empty_cache()
    say("")
    say("2. contraction kernel lnlike_grad_kernel<2> alone (torch.profiler, mean of 3 calls); 2 exponentials per")
    say("   lower-triangle entry (N^2 / 2 entries), bytes = the -K^-1 lower triangle read once (4 N^2).  The likelihood's")
    say("   fill_lower_kernel runs at 575 Gexp/s (profiles/fill_time_r02.txt).")
    say("%6s %10s %10s %10s %14s" % ("N", "us", "Gexp/s", "GB/s", "share of call"))
    for N, us, tot in contraction:
        say("%6d %10.1f %10.1f %10.1f %13.1f%%" % (N, us, 2 * N * N / 2 / (us * 1e3), 4.0 * N * N / (us * 1e3),
                                                  100.0 * us / tot))
    say("")
    model, chunks = synthetic.config_chunks("C4")
    p = synthetic.default_params(model)
    farm = ChunkFarm(model, chunks)
    farm.lnprob(p); farm.lnprob_and_grad(p)
    torch.cuda.synchronize()

    def wall(fn, reps):
        fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
        return 1e3 * float(np.median(ts))
    t_lp = wall(lambda: farm.lnprob(p), 10)
    t_gr = wall(lambda: farm.lnprob_and_grad(p), 5)
    npar = farm.n_params
    say("3. ChunkFarm on C4 (%d SB2 chunks, N = %d .. %d), one GPU, median host wall time (both end in a device"
        % (len(chunks), min(farm.Ns), max(farm.Ns)))
    say("   synchronise)")
    say("   lnprob                      %10.2f ms" % t_lp)
    say("   lnprob_and_grad             %10.2f ms   (%.1f x lnprob)" % (t_gr, t_gr / t_lp))
    say("   forward differences         %10.2f ms   (%d x lnprob: lnprob at p and at p + h e_k, k < %d)"
        % ((npar + 1) * t_lp, npar + 1, npar))
    farm.close()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "time_grad.txt"))
    main(ap.parse_args().out)
