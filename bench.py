#!/usr/bin/env python
"""bench.py — lnlike evaluations/s of the PSOAP chunk farm on N B200s (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torch.distributed.run)
  python bench.py --impl reference ...                     (the reference's CPU path on the host cores)
  python bench.py ... --dump-outputs DIR                   (also write the last timed step's output to DIR)

A "step" is one full likelihood evaluation (one MCMC proposal): orbit velocities -> Doppler-shifted covariance
fill -> FP64 Cholesky + solve + log-determinant for every chunk of the workload, and the cross-rank reduction of
the per-chunk scalars.  Default workload C4 (BASELINE.json configs[3], the one the metric "SB2, all chunks at
1/2/4/8 B200" is quoted on): 256 synthetic SB2 chunks, N = 2000..6000, sharded over the ranks by LPT on N^3
(strong scaling: the 256 chunks are fixed).  --workload C1|C2|C3|C5 times the single-chunk configs.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "lnlike evals/sec (SB2, all chunks)"
WORKLOADS = {
    "C1": "C1: SB1 lnlike_f, 1 chunk 20 epochs x 200 px, N=4000",
    "C2": "C2: SB2 lnlike_f_g, 1 chunk 30 epochs x 300 px, N=9000",
    "C3": "C3: ST3 lnlike_f_g_h, 1 chunk 40 epochs x 250 px, N=10000",
    "C4": "C4: SB2 chunk farm, 256 chunks x 20 epochs, N=2000..6000 (sum N^3/3 = 6.8e12 flop)",
    "C5": "C5: SB2 lnlike_f_g, 1 chunk 64 epochs x 512 px, N=32768",
    "C6": "C6: SB2 chunk farm at the reference's own chunk size, 512 chunks x 20 epochs x 80 px, N=1600",
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.rows = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.1 <= t <= t1 + 0.3):
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                "reasons": sorted(reasons)}


CPU_SAMPLE = {"C4": 64, "C6": 64}     # chunks of the configuration evaluated per CPU step (every 4th chunk of C4's 256)


def workload_config(workload, n_chunks, model, world, nbranch):
    """The `config` object of the JSON line; the reference arm prints the same keys."""
    return {"workload": WORKLOADS[workload], "n_chunks": n_chunks, "model": model,
            "partition": "LPT by N^3 + chain term over %d rank(s)" % world, "nbranch": nbranch,
            "l2": "per-step working set (every chunk matrix is rebuilt and factored in place, 32-288 MB "
                  "each) exceeds the 126 MB L2; no flush needed",
            "collective": "one NCCL all_reduce(SUM) of the %d-entry FP64 lnlike vector" % n_chunks
                          if world > 1 else "none (single rank)"}


def cpu_farm(workload, steps, warmup, blas_threads=None):
    """oracle/cpu_farm.py as a subprocess (never shares this process's CUDA context): the reference's CPU path on
    all host cores, one BLAS thread per worker, chunks handed out dynamically, largest first."""
    cmd = [sys.executable, "-m", "oracle.cpu_farm", "--config", workload, "--sample", str(CPU_SAMPLE.get(workload, 1)),
           "--steps", str(steps), "--warmup", str(warmup)]
    if blas_threads:
        cmd += ["--blas-threads", str(blas_threads)]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("oracle.cpu_farm failed: " + out.stderr[-400:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def cpu_baseline_record(r):
    return {"value": r["evals_per_s"], "unit": "evals/s", "cores": r["cores"], "kind": r["kind"],
            "sample": sample_text(r), "workers": r["workers"], "blas_threads_per_worker": r["blas_threads_per_worker"],
            "extrapolated": r["extrapolated"], "scale_to_full": r["scale_to_full"],
            "seconds_per_sample_eval": r["seconds_per_sample_eval"], "cpu_seconds_full": r["cpu_seconds_full"],
            "evals_per_s_from_cpu_seconds": r["evals_per_s_from_cpu_seconds"], "pool_efficiency": r["pool_efficiency"],
            "fill_fraction": r["fill_fraction"], "lapack_fraction": r["lapack_fraction"],
            "sample_N": r["sample_N"], "per_chunk_seconds": [round(x, 4) for x in r["per_chunk_seconds"]]}


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores (oracle/cpu_farm.py as a subprocess:
    reference Cython fill from oracle/_ref + scipy LAPACK, all host cores).  Each step is one pass over a bounded
    sample of the workload (C4: 64 of the 256 chunks, every 4th); value = 1 / (measured seconds per pass x the
    sample-to-workload scale taken from the measured per-chunk seconds)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_farm(args.workload, args.steps, args.warmup)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["evals_per_s"], "unit": "evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * r["seconds_per_sample_eval"], "ms_per_full_evaluation": 1e3 / r["evals_per_s"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, r["n_chunks"], r["model"], world, args.nbranch),
        "cpu_baseline": cpu_baseline_record(r),
        "e2e": {"value": r["evals_per_s"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def sample_text(r):
    if not r["extrapolated"]:
        return ("all %d chunks evaluated by %d worker processes x %d BLAS thread(s) (reference Cython fill + scipy "
                "LAPACK, python glue restated in oracle/oracle.py), dynamic pool, %.2f s per evaluation"
                % (r["n_chunks"], r["workers"], r["blas_threads_per_worker"], r["seconds_per_sample_eval"]))
    return ("%d of %d chunks (every %dth, N=%d..%d) evaluated by %d worker processes x %d BLAS thread(s) (reference "
            "Cython fill + scipy LAPACK, python glue restated in oracle/oracle.py), dynamic pool largest first, "
            "%.2f s per sample pass (pool efficiency %.2f), scaled to the full workload by the measured per-chunk "
            "seconds interpolated in N (x%.2f)"
            % (len(r["sample_chunks"]), r["n_chunks"], max(1, r["n_chunks"] // len(r["sample_chunks"])),
               min(r["sample_N"]), max(r["sample_N"]), r["workers"], r["blas_threads_per_worker"],
               r["seconds_per_sample_eval"], r["pool_efficiency"], r["scale_to_full"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--nbranch", type=int, default=0, help="chunks in flight per GPU (0: 64; 128 for the small chunks of C6)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (the per-chunk log-likelihood "
                         "vector, float64) to DIR/chunk_lnlikes.npy; the inputs depend only on the arguments, so two "
                         "builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.nbranch <= 0:   # measured: C4 4.60 evals/s with 32 branches, 4.62 with 64 (4.66 with rank-1024 updates), 4.60 with 96;
        args.nbranch = 128 if args.workload == "C6" else 64   # C6 (N = 1600) 31.0 / 34.2 / 34.9 with 32 / 64 / 128
    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    # CPU baseline first (rank 0, N=1 only), as its own process, before this process touches CUDA
    cpu_baseline, cpu_run = None, None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        try:
            # bounded sample (C4: 64 of the 256 chunks), 1 warm-up pass + 2 timed passes (C5, one N = 32768 matrix:
            # a single pass of about a minute)
            cpu_run = cpu_farm(args.workload, *((1, 0) if args.workload == "C5" else (2, 1)))
            cpu_baseline = cpu_baseline_record(cpu_run)
            if cpu_run["n_chunks"] == 1 and args.workload != "C5":
                # BASELINE.md asks for the pair "BLAS threads = all cores" and "= 1" on the single-matrix configurations
                one = cpu_farm(args.workload, 1, 0, blas_threads=1)
                cpu_baseline["blas_threads_1"] = {"value": one["evals_per_s"], "unit": "evals/s",
                                                  "fill_fraction": one["fill_fraction"],
                                                  "lapack_fraction": one["lapack_fraction"]}
        except Exception as exc:  # report, do not hide
            cpu_baseline = {"value": None, "unit": "evals/s", "cores": os.cpu_count(), "kind": "port",
                            "sample": "failed: " + str(exc)[-300:]}

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from psoap_b200 import _lib, synthetic
    from psoap_b200.farm import ChunkFarm
    lib = _lib.load()

    model, chunks = synthetic.config_chunks(args.workload)
    p = synthetic.default_params(model)
    farm = ChunkFarm(model, chunks, nbranch=args.nbranch, rank=rank, world_size=world)
    flops_total = float(sum(c["N"] ** 3 / 3.0 + 2.0 * c["N"] ** 2 for c in chunks))

    def proposal(k):
        # a fresh proposal every step (tiny random-walk around the truth), identical on every rank
        q = p.copy()
        q[1] *= 1.0 + 1e-3 * np.sin(k + 1.0)
        q[-1] *= 1.0 + 1e-3 * np.cos(k + 1.0)
        return q

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- kernel-only leg: parameters already on the device, chunk data resident, no host sync inside ----
    p_dev = [torch.from_numpy(proposal(k)).cuda() for k in range(args.warmup + args.steps)]
    for k in range(args.warmup):
        farm.chunk_lnlikes_device(p_dev[k])
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = lib.psoap_launch_count()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for k in range(args.warmup, args.warmup + args.steps):
        lnl_last = farm.chunk_lnlikes_device(p_dev[k])
    e1.record()
    barrier()
    t_wall1 = time.time()
    launches = lib.psoap_launch_count() - launches0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        lt = torch.tensor([float(launches)], dtype=torch.float64, device="cuda")
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    ms_total = float(ms.item())
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    value = args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        # read before the next evaluation overwrites the farm's result buffer (with several ranks the all-reduce has
        # already filled in every chunk)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "chunk_lnlikes.npy"), lnl_last.cpu().numpy())
    lnl_check = float(np.sum(farm.chunk_lnlikes_device(p_dev[-1]).cpu().numpy()))

    # ---- parity, asserted in the same run: the chunks the CPU arm sampled, same parameter vector ----------
    parity = None
    if cpu_run is not None:
        got = farm.chunk_lnlikes(np.asarray(cpu_run["params"])).cpu().numpy()[cpu_run["sample_chunks"]]
        ref = np.asarray(cpu_run["lnlike_per_chunk"])
        rel = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
        parity = {"n": int(len(ref)), "max_rel_err": float(rel.max()), "tol": 1e-10,
                  "against": "reference CPU path (%s fill + scipy LAPACK) on the %d sampled chunks, per chunk"
                             % ("oracle/_ref Cython" if cpu_run["kind"] == "reference" else "oracle C", len(ref))}
        assert np.all(np.isfinite(ref)) and rel.max() <= 1e-10, "parity against the CPU reference failed: %r" % parity

    # ---- per-rank compute time of one evaluation WITHOUT the collective (the all-reduce inside the timed region
    #      equalises the ranks' clocks, so the imbalance cannot be read from it) --------------------------------
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for k in range(3):
        farm.lnprob_device(p_dev[k % len(p_dev)])
    r1.record()
    torch.cuda.synchronize()
    mine = torch.tensor([r0.elapsed_time(r1) / 3.0, farm.cost_of_mine()], dtype=torch.float64, device="cuda")
    allr = [torch.zeros_like(mine) for _ in range(world)]
    if world > 1:
        dist.all_gather(allr, mine)
    else:
        allr = [mine]
    rank_ms = [float(t[0].item()) for t in allr]
    rank_cost = [float(t[1].item()) for t in allr]
    ranks = {"ms_min": min(rank_ms), "ms_mean": float(np.mean(rank_ms)), "ms_max": max(rank_ms), "ms": rank_ms,
             "cost_model_imbalance": max(rank_cost) / float(np.mean(rank_cost)) - 1.0,
             "measured_imbalance": max(rank_ms) / float(np.mean(rank_ms)) - 1.0,
             "what": "device time of one evaluation of the rank's own chunks without the all-reduce (mean of 3); "
                     "imbalance = max / mean - 1"}

    # ---- end-to-end leg: host parameter vector in, host float out, chunk vectors re-uploaded from pinned
    #      host memory every step, device->host read of the per-chunk log-likelihoods every step ------------
    for k in range(2):
        farm.refresh_data(); farm.lnprob(proposal(k))
    barrier()
    t0 = time.perf_counter()
    h2d = 0
    for k in range(args.warmup, args.warmup + args.steps):
        h2d = farm.refresh_data() + farm.n_params * 8
        farm.lnprob(proposal(k))
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    hb = torch.tensor([float(h2d)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dist.all_reduce(hb, op=dist.ReduceOp.SUM)
    e2e_value = args.steps / float(dt.item())

    # ---- dominant kernel (DMMA trailing update) timed alone + live FP64 tensor-pipe peak (rank 0) -----
    roofline = None
    if rank == 0:
        import ctypes
        peak = ctypes.c_double()
        _lib.check(lib.psoap_fp64_peak_tflops(ctypes.byref(peak)))
        avg_ms, fl = ctypes.c_double(), ctypes.c_double()
        m_syrk = {"C1": 4096, "C4": 4096, "C6": 1536}.get(args.workload, 8192)
        # the rank the orchestration uses for this workload: 1024 in the graph farm (8 panels per update), 512 for one
        # very large matrix, 256 for one mid-size matrix
        k_syrk = 1024 if args.workload in ("C4", "C6") else (512 if args.workload == "C5" else 256)
        _lib.check(lib.psoap_bench_syrk(m_syrk, k_syrk, 20, ctypes.byref(avg_ms), ctypes.byref(fl)))
        achieved = fl.value / (avg_ms.value * 1e-3) * 1e-12
        # the same launch with its partial last round dealt out as quarter tiles: faster ALONE, slower in every path that
        # ships (api.cu g_tail_split), so it is reported beside the shipped configuration, not instead of it
        t_ms = ctypes.c_double()
        _lib.check(lib.psoap_bench_syrk_split(m_syrk, k_syrk, 20, 1, ctypes.byref(t_ms), ctypes.byref(fl)))
        achieved_tail = fl.value / (t_ms.value * 1e-3) * 1e-12
        step_tflops = flops_total * value * 1e-12 / world
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "syrk_traffic.json")
        if os.path.exists(tfile):
            traffic = json.load(open(tfile)).get("dram_bytes_per_launch_m%d_k%d" % (m_syrk, k_syrk))
        # the covariance fill alone (HBM-write / FP64-exp bound): the largest chunk of the workload
        big = max(chunks, key=lambda c: c["N"])
        vel_h = synthetic.host_velocities(model, p[:_lib.N_ORB[model]], big["date1D"])
        lw_dev = [torch.from_numpy(np.ascontiguousarray(big["lwl"] - vel_h[c][big["epoch"]] / synthetic.c_kms)).cuda()
                  for c in range(_lib.NCOMP[model])] + [None] * (3 - _lib.NCOMP[model])
        pg = p[_lib.N_ORB[model]:]
        amp_a, l_a = _lib.dbl_array(pg[0::2]), _lib.dbl_array(pg[1::2])
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
        pfile = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pfile):
            hbm_peak, hbm_src = float(json.load(open(pfile))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        fill = {"N": big["N"], "ncomp": _lib.NCOMP[model], "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src}
        nb = float(big["N"])
        for kind, name, nbytes in ((0, "lower", 4.0 * nb * nb), (1, "full", 8.0 * nb * nb)):
            t_ms = ctypes.c_double()
            _lib.check(lib.psoap_bench_fill(kind, _lib.NCOMP[model], big["N"], _lib.ptr(lw_dev[0]), _lib.ptr(lw_dev[1]),
                                            _lib.ptr(lw_dev[2]), amp_a, l_a, 20, ctypes.byref(t_ms)))
            gbs = nbytes / (t_ms.value * 1e-3) * 1e-9
            fill[name] = {"us": t_ms.value * 1e3, "algorithmic_bytes": nbytes, "gbs": gbs, "frac_hbm": gbs / hbm_peak,
                          "gexp_s": _lib.NCOMP[model] * nb * (nb - 1) / 2.0 / (t_ms.value * 1e-3) * 1e-9}
        fill["what"] = ("lower = fill_lower_kernel, the fill the likelihood uses (column-major lower triangle, 4 N^2 "
                        "algorithmic bytes); full = fill_full_kernel, the fill_V11_* operator surface (row-major, both "
                        "triangles, 8 N^2 bytes); gexp_s counts ncomp N (N-1) / 2 exponentials, whether evaluated or "
                        "known to underflow to an exact zero; mean of 20 launches, CUDA events on the launch stream")
        roofline = {"bound": "tensor", "kernel": "syrk3_kernel (tensor-map TMA + DMMA.8x8x4 rank-%d trailing update of an m=%d lower triangle)" % (k_syrk, m_syrk),
                    "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s", "frac": achieved / peak.value,
                    "traffic": traffic,
                    "peak_source": "live DMMA.8x8x4 register-resident loop on all SMs (psoap_fp64_peak_tflops); "
                                   "MEASURED_PEAKS.json has no FP64 entry",
                    "how": "achieved = algorithmic flops of one launch (K m (m+1), the DSYRK convention; the upper halves "
                           "of the diagonal tiles are computed but not counted) / mean duration of 20 back-to-back launches of that kernel alone, "
                           "CUDA events on its launch stream, taken inside bench.py right after the timed region "
                           "(inside the evaluation graph the kernels of 32 branches overlap, so a per-kernel "
                           "duration does not exist there); step_tflops_per_gpu = algorithmic flops of the timed "
                           "region (sum over chunks of N^3/3 + 2N^2) / its measured time",
                    "step_tflops_per_gpu": step_tflops, "step_frac": step_tflops / peak.value,
                    "algorithmic_flops_per_eval": flops_total, "fill": fill,
                    "alone_with_quarter_tail": {
                        "achieved": achieved_tail, "frac": achieved_tail / peak.value,
                        "note": "same launch, the partial last round of its tiles dealt out as quarter tiles "
                                "(psoap_bench_syrk_split): what wave quantisation costs this kernel when NOTHING else "
                                "runs.  Not shipped: in the farm that round is filled by the other branches' kernels "
                                "and the less efficient quarter tiles cost 3 % of the step (PSOAP_TAIL=1)"}}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, len(chunks), model, world, args.nbranch),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": int(hb.item()),
                    "d2h_bytes_per_step": len(chunks) * 8 * world},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "parity": parity,
            "ranks": ranks,
            "lnlike_sum": lnl_check,
        }
        print(json.dumps(line), flush=True)
    farm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
