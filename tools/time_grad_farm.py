"""Time the farm's gradient graph (ChunkFarm.lnprob_and_grad_many) against the likelihood graph and the sequential
gradient (ChunkFarm.lnprob_and_grad, one chunk at a time on the direct API), one GPU.

  1. C4 (256 SB2 chunks, N = 2000 .. 6000), one proposal: lnprob, lnprob_and_grad, and lnprob_and_grad_many with
     grad_nbranch = 16 / 32 / 64 (with the bytes each gradient graph allocates);
  2. ensembles: C1 (one SB1 chunk, N = 4000) with K = 8 proposals and every 8th chunk of C4 (32 chunks) with K = 4:
     lnprob_many, lnprob_and_grad_many and K x lnprob_and_grad.
Every figure is the median host wall time of calls that end in a device synchronise, the variants of a table
alternating call by call after one warm-up call each.  In the same run the graph's rows are checked against the
sequential rows with the tolerance of tests/test_gradient_farm.py, and the rows of the three branch counts against
each other (bits).  Writes the report to --out (default profiles/time_grad_farm.txt), with the card name and power
limit read in the same run.
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


def alternate(variants, reps):
    """variants: {name: fn}; one warm-up call each, then `reps` rounds calling each once; median ms per variant."""
    for fn in variants.values():
        fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in variants}
    for _ in range(reps):
        for k, fn in variants.items():
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts[k].append(time.perf_counter() - t0)
    return {k: 1e3 * float(np.median(v)) for k, v in ts.items()}


def check_rows(farm, P, rows, rng):
    """Graph rows [K, n_chunks, n_params + 1] against chunk_lnlike_grads of every proposal: lnlike to 1e-12, and
    |g_graph . u - g_seq . u| <= 1e-10 sum_k |g_seq,k u_k| for random u.  Returns (pairs checked, worst ratio)."""
    worst, n = 0.0, 0
    for k, p in enumerate(P):
        ref = farm.chunk_lnlike_grads(p).cpu().numpy()
        assert np.all(np.abs(rows[k, :, 0] - ref[:, 0]) <= 1e-12 * np.abs(ref[:, 0])), "lnlike"
        for _ in range(2):
            u = rng.standard_normal(farm.n_params)
            err = np.abs(rows[k, :, 1:] @ u - ref[:, 1:] @ u)
            scale = np.sum(np.abs(ref[:, 1:] * u), axis=1)
            worst = max(worst, float(np.max(err / scale)))
        n += len(ref)
    assert worst <= 1e-10, worst
    return n, worst


def proposals(p, K, seed):
    rng = np.random.default_rng(seed)
    return np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])


def main(out_path, reps):
    lib = _lib.load()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say("card: %s (name, power limit, max SM clock; read in this run)" % (smi[0] if smi else "unknown"))
    say("median host wall time of %d alternating calls per variant (after one warm-up call each), each ending in a"
        % reps)
    say("device synchronise")
    rng = np.random.default_rng(0)
    GB = 1e-9

    model, chunks = synthetic.config_chunks("C4")
    p = synthetic.default_params(model)
    P1 = p[None, :]
    say()
    say("1. C4 (%d SB2 chunks, N = %d .. %d), K = 1" % (len(chunks), min(len(c["fl"]) for c in chunks),
                                                       max(len(c["fl"]) for c in chunks)))
    a = ChunkFarm(model, chunks, grad_nbranch=32)           # nbranch 32 for lnprob
    b = ChunkFarm(model, chunks, nbranch=1, grad_nbranch=16)
    res = alternate({"lnprob": lambda: a.lnprob(p), "lnprob_and_grad": lambda: a.lnprob_and_grad(p),
                     "many32": lambda: a.lnprob_and_grad_many(P1), "many16": lambda: b.lnprob_and_grad_many(P1)},
                    reps)
    rows = {32: a.chunk_lnlike_grads_many(P1).cpu().numpy(), 16: b.chunk_lnlike_grads_many(P1).cpu().numpy()}
    nbytes = {16: lib.psoap_farm_grad_workspace_bytes(b._farm, 16), 32: lib.psoap_farm_grad_workspace_bytes(a._farm, 32)}
    b.close()
    del b
    torch.cuda.empty_cache()
    c = ChunkFarm(model, chunks, nbranch=1, grad_nbranch=64)
    res2 = alternate({"lnprob": lambda: a.lnprob(p), "many32": lambda: a.lnprob_and_grad_many(P1),
                      "many64": lambda: c.lnprob_and_grad_many(P1)}, reps)
    rows[64] = c.chunk_lnlike_grads_many(P1).cpu().numpy()
    nbytes[64] = lib.psoap_farm_grad_workspace_bytes(c._farm, 64)
    c.close()
    del c
    torch.cuda.empty_cache()
    t_lp = res["lnprob"]
    say("   %-34s %10.2f ms" % ("lnprob", t_lp))
    say("   %-34s %10.2f ms   (%.2f x lnprob)" % ("lnprob_and_grad (sequential)", res["lnprob_and_grad"],
                                                  res["lnprob_and_grad"] / t_lp))
    for nb, key, src in ((16, "many16", res), (32, "many32", res), (64, "many64", res2)):
        t = src[key]
        tl = src["lnprob"]
        say("   %-34s %10.2f ms   (%.2f x lnprob of the same pass; %.1f GB for the gradient graph)"
            % ("lnprob_and_grad_many, %d branches" % nb, t, t / tl, nbytes[nb] * GB))
    say("   (second pass, alternating lnprob / 32 / 64 branches: lnprob %.2f ms, 32 branches %.2f ms)"
        % (res2["lnprob"], res2["many32"]))
    same = all(np.array_equal(rows[nb], rows[32]) for nb in (16, 64))
    n, worst = check_rows(a, P1, rows[32], rng)
    say("   rows: 16 / 32 / 64 branches bit-identical: %s; against the sequential rows: %d rows, worst"
        " |dg.u| / sum|g u| = %.2e (tolerance 1e-10)" % (same, n, worst))
    a.close()
    del a
    torch.cuda.empty_cache()

    say()
    say("2. ensembles")
    say("   %-30s %3s %14s %22s %18s %10s" % ("problem", "K", "lnprob_many ms", "lnprob_and_grad_many ms",
                                              "K x sequential ms", "speed-up"))
    c4_sub = chunks[::8]
    for name, (mdl, chs), K in (("C1 (1 x N = 4000)", synthetic.config_chunks("C1"), 8),
                                ("C4 every 8th (32 chunks)", ("SB2", c4_sub), 4)):
        P = proposals(synthetic.default_params(mdl), K, seed=K)
        f = ChunkFarm(mdl, chs, n_proposals=K)
        r = alternate({"many": lambda: f.lnprob_many(P), "grad": lambda: f.lnprob_and_grad_many(P),
                       "seq": lambda: [f.lnprob_and_grad(q) for q in P]}, reps)
        n, worst = check_rows(f, P, f.chunk_lnlike_grads_many(P).cpu().numpy(), rng)
        say("   %-30s %3d %14.2f %22.2f %18.2f %9.2fx   (%.2f x lnprob_many; %d rows checked, worst %.1e)"
            % (name, K, r["many"], r["grad"], r["seq"], r["seq"] / r["grad"], r["grad"] / r["many"], n, worst))
        f.close()
        del f
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "time_grad_farm.txt"))
    ap.add_argument("--reps", type=int, default=5)
    main(ap.parse_args().out, ap.parse_args().reps)
