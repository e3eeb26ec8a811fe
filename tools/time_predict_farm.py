"""Time the farm's prediction graph (ChunkFarm.predict_components) against the sequential path a user has today, one GPU.

The sequential path is scripts/psoap_retrieve_SB2.py's loop: per proposal and chunk, host velocities
(orbit.velocities), the Doppler shift (data.replicate_wls) and one covariance.predict_f_g call; the flux, noise and
grids are resident on the device, so both paths leave mu and Sigma on the device.  Problems, with the retrieve script's
grid of m = 2 n_pix points per component (M = 400 .. 1200):
  1. C4 (256 SB2 chunks, N = 2000 .. 6000), K = 1, predict_nbranch = 16 / 32 / 64;
  2. every 8th chunk of C4 (32 chunks), K = 8, predict_nbranch = 16 / 32 / 64.
Every figure is the median host wall time of calls that end in a device synchronise, the variants of a table
alternating call by call after one warm-up call each; the rate counts N^3/3 + N^2 M + N M^2 flops per item.  In the
same run the graph's outputs are checked against the sequential ones, and the outputs of the three branch counts
against each other (bits).  Writes the report to --out (default profiles/time_predict_farm.txt), with the card name and
power limit read in the same run.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from psoap_b200 import _lib, covariance, data, orbit, synthetic  # noqa: E402
from psoap_b200.farm import ChunkFarm  # noqa: E402

MUS = (0.5, 0.5)


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


def proposals(p, K, seed):
    rng = np.random.default_rng(seed)
    return np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])


def grid_of(ch):
    """The retrieve script's grid: 2 n_pix points over the chunk's range."""
    m = 2 * ch["n_pix"]
    return np.linspace(ch["lwl"].min(), ch["lwl"].max(), m)


def flops(chunks, K):
    f = 0.0
    for ch in chunks:
        N, M = float(len(ch["fl"])), 2.0 * 2 * ch["n_pix"]
        f += N ** 3 / 3 + N * N * M + N * M * M
    return K * f


class Sequential:
    """The per-chunk loop of the retrieve script for SB2, with the chunk's vectors and grid resident on the device."""

    def __init__(self, chunks):
        self.chunks = chunks
        self.dev = [(torch.from_numpy(ch["fl"]).cuda(), torch.from_numpy(ch["sigma"]).cuda(),
                     torch.from_numpy(grid_of(ch)).cuda()) for ch in chunks]

    def __call__(self, P):
        out = []
        for p in P:
            for ch, (fl, sg, g) in zip(self.chunks, self.dev):
                v = orbit.velocities("SB2", p[:7], ch["date1D"]).cpu().numpy()
                lw = data.replicate_wls(ch["lwl"], v, ch["mask"])
                out.append(covariance.predict_f_g(lw[0], lw[1], fl, sg, g, g, MUS[0], p[7], p[8], MUS[1], p[9], p[10]))
        return out


def worst_diff(outs, seq, K):
    """max |graph - sequential| over mu and Sigma, relative to max |Sigma| (the terms' scale)."""
    w = 0.0
    for i, (mu, S) in enumerate(outs):
        for k in range(K):
            mu_s, S_s = seq[k * len(outs) + i]
            scale = float(S_s.abs().max())
            w = max(w, float((mu[k] - mu_s).abs().max()) / scale, float((S[k] - S_s).abs().max()) / scale)
    return w


def main(out_path, reps):
    _lib.load()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say("card: %s (name, power limit, max SM clock; read in this run)" % (smi[0] if smi else "unknown"))
    say("median host wall time of %d alternating calls per variant (after one warm-up call each), each ending in a"
        % reps)
    say("device synchronise; rate = sum over items of N^3/3 + N^2 M + N M^2 over that time")
    model, c4 = synthetic.config_chunks("C4")
    p = synthetic.default_params(model)
    for title, chunks, K in (("1. C4 (256 SB2 chunks, N = 2000 .. 6000, M = 400 .. 1200), K = 1", c4, 1),
                             ("2. every 8th chunk of C4 (32 chunks), K = 8", c4[::8], 8)):
        say()
        say(title)
        P = proposals(p, K, seed=K)
        seq = Sequential(chunks)
        grids = [grid_of(ch) for ch in chunks]
        fl = flops(chunks, K)
        farms, outs, nbytes, res = {}, {}, {}, {}
        for nb in (16, 32, 64):
            f = ChunkFarm(model, chunks, n_proposals=K, nbranch=1)
            f.attach_prediction_grids(grids, predict_nbranch=nb)
            nbytes[nb] = int(f._pred["ws"].numel())
            farms[nb] = f
            r = alternate({"graph": lambda: f.predict_components(P, MUS), "seq": lambda: seq(P)}, reps)
            res[nb] = r
            outs[nb] = [(mu.cpu(), S.cpu()) for mu, S in f.predict_components(P, MUS)]
            f.close()
            del farms[nb], f
            torch.cuda.empty_cache()
        ref = [(mu.cpu(), S.cpu()) for mu, S in seq(P)]
        same = all(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) for nb in (32, 64)
                   for a, b in zip(outs[nb], outs[16]))
        say("   %-38s %12s %12s %14s %12s" % ("variant", "graph ms", "seq ms", "graph TFLOP/s", "seq / graph"))
        for nb in (16, 32, 64):
            r = res[nb]
            say("   %-38s %12.2f %12.2f %14.2f %11.2fx" % ("predict_nbranch = %d (%.1f GB)" % (nb, nbytes[nb] * 1e-9),
                                                          r["graph"], r["seq"], fl / (r["graph"] * 1e-3) * 1e-12,
                                                          r["seq"] / r["graph"]))
        say("   outputs: 16 / 32 / 64 branches bit-identical: %s; against the sequential path: worst |d| / max|Sigma|"
            " = %.2e" % (same, worst_diff(outs[16], ref, K)))
        del seq, outs, ref
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "time_predict_farm.txt"))
    ap.add_argument("--reps", type=int, default=5)
    main(ap.parse_args().out, ap.parse_args().reps)
