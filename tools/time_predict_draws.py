"""Time posterior draws of the component spectra on the device (ChunkFarm.draw_components) against the prediction alone
(predict_components) and against the host arm a user has today, one GPU.

The host arm is scripts/psoap_retrieve_SB2.py's step 3: predict_components, Sigma copied to the host, then
numpy.random.default_rng(seed).multivariate_normal(mu, Sigma, S) per (proposal, chunk).  Problems, with the retrieve
script's grid of m = 2 n_pix points per component (M = 400 .. 1200) and S = 64 draws per item:
  1. C4 (256 SB2 chunks), K = 1;
  2. every 8th chunk of C4 (32 chunks), K = 8.
The device variants are the median host wall time of calls that end in a device synchronise, alternating call by call
after one warm-up call each; the host arm (minutes per call) is timed in the same rounds, once per round.  Writes the
report to --out (default profiles/time_predict_draws.txt), with the card name, power limit and SM clock read in the same
run.
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from psoap_b200 import synthetic  # noqa: E402
from psoap_b200.farm import ChunkFarm  # noqa: E402

MUS = (0.5, 0.5)


def timed(fn):
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=1)
    ap.add_argument("--draws", type=int, default=64)
    ap.add_argument("--out", default=os.path.join("profiles", "time_predict_draws.txt"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_predict_draws needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    _, c4 = synthetic.config_chunks("C4")
    p = synthetic.default_params("SB2")
    lines = ["# time_predict_draws: %s (name, power limit, max SM clock, SM clock at start)" % smi,
             "# S = %d draws per item, retrieve grid m = 2 n_pix, SB2 (M = 4 n_pix); medians of wall time ending in a "
             "device synchronise, ms" % a.draws]
    for name, chunks, K in (("C4, K = 1", c4, 1), ("every 8th chunk of C4, K = 8", c4[::8], 8)):
        rng = np.random.default_rng(0)
        P = np.stack([p * (1.0 + 1e-3 * k * rng.uniform(-1.0, 1.0, p.size)) for k in range(K)])
        grids = [np.linspace(ch["lwl"].min(), ch["lwl"].max(), 2 * ch["n_pix"]) for ch in chunks]
        plain = ChunkFarm("SB2", chunks, n_proposals=K)
        plain.attach_prediction_grids(grids)
        drawn = ChunkFarm("SB2", chunks, n_proposals=K)
        drawn.attach_prediction_grids(grids, n_draws=a.draws)

        def host_arm():
            out = plain.predict_components(P, MUS)
            gen = np.random.default_rng(1)
            for mu, S in out:
                mu, S = mu.cpu().numpy(), S.cpu().numpy()
                for k in range(K):
                    gen.multivariate_normal(mu[k], S[k], a.draws)

        dev = {"predict_components": lambda: plain.predict_components(P, MUS),
               "draw_components": lambda: drawn.draw_components(P, MUS, seed=7)}
        for fn in dev.values():
            fn()
        torch.cuda.synchronize()
        ts = {k: [] for k in list(dev) + ["host arm"]}
        for r in range(a.reps):
            for k, fn in dev.items():
                ts[k].append(timed(fn))
            if r < a.host_reps:
                ts["host arm"].append(timed(host_arm))
        # the draws farm's prediction outputs are the plain farm's bits
        same = all(torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])
                   for x, y in zip(plain.predict_components(P, MUS), drawn.draw_components(P, MUS, seed=7)))
        med = {k: float(np.median(v)) for k, v in ts.items()}
        lines.append("%s: %d items, predict_components %.2f, draw_components %.2f (+%.2f), host arm %.0f (%d call%s); "
                     "mu and Sigma bit-identical: %s"
                     % (name, K * len(chunks), med["predict_components"], med["draw_components"],
                        med["draw_components"] - med["predict_components"], med["host arm"], len(ts["host arm"]),
                        "" if len(ts["host arm"]) == 1 else "s", same))
        print(lines[-1], flush=True)
        plain.close()
        drawn.close()
        del plain, drawn
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
