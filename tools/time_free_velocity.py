"""Time the free-velocity farm (ChunkFarm(..., free_velocities=True)) against the orbit farm on the same chunks, one GPU.

C4 (256 SB2 chunks, N = 2000 .. 6000, 20 epochs each at dates of their own: Ng = 5120 global epochs, so the free vector
has 2 x 5120 + 4 entries): lnprob and lnprob_and_grad_many (grad_nbranch = 16) in orbit and free mode, K = 1, the free
vector holding the orbit's velocities (psoap_orbit_velocities on the device at the global epochs).  The free path swaps
the O(n_epochs) orbit kernel (and, for the gradient, the orbit Jacobian) for a gather, so the times should agree within
noise; the free gradient rows are 2 Ng + 4 wide instead of 11, which the host-side sum sees.  Every figure is the median
host wall time of calls that end in a device synchronise, the variants alternating call by call after one warm-up call
each.  The same run checks that free-mode lnprob is the orbit farm's bits.  Writes the report to --out (default
profiles/time_free_velocity.txt), with the card name, power limit and clocks read in the same run.
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


def orbit_velocities(model, p, dates):
    lib = _lib.load()
    pd = torch.from_numpy(np.ascontiguousarray(p)).cuda()
    dd = torch.from_numpy(np.ascontiguousarray(dates)).cuda()
    vel = torch.empty((_lib.NCOMP[model], len(dates)), dtype=torch.float64, device="cuda")
    _lib.check(lib.psoap_orbit_velocities(_lib.MODELS[model], _lib.ptr(pd), _lib.ptr(dd), len(dates), _lib.ptr(vel),
                                          None, _lib.stream_ptr()))
    return vel.cpu().numpy()


def main(out_path, reps):
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks.mem"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    say("card: %s (%s; read in this run)" % (smi[0] if smi else "unknown", q))
    say("median host wall time of %d alternating calls per variant (after one warm-up call each), each ending in a"
        % reps)
    say("device synchronise")
    model, chunks = synthetic.config_chunks("C4")
    p = synthetic.default_params(model)
    orb = ChunkFarm(model, chunks, grad_nbranch=16)
    fre = ChunkFarm(model, chunks, grad_nbranch=16, free_velocities=True)
    Ng = len(fre.epochs)
    v = np.concatenate([orbit_velocities(model, p, fre.epochs).reshape(-1), p[_lib.N_ORB[model]:]])
    say()
    say("C4 (%d SB2 chunks, N = %d .. %d), K = 1; free mode: Ng = %d global epochs, %d parameters"
        % (len(chunks), min(len(c["fl"]) for c in chunks), max(len(c["fl"]) for c in chunks), Ng, fre.n_params))
    same = fre.lnprob(v) == orb.lnprob(p) and torch.equal(fre.chunk_lnlikes(v), orb.chunk_lnlikes(p))
    res = alternate({"orbit lnprob": lambda: orb.lnprob(p), "free lnprob": lambda: fre.lnprob(v),
                     "orbit lnprob_and_grad_many": lambda: orb.lnprob_and_grad_many(p[None]),
                     "free lnprob_and_grad_many": lambda: fre.lnprob_and_grad_many(v[None])}, reps)
    for what in ("lnprob", "lnprob_and_grad_many"):
        to, tf = res["orbit " + what], res["free " + what]
        say("   %-22s orbit %9.2f ms   free %9.2f ms   (free / orbit %.3f)" % (what, to, tf, tf / to))
    say("   launches per likelihood evaluation: orbit %d, free %d" % (orb.launches_per_eval, fre.launches_per_eval))
    say("   free-mode lnprob and per-chunk lnlikes at the orbit's velocities are the orbit farm's bits: %s" % same)
    orb.close()
    fre.close()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "time_free_velocity.txt"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    main(args.out, args.reps)
