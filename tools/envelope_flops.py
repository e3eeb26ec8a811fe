"""CPU: the factorisation envelope of a workload's chunks and the flops it saves.

For every `--stride`-th chunk of a synthetic configuration (pixels in wavelength order, as ChunkFarm packs them,
velocities at the package's default parameters) prints N, the row blocks T, the envelope tend[e] at every group end,
and the DMMA flops the grouped factorisation executes (psoap_b200.envelope): dense, restricted to the envelope's rows,
and with the update tiles' k loops also starting at each row block's profile (what the device runs).
The flags come from numpy's exp of the device's (p2 r) r; the device's own envelope is printed by
tools/time_envelope.py.

    python tools/envelope_flops.py --config C4 --stride 16 --group 8
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from psoap_b200 import envelope, synthetic  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C4")
    ap.add_argument("--stride", type=int, default=16)
    ap.add_argument("--group", type=int, default=8)
    ap.add_argument("--unsorted", action="store_true", help="keep the epoch-major pixel order")
    args = ap.parse_args()
    model, chunks = synthetic.config_chunks(args.config)
    p = synthetic.default_params(model)
    norb = len(synthetic.ORBIT_PARAMS[model])
    ncomp = synthetic.NCOMP[model]
    amps, ls = p[norb::2][:ncomp], p[norb + 1::2][:ncomp]
    tot_dense = tot_env = tot_k = 0.0
    print("%-6s %5s %4s %14s %14s %14s %7s  tend at group ends" % ("chunk", "N", "T", "dense GF", "restricted GF",
                                                                    "k start GF", "ratio"))
    for i in range(0, len(chunks), args.stride):
        ch = chunks[i]
        vel = synthetic.host_velocities(model, p[:norb], ch["date1D"])
        if args.unsorted:
            ep = ch["epoch"]
            zs = np.array([ch["lwl"] + (-np.asarray(v)[ep]) / synthetic.c_kms for v in vel])
        else:
            _, zs = envelope.sorted_chunk_z(ch, vel)
        flags = envelope.tile_flags_from_z(zs, amps, ls, ch["sigma"])
        tend = envelope.tend_by_end(flags)
        T = flags.shape[0]
        dense = envelope.executed_flops(T, args.group)
        env = envelope.executed_flops(T, args.group, tend)
        kst = envelope.executed_flops(T, args.group, tend, envelope.row_profile(flags))
        tot_dense += dense
        tot_env += env
        tot_k += kst
        ends = envelope.group_starts(T, args.group)[1:]
        print("%-6d %5d %4d %14.2f %14.2f %14.2f %7.3f  %s" % (i, len(ch["fl"]), T, dense / 1e9, env / 1e9, kst / 1e9,
                                                             dense / kst, " ".join(str(int(tend[e])) for e in ends)))
    print("total: dense %.1f GF, restricted %.1f GF, with the k start %.1f GF, dense / executed %.3f"
          % (tot_dense / 1e9, tot_env / 1e9, tot_k / 1e9, tot_dense / tot_k))


if __name__ == "__main__":
    main()
