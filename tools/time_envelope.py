"""GPU: the envelope the device computes for a workload's chunks, the flops it executes, and the time of one chunk.

For every `--stride`-th chunk of a synthetic configuration (pixels in wavelength order, as ChunkFarm packs them, at
the package's default parameters) runs psoap_lnlike, reads the envelope back from its workspace
(psoap_lnlike_envelope_view) and prints it with the DMMA flops the grouped factorisation executes, dense and
restricted (psoap_b200.envelope.executed_flops), and the call's time (CUDA events, median of `--reps`) in wavelength
and in epoch-major order.  Prints the card's name, power limit and SM clock first.

    python tools/time_envelope.py --config C4 --stride 16 --out profiles/time_envelope_c4.txt
"""
import argparse
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from psoap_b200 import _lib, envelope, synthetic  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run_chunk(lib, torch, zs, fl, sg, amps, ls, reps):
    N, ncomp = len(fl), len(zs)
    zd = [torch.tensor(np.ascontiguousarray(z), dtype=torch.float64, device="cuda") for z in zs]
    fd = torch.tensor(fl, dtype=torch.float64, device="cuda")
    sd = torch.tensor(sg, dtype=torch.float64, device="cuda")
    nbytes = lib.psoap_lnlike_workspace_bytes(N)
    ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
    wp = (ws.data_ptr() + 255) // 256 * 256
    res = torch.empty(4, dtype=torch.float64, device="cuda")
    ptrs = [z.data_ptr() for z in zd] + [None] * (3 - ncomp)
    st = torch.cuda.current_stream().cuda_stream

    def call():
        _lib.check(lib.psoap_lnlike(ncomp, N, ptrs[0], ptrs[1], ptrs[2], fd.data_ptr(), sd.data_ptr(),
                                    _lib.dbl_array(amps), _lib.dbl_array(ls), 1.0, wp, nbytes, res.data_ptr(), st))
    for _ in range(3):
        call()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    tp, T = _lib.vp(), ctypes.c_int()
    _lib.check(lib.psoap_lnlike_envelope_view(wp, N, ctypes.byref(tp), ctypes.byref(T)))
    off = tp.value - ws.data_ptr()
    tend = ws[off:off + 4 * (T.value + 1)].view(torch.int32).cpu().numpy().astype(np.int64)
    return tend, float(np.median(times)), float(res[0].item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C4")
    ap.add_argument("--stride", type=int, default=16)
    ap.add_argument("--group", type=int, default=8, help="group size of the flop model (the farm's G)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = _lib.load()
    torch = _lib.torch_cuda()
    model, chunks = synthetic.config_chunks(args.config)
    p = synthetic.default_params(model)
    norb = len(synthetic.ORBIT_PARAMS[model])
    ncomp = synthetic.NCOMP[model]
    amps, ls = list(p[norb::2][:ncomp]), list(p[norb + 1::2][:ncomp])
    lines = ["card: " + card(), "config %s, every %d-th chunk, flops for groups of %d" % (args.config, args.stride, args.group),
             "%-6s %5s %4s %9s %9s %7s %9s %9s  tend at group ends (device)" % (
                 "chunk", "N", "T", "dense GF", "exec GF", "ratio", "ms sorted", "ms epoch")]
    tot = [0.0, 0.0, 0.0, 0.0]
    for i in range(0, len(chunks), args.stride):
        ch = chunks[i]
        vel = synthetic.host_velocities(model, p[:norb], ch["date1D"])
        order, zs = envelope.sorted_chunk_z(ch, vel)
        fl, sg = np.asarray(ch["fl"])[order], np.asarray(ch["sigma"])[order]
        tend, ms_sorted, _ = run_chunk(lib, torch, zs, fl, sg, amps, ls, args.reps)
        zs_e = np.array([ch["lwl"] + (-np.asarray(v)[ch["epoch"]]) / synthetic.c_kms for v in vel])
        _, ms_epoch, _ = run_chunk(lib, torch, zs_e, ch["fl"], ch["sigma"], amps, ls, args.reps)
        T = len(tend) - 1
        dense = envelope.executed_flops(T, args.group)
        ex = envelope.executed_flops(T, args.group, tend)
        for k, v in enumerate((dense, ex, ms_sorted, ms_epoch)):
            tot[k] += v
        ends = envelope.group_starts(T, args.group)[1:]
        lines.append("%-6d %5d %4d %9.2f %9.2f %7.3f %9.3f %9.3f  %s" % (
            i, len(fl), T, dense / 1e9, ex / 1e9, dense / ex, ms_sorted, ms_epoch, " ".join(str(int(tend[e])) for e in ends)))
    lines.append("total: dense %.1f GF, executed %.1f GF (dense / executed %.3f); single-call time sorted %.2f ms, "
                 "epoch-major %.2f ms" % (tot[0] / 1e9, tot[1] / 1e9, tot[0] / tot[1], tot[2], tot[3]))
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
