"""ChunkFarm — the B200 replacement of the reference's multiprocessing chunk farm
(psoap/sample_parallel.py: Worker.initialize :126-166, Worker.lnprob :168-198, master lnprob :371-390).

The reference forks one process per chunk; each keeps its chunk resident and, per proposal, receives the
parameter vector over a Pipe and sends one float back; the master np.sum()s them.  Here every rank (one process
per GPU) owns a static subset of the chunks (longest-processing-time partition by N^3), keeps them resident in
HBM, and evaluates all of them with ONE CUDA-graph launch: orbit velocities -> Doppler-shifted covariance fill
-> blocked FP64 Cholesky with fused solve/logdet, several chunks in flight on independent graph branches.
Per proposal only the parameter vector goes down and one record per chunk comes back.  Across ranks the
per-chunk log-likelihoods are combined with a single all-reduce of a length-n_chunks FP64 vector (own entries
filled, others zero: exact and order independent), then summed in chunk order like the reference's np.sum.
"""
import ctypes

import numpy as np

from . import _lib
from .data import epoch_index


def lpt_partition(costs, nparts):
    """Longest-processing-time-first partition: returns a list of index lists, deterministic."""
    order = sorted(range(len(costs)), key=lambda i: (-costs[i], i))
    loads = [0.0] * nparts
    parts = [[] for _ in range(nparts)]
    for i in order:
        b = min(range(nparts), key=lambda k: (loads[k], k))
        parts[b].append(i)
        loads[b] += costs[i]
    return parts


# Cost model of one chunk for the static partition, in units of N^3: the O(N^3) trailing updates, the O(N^2) fill and
# panel solves, and the O(N) chain of dependent diagonal blocks (N / 128 panels, each a potrf + trsm + column update
# that cannot use more than a few SMs).  ALPHA2 / ALPHA1 are fitted to the measured farm throughput of uniform-size
# farms on a B200 (tools/farm_cost_fit.py, profiles/README.md "cost model"); only their ratio to the cubic term matters.
# Round-2 fit (64 equal chunks, 32 branches, N = 1600 .. 6000): t(N) = 9.96e-15 N^3 - 2.6e-13 N^2 + 1.76e-8 N seconds:
# the quadratic term is nil, the linear one is 44 % of the cubic at N = 2000 and 5 % at N = 6000.
ALPHA2 = 0.0        # t(N) ~ N^3 + ALPHA2 N^2 + ALPHA1 N
ALPHA1 = 1.77e6


def chunk_cost(N):
    n = float(N)
    return n ** 3 + ALPHA2 * n * n + ALPHA1 * n


class ChunkFarm:
    """model: "SB1" | "SB2" | "ST1" | "ST2" | "ST3".
    chunks: list of dicts with lwl, fl, sigma (masked 1-D), mask [n_epochs, n_pix] (or `epoch` int32 [N]) and
    date1D — the attributes a reference Chunk exposes after apply_mask() (data.py:120-147).
    rank/world_size: static partition of the chunks over GPUs; process_group: torch.distributed group (or None).
    """

    def __init__(self, model, chunks, mu_GP=1.0, soften=1.0, nbranch=32, rank=0, world_size=1, process_group=None,
                 n_proposals=1):
        lib = _lib.load()
        torch = _lib.torch_cuda()
        self.model = model
        self.n_proposals = int(n_proposals)
        self.n_chunks = len(chunks)
        self.n_params = _lib.N_ORB[model] + 2 * _lib.NCOMP[model]
        self.rank, self.world_size, self.group = rank, world_size, process_group
        self.parts = lpt_partition([chunk_cost(len(ch["fl"])) for ch in chunks], world_size)
        # a chunk whose mask removed every pixel contributes -0.0 in the reference (sums over nothing): it takes no
        # device work here and its entry of the per-chunk vector stays 0
        self.mine = [i for i in sorted(self.parts[rank]) if len(chunks[i]["fl"]) > 0]
        self._cost_mine = float(sum(chunk_cost(len(chunks[i]["fl"])) for i in self.parts[rank]))
        # every chunk vector lives in ONE pinned host buffer and ONE device buffer (256-byte aligned slices), so a
        # refresh of the resident data is a single host->device copy
        hosts, offsets, total = [], [], 0
        for idx in self.mine:
            ch = chunks[idx]
            ep = ch["epoch"] if "epoch" in ch else epoch_index(ch["mask"])
            host = dict(lwl=np.ascontiguousarray(ch["lwl"], dtype=np.float64),
                        fl=np.ascontiguousarray(ch["fl"], dtype=np.float64),
                        sigma=np.ascontiguousarray(np.asarray(ch["sigma"], dtype=np.float64) * soften),
                        dates=np.ascontiguousarray(ch["date1D"], dtype=np.float64),
                        epoch=np.ascontiguousarray(ep, dtype=np.int32))
            N = len(host["fl"])
            if not (len(host["lwl"]) == len(host["sigma"]) == len(host["epoch"]) == N):
                raise ValueError("chunk %d: lwl, fl, sigma and the mask must select the same number of pixels" % idx)
            # the device reads vel[c * n_epochs + epoch[i]]: an index outside date1D would be an out-of-bounds read
            # (the reference raises a broadcasting error for a mask that does not match date1D, data.py:61)
            if "mask" in ch and np.asarray(ch["mask"]).shape[0] != len(host["dates"]):
                raise ValueError("chunk %d: the mask has %d rows but date1D has %d epochs"
                                 % (idx, np.asarray(ch["mask"]).shape[0], len(host["dates"])))
            if N and (host["epoch"].min() < 0 or host["epoch"].max() >= len(host["dates"])):
                raise ValueError("chunk %d: epoch indices must lie in [0, %d)" % (idx, len(host["dates"])))
            off = {}
            for k2, v in host.items():
                off[k2] = total
                total += (v.nbytes + 255) // 256 * 256
            hosts.append(host)
            offsets.append(off)
        self._host_buf = torch.empty(max(total, 256), dtype=torch.uint8).pin_memory()
        self._dev_buf = torch.empty(max(total, 256), dtype=torch.uint8, device="cuda")
        hb = self._host_buf.numpy()
        descs = (_lib.PsoapChunk * max(1, len(self.mine)))()
        Ns, nes = [], []
        base = self._dev_buf.data_ptr()
        for k, (host, off) in enumerate(zip(hosts, offsets)):
            for k2, v in host.items():
                hb[off[k2]:off[k2] + v.nbytes] = v.view(np.uint8).reshape(-1)
            d = descs[k]
            # chain links chosen from the GLOBAL problem, not from this rank's share: fewer than 8 (proposal, chunk) pairs
            # in all -> the latency chain (7), else the throughput chain (3); same bits on 1, 2, 4 or 8 GPUs
            # ... and the panels per trailing update likewise: rank-1024 updates (8) when there are at least 64 pairs to
            # hide their long heads behind, else rank-512 (4)
            n_pairs = self.n_chunks * self.n_proposals
            chain = 7 if n_pairs < 8 else 3
            group = 8 if n_pairs >= 64 else 4
            d.reserved = chain | (group << 8)
            d.N, d.n_epochs = len(host["fl"]), len(host["dates"])
            d.lwl, d.epoch, d.fl = base + off["lwl"], base + off["epoch"], base + off["fl"]
            d.sigma, d.dates = base + off["sigma"], base + off["dates"]
            Ns.append(d.N)
            nes.append(d.n_epochs)
        self._data_bytes = total
        self._dev_buf.copy_(self._host_buf, non_blocking=True)
        torch.cuda.synchronize()
        self.Ns = Ns
        self.mu_GP = float(mu_GP)
        self._descs = descs          # kept for the gradient entry, which takes one chunk at a time
        self._n_epochs = nes
        self._grad_ws = None         # allocated by the first lnprob_and_grad call
        self._farm = _lib.vp(None)
        K = self.n_proposals
        self._results = torch.zeros((K, max(1, len(self.mine)), 4), dtype=torch.float64, device="cuda")
        self._p_dev = torch.zeros((K, self.n_params), dtype=torch.float64, device="cuda")
        self._p_pin = torch.zeros((K, self.n_params), dtype=torch.float64).pin_memory()
        self._p_event = None
        self._lnl_all = torch.zeros((K, self.n_chunks), dtype=torch.float64, device="cuda")
        self._lnl_pin = torch.zeros((K, self.n_chunks), dtype=torch.float64).pin_memory()
        self._mine_idx = torch.tensor(self.mine, dtype=torch.int64, device="cuda")
        self.launches_per_eval = 0
        if self.mine:
            nb = max(1, min(nbranch, len(self.mine) * K))
            nbytes = lib.psoap_farm_workspace_bytes_batched(len(self.mine), (ctypes.c_int64 * len(Ns))(*Ns),
                                                            (ctypes.c_int32 * len(nes))(*nes), K, nb)
            self._ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
            _lib.check(lib.psoap_farm_create_batched(ctypes.byref(self._farm), _lib.MODELS[model], len(self.mine),
                                                     descs, K, nb, float(mu_GP), _lib.ptr(self._ws), nbytes))
            self.launches_per_eval = lib.psoap_farm_launches_per_eval(self._farm)

    # -- per-rank work --------------------------------------------------------------------------------
    def cost_of_mine(self):
        """This rank's load under the partition's cost model (bench.py reports max / mean over ranks)."""
        return self._cost_mine

    def flops_per_eval(self):
        """Algorithmic flops of this rank's chunks: N^3/3 + 2 N^2 each (SURVEY.md §8d)."""
        return float(sum(n ** 3 / 3.0 + 2.0 * n ** 2 for n in self.Ns))

    def refresh_data(self):
        """Re-upload this rank's chunk vectors from pinned host memory (bench.py's e2e leg): one async copy."""
        self._dev_buf.copy_(self._host_buf, non_blocking=True)
        return self._data_bytes

    def lnprob_device(self, p_dev):
        """Evaluate this rank's chunks for the device parameter vector(s) p_dev ([n_params], or
        [n_proposals, n_params]; full registered vector, orbital then GP, utils.py:4-8).  Asynchronous; returns the
        [n_proposals, n_mine, 4] result tensor (lnlike, logdet, quad, info)."""
        if self.mine:
            _lib.check(_lib.load().psoap_farm_lnprob(self._farm, _lib.ptr(p_dev), _lib.ptr(self._results),
                                                     _lib.stream_ptr()))
        return self._results

    def chunk_lnlikes_device(self, p_dev):
        """All chunks' log-likelihoods for DEVICE parameter vector(s), as a device tensor [n_proposals, n_chunks]
        ([n_chunks] when n_proposals == 1); asynchronous (no host synchronisation).  With world_size > 1 it ends
        with the one collective of the path."""
        res = self.lnprob_device(p_dev)
        self._lnl_all.zero_()
        if self.mine:
            self._lnl_all.index_copy_(1, self._mine_idx, res[:, :len(self.mine), 0])
        if self.world_size > 1:
            self._allreduce(self._lnl_all)
        return self._lnl_all[0] if self.n_proposals == 1 else self._lnl_all

    def chunk_lnlikes(self, p):
        """Same for HOST parameter vector(s) p (staged through pinned memory)."""
        torch = _lib.torch_cuda()
        p = np.asarray(p, dtype=np.float64).reshape(-1, self.n_params) if np.size(p) == self.n_proposals * self.n_params \
            else None
        if p is None:
            raise ValueError("p must hold %d x %d registered parameters of %s"
                             % (self.n_proposals, self.n_params, self.model))
        # the previous call's asynchronous upload may still be reading the pinned staging buffer
        if self._p_event is not None:
            self._p_event.synchronize()
        self._p_pin.copy_(torch.from_numpy(np.ascontiguousarray(p)))
        self._p_dev.copy_(self._p_pin, non_blocking=True)
        if self._p_event is None:
            self._p_event = torch.cuda.Event()
        self._p_event.record()
        return self.chunk_lnlikes_device(self._p_dev)

    def _allreduce(self, t):
        import torch.distributed as dist
        # -inf entries are legal values here; SUM keeps them (-inf + 0 = -inf) exactly like np.sum does
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def lnprob(self, p):
        """sample_parallel.py:371-390 without the prior: sum over chunks, in chunk order, of the per-chunk lnlike."""
        lnl = self.chunk_lnlikes(p)
        self._lnl_pin.copy_(self._lnl_all, non_blocking=False)
        sums = np.sum(self._lnl_pin.numpy(), axis=1)
        return float(sums[0]) if self.n_proposals == 1 else sums

    def chunk_lnlike_grads(self, p):
        """Per-chunk (lnlike, gradient) rows for the full registered vector p (orbital then GP, utils.py:4-8): device
        tensor [n_chunks, n_params + 1].  This rank's chunks go one at a time through psoap_chunk_lnprob_grad, each
        writing its row at its global chunk index; the other rows are zero, and with world_size > 1 the tensor is
        all-reduced (exact: every row has one contributor).  The first call allocates one workspace for the largest
        own chunk; a farm that never asks for a gradient holds none.  Gradient rows are NaN where lnlike is -inf."""
        lib = _lib.load()
        torch = _lib.torch_cuda()
        p = np.asarray(p, dtype=np.float64)
        if p.size != self.n_params:
            raise ValueError("p must hold the %d registered parameters of %s" % (self.n_params, self.model))
        npar = self.n_params
        rows = torch.zeros((self.n_chunks, npar + 1), dtype=torch.float64, device="cuda")
        if self.mine:
            model = _lib.MODELS[self.model]
            if self._grad_ws is None:
                need = max(lib.psoap_chunk_lnprob_grad_workspace_bytes(model, N, ne)
                           for N, ne in zip(self.Ns, self._n_epochs))
                self._grad_ws = (torch.empty(need + 256, dtype=torch.uint8, device="cuda"), need)
            ws, nbytes = self._grad_ws
            p_dev = torch.from_numpy(p.reshape(-1).copy()).cuda()
            res = torch.empty((len(self.mine), 4), dtype=torch.float64, device="cuda")
            base, stride = rows.data_ptr(), (npar + 1) * 8
            for k, idx in enumerate(self.mine):
                _lib.check(lib.psoap_chunk_lnprob_grad(model, ctypes.byref(self._descs[k]), _lib.ptr(p_dev),
                                                       self.mu_GP, _lib.ptr(ws), nbytes, _lib.ptr(res[k]),
                                                       _lib.vp(base + idx * stride + 8), _lib.stream_ptr()))
            rows[:, 0].index_copy_(0, self._mine_idx, res[:, 0])
        if self.world_size > 1:
            self._allreduce(rows)
        return rows

    def lnprob_and_grad(self, p):
        """lnprob(p) and its gradient with respect to p: (float, ndarray [n_params]).  The per-chunk rows of
        chunk_lnlike_grads are summed in chunk order on the host, so the bits do not depend on the number of GPUs."""
        h = self.chunk_lnlike_grads(p).cpu().numpy()
        return float(np.sum(h[:, 0])), np.sum(h[:, 1:], axis=0)

    def lnprob_many(self, P):
        """Ensemble evaluation (SURVEY.md §8f-2): P is [n_proposals, n_params]; one graph launch evaluates every
        (proposal, chunk) pair; returns the n_proposals summed log-likelihoods."""
        return np.atleast_1d(self.lnprob(P))

    def close(self):
        if self._farm:
            _lib.load().psoap_farm_destroy(self._farm)
            self._farm = _lib.vp(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def combine_chunk_lnlikes(per_rank_vectors):
    """Host-side statement of the cross-rank reduction (used by the gloo tests): element-wise sum of vectors
    that are zero outside each rank's own chunks, then np.sum in chunk order."""
    total = np.zeros_like(per_rank_vectors[0])
    for v in per_rank_vectors:
        total = total + v
    return float(np.sum(total)), total
