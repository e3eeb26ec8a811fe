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


# Default (proposal, chunk) pairs in flight in the gradient graph (capped by nbranch).  Measured on a B200 (1000 W), C4,
# one proposal (tools/time_grad_farm.py): 16 / 32 / 64 branches 784 / 781 / 780 ms for 21.8 / 43.5 / 87.1 GB; the
# branches beyond 16 buy nothing the SMs could use, so 16, at half the memory of 32.
GRAD_NBRANCH = 16

# Default (proposal, chunk) items in flight in the prediction graph (capped by the number of items).  The gradient
# graph's default; the best value for prediction is not measured.
PREDICT_NBRANCH = 16


def prediction_grids(grids, n_pix, ncomp):
    """The per-chunk grids of ChunkFarm.attach_prediction_grids as [ncomp, m] float64 arrays: a 1-D entry serves every
    component, a 2-D one is [ncomp, m] (lwl_f_predict, lwl_g_predict[, lwl_h_predict] of predict_f_g / _f_g_h).
    n_pix: the number of pixels of every chunk, in global chunk order."""
    if len(grids) != len(n_pix):
        raise ValueError("one prediction grid per chunk: got %d grids for %d chunks" % (len(grids), len(n_pix)))
    out = []
    for i, (g, n) in enumerate(zip(grids, n_pix)):
        a = np.asarray(g, dtype=np.float64)
        if a.ndim == 1:
            a = np.broadcast_to(a, (ncomp, a.size))
        if a.ndim != 2 or a.shape[0] != ncomp:
            raise ValueError("chunk %d: a prediction grid is 1-D or [%d, m], not of shape %s" % (i, ncomp, np.shape(g)))
        if not np.all(np.isfinite(a)):
            raise ValueError("chunk %d: the prediction grid holds non-finite values" % i)
        if n == 0 and a.shape[1] != 0:
            raise ValueError("chunk %d has no pixels: its prediction grid must be empty" % i)
        out.append(np.ascontiguousarray(a))
    return out


def combine_predictions(mu, var):
    """Posterior-averaged spectrum and its variance over K samples by the law of total variance: mean of the variances
    plus the variance of the means.  mu, var: [K, M] (one chunk's outputs of predict_components, var the diagonal of
    Sigma).  Sums over the samples run in sample order."""
    mu, var = np.asarray(mu, dtype=np.float64), np.asarray(var, dtype=np.float64)
    K = mu.shape[0]
    mean = np.add.reduce(mu, axis=0) / K
    return mean, np.add.reduce(var, axis=0) / K + np.add.reduce((mu - mean) ** 2, axis=0) / K


class ChunkFarm:
    """model: "SB1" | "SB2" | "ST1" | "ST2" | "ST3".
    chunks: list of dicts with lwl, fl, sigma (masked 1-D), mask [n_epochs, n_pix] (or `epoch` int32 [N]) and
    date1D — the attributes a reference Chunk exposes after apply_mask() (data.py:120-147).
    rank/world_size: static partition of the chunks over GPUs; process_group: torch.distributed group (or None).
    grad_nbranch: (proposal, chunk) pairs in flight in the gradient graph of chunk_lnlike_grads_many (default
    GRAD_NBRANCH, at most nbranch); each branch holds the identity-bordered matrix of the largest chunk, 8 (2 N)^2 bytes.
    """

    def __init__(self, model, chunks, mu_GP=1.0, soften=1.0, nbranch=32, rank=0, world_size=1, process_group=None,
                 n_proposals=1, grad_nbranch=None):
        self.grad_nbranch = int(grad_nbranch) if grad_nbranch is not None else min(nbranch, GRAD_NBRANCH)
        if self.grad_nbranch < 1:
            raise ValueError("grad_nbranch must be at least 1")
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
            # pixels in wavelength order, epochs interleaved: the covariance is then exactly zero outside a narrow
            # envelope that the factorisation skips (DESIGN §9).  The likelihood and its parameter gradient do not
            # depend on the pixel order; every farm path reads these buffers, so all of them see the same order.
            order = np.argsort(host["lwl"], kind="stable")
            for k2 in ("lwl", "fl", "sigma", "epoch"):
                host[k2] = np.ascontiguousarray(host[k2][order])
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
        self._grad_farm_ws = None    # allocated, and the gradient graph attached, by the first *_many gradient call
        self._n_pix = [len(ch["fl"]) for ch in chunks]
        self._pred = None            # attach_prediction_grids
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

    def chunk_fishers(self, p):
        """Per-chunk expected Fisher information F_ab = 1/2 tr(K^-1 dK/dp_a K^-1 dK/dp_b) at the full registered vector p
        (orbital then GP): device tensor [n_chunks, n_params, n_params].  This rank's chunks go one at a time through
        psoap_chunk_fisher (each chunk's n_params products fill the GPU), each written at its global chunk index; the
        other entries are zero, and with world_size > 1 the tensor is all-reduced (exact: every entry has one
        contributor).  The workspace, (4 + n_params) 8 N^2 bytes for the largest own chunk, is allocated for the call
        and released after it.  A chunk's matrix is NaN where its lnlike is -inf."""
        lib = _lib.load()
        torch = _lib.torch_cuda()
        p = np.asarray(p, dtype=np.float64)
        if p.size != self.n_params:
            raise ValueError("p must hold the %d registered parameters of %s" % (self.n_params, self.model))
        npar = self.n_params
        out = torch.zeros((self.n_chunks, npar, npar), dtype=torch.float64, device="cuda")
        if self.mine:
            model = _lib.MODELS[self.model]
            nbytes = max(lib.psoap_chunk_fisher_workspace_bytes(model, N, ne) for N, ne in zip(self.Ns, self._n_epochs))
            try:
                ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            except torch.cuda.OutOfMemoryError as e:
                raise MemoryError("the Fisher information of the largest chunk needs %d bytes of device memory"
                                  % nbytes) from e
            p_dev = torch.from_numpy(p.reshape(-1).copy()).cuda()
            res = torch.empty(4, dtype=torch.float64, device="cuda")
            for k, idx in enumerate(self.mine):
                _lib.check(lib.psoap_chunk_fisher(model, ctypes.byref(self._descs[k]), _lib.ptr(p_dev), self.mu_GP,
                                                  _lib.ptr(ws), nbytes, _lib.ptr(res), None, _lib.ptr(out[idx]),
                                                  _lib.stream_ptr()))
        if self.world_size > 1:
            self._allreduce(out)
        return out

    def fisher(self, p):
        """Expected Fisher information of the farm's likelihood at p: ndarray [n_params, n_params], the per-chunk
        matrices of chunk_fishers summed in chunk order on the host (as lnprob_and_grad sums), so the bits do not
        depend on the number of GPUs.  Chunks are independent, so this is the Fisher information of the whole data."""
        return np.sum(self.chunk_fishers(p).cpu().numpy(), axis=0)

    def lnprob_many(self, P):
        """Ensemble evaluation (SURVEY.md §8f-2): P is [n_proposals, n_params]; one graph launch evaluates every
        (proposal, chunk) pair; returns the n_proposals summed log-likelihoods."""
        return np.atleast_1d(self.lnprob(P))

    def _attach_grad_graph(self):
        lib = _lib.load()
        torch = _lib.torch_cuda()
        nbytes = lib.psoap_farm_grad_workspace_bytes(self._farm, self.grad_nbranch)
        try:
            ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
        except torch.cuda.OutOfMemoryError as e:
            raise MemoryError("the gradient graph needs %d bytes of device memory for grad_nbranch = %d (one "
                              "identity-bordered matrix of the largest chunk per branch); pass a smaller grad_nbranch"
                              % (nbytes, self.grad_nbranch)) from e
        _lib.check(lib.psoap_farm_grad_attach(self._farm, self.grad_nbranch, _lib.ptr(ws), nbytes))
        self._grad_farm_ws = ws

    def chunk_lnlike_grads_many(self, P):
        """Per-(proposal, chunk) (lnlike, gradient) rows for the n_proposals registered vectors P ([n_proposals,
        n_params]): device tensor [n_proposals, n_chunks, n_params + 1].  One launch of the farm's gradient graph
        evaluates every (proposal, chunk) pair of this rank, grad_nbranch of them in flight; the rows go at their
        global chunk index, the other rows are zero, and with world_size > 1 the tensor is all-reduced (exact: every
        row has one contributor).  The first call allocates the graph's workspace and captures it; a farm that never
        asks for it holds neither.  Gradient rows are NaN where lnlike is -inf."""
        lib = _lib.load()
        torch = _lib.torch_cuda()
        P = np.asarray(P, dtype=np.float64)
        K, npar = self.n_proposals, self.n_params
        if P.size != K * npar:
            raise ValueError("P must hold %d x %d registered parameters of %s" % (K, npar, self.model))
        rows = torch.zeros((K, self.n_chunks, npar + 1), dtype=torch.float64, device="cuda")
        if self.mine:
            if self._grad_farm_ws is None:
                self._attach_grad_graph()
            p_dev = torch.from_numpy(np.ascontiguousarray(P.reshape(K, npar))).cuda()
            res = torch.empty((K, len(self.mine), 4), dtype=torch.float64, device="cuda")
            grad = torch.empty((K, len(self.mine), npar), dtype=torch.float64, device="cuda")
            _lib.check(lib.psoap_farm_lnprob_grad(self._farm, _lib.ptr(p_dev), _lib.ptr(res), _lib.ptr(grad),
                                                  _lib.stream_ptr()))
            rows.index_copy_(1, self._mine_idx, torch.cat([res[:, :, :1], grad], dim=2))
        if self.world_size > 1:
            self._allreduce(rows)
        return rows

    def lnprob_and_grad_many(self, P):
        """lnprob and its gradient for each of the n_proposals vectors P: (ndarray [n_proposals], ndarray
        [n_proposals, n_params]).  Each proposal's rows are summed in chunk order on the host as lnprob_and_grad
        sums them, so the bits do not depend on the number of GPUs."""
        h = self.chunk_lnlike_grads_many(P).cpu().numpy()
        lnp = np.array([float(np.sum(hk[:, 0])) for hk in h])
        return lnp, np.stack([np.sum(hk[:, 1:], axis=0) for hk in h])

    def attach_prediction_grids(self, grids, sigma="full", predict_nbranch=None):
        """Attach the prediction graph (psoap_farm_predict_attach) for predict_components: grids holds one entry per
        chunk in global chunk order, a 1-D rest-frame ln-wavelength grid used for every component or an [ncomp, m]
        array (lwl_f_predict, lwl_g_predict[, lwl_h_predict] of predict_f_g / _f_g_h); a chunk without pixels takes an
        empty grid.  sigma: "full" (Sigma) or "diag" (its diagonal).  predict_nbranch: (proposal, chunk) items in
        flight (default PREDICT_NBRANCH); each branch holds the bordered matrix of the largest item,
        8 (padded(N) + padded(ncomp m))^2 bytes.  The grids are uploaded once; a farm that never calls this allocates
        and captures nothing for prediction."""
        if self._pred is not None:
            raise RuntimeError("the prediction grids are already attached to this farm")
        if sigma not in ("full", "diag"):
            raise ValueError('sigma must be "full" or "diag", not %r' % (sigma,))
        nb = int(predict_nbranch) if predict_nbranch is not None else PREDICT_NBRANCH
        if nb < 1:
            raise ValueError("predict_nbranch must be at least 1")
        ncomp = _lib.NCOMP[self.model]
        gr = prediction_grids(grids, self._n_pix, ncomp)
        lib = _lib.load()
        torch = _lib.torch_cuda()
        K, mode = self.n_proposals, (0 if sigma == "full" else 1)
        m_all = [g.shape[1] for g in gr]
        M_all = [ncomp * m for m in m_all]
        size = [M * M if mode == 0 else M for M in M_all]
        # the outputs of all chunks in one flat buffer per kind, chunk after chunk and each chunk's proposals side by
        # side: the layout psoap_farm_predict_attach returns for a farm that holds every chunk
        d0 = np.concatenate([[0], np.cumsum([K * M for M in M_all])]).astype(np.int64)
        s0 = np.concatenate([[0], np.cumsum([K * x for x in size])]).astype(np.int64)
        pred = dict(mode=mode, m=m_all, M=M_all, d0=d0, s0=s0, ws=None, grids=None, off=None)
        if self.mine:
            total, offs = 0, []
            for i in self.mine:
                offs.append(total)
                total += (gr[i].nbytes + 255) // 256 * 256
            gdev = torch.empty(max(total, 256), dtype=torch.uint8, device="cuda")
            host = np.zeros(max(total, 256), dtype=np.uint8)
            for i, o in zip(self.mine, offs):
                host[o:o + gr[i].nbytes] = gr[i].view(np.uint8).reshape(-1)
            gdev.copy_(torch.from_numpy(host))
            base = gdev.data_ptr()
            ptrs = (_lib.vp * (len(self.mine) * ncomp))(
                *[_lib.vp(base + o + c * m_all[i] * 8) for i, o in zip(self.mine, offs) for c in range(ncomp)])
            m_mine = (ctypes.c_int64 * len(self.mine))(*[m_all[i] for i in self.mine])
            nbytes = lib.psoap_farm_predict_workspace_bytes(self._farm, nb, m_mine, mode)
            try:
                ws = torch.empty(nbytes + 256, dtype=torch.uint8, device="cuda")
            except torch.cuda.OutOfMemoryError as e:
                raise MemoryError("the prediction graph needs %d bytes of device memory for predict_nbranch = %d (one "
                                  "bordered matrix of the largest item per branch); pass a smaller predict_nbranch"
                                  % (nbytes, nb)) from e
            nitems = K * len(self.mine)
            off = (ctypes.c_int64 * (2 * (nitems + 1)))()
            _lib.check(lib.psoap_farm_predict_attach(self._farm, nb, m_mine, ptrs, mode, _lib.ptr(ws), nbytes, off))
            off = np.frombuffer(off, dtype=np.int64).reshape(2, nitems + 1).copy()
            pred.update(ws=ws, grids=gdev, off=off)
        self._pred = pred

    def predict_components(self, P, mus):
        """The component spectra of every chunk at the n_proposals registered vectors P ([n_proposals, n_params]), as
        predict_f_g / predict_f_g_h compute them from the chunk's pixels shifted by each proposal's velocities, with one
        launch of the prediction graph (attach_prediction_grids first).  mus: the ncomp component means (mu_f, mu_g[,
        mu_h]).  Returns, per chunk in global chunk order, (mu [n_proposals, ncomp m], Sigma [n_proposals, M, M]) or,
        with sigma="diag", (mu, var [n_proposals, M]), M = ncomp m, as device tensors.  Each rank fills its own chunks
        into one flat buffer per kind, which is all-reduced once (exact: every entry has one contributor).  Raises
        numpy.linalg.LinAlgError for an item whose data block is not positive definite and ValueError for one whose
        velocities reach c or whose GP parameters are negative, naming the proposal and the chunk."""
        ncomp = _lib.NCOMP[self.model]
        K, npar = self.n_proposals, self.n_params
        P = np.asarray(P, dtype=np.float64)
        if P.size != K * npar:
            raise ValueError("P must hold %d x %d registered parameters of %s" % (K, npar, self.model))
        mus = np.asarray(mus, dtype=np.float64).reshape(-1)
        if mus.size != ncomp:
            raise ValueError("mus must hold the %d component means of %s" % (ncomp, self.model))
        if self._pred is None:
            raise RuntimeError("attach_prediction_grids must be called before predict_components")
        q = self._pred
        lib = _lib.load()
        torch = _lib.torch_cuda()
        delta = torch.zeros(int(q["d0"][-1]), dtype=torch.float64, device="cuda")
        sig = torch.zeros(int(q["s0"][-1]), dtype=torch.float64, device="cuda")
        res = torch.zeros((K, self.n_chunks, 4), dtype=torch.float64, device="cuda")
        if self.mine:
            off = q["off"]
            n_mine = len(self.mine)
            p_dev = torch.from_numpy(np.ascontiguousarray(P.reshape(K, npar))).cuda()
            dl = torch.empty(max(1, int(off[0, -1])), dtype=torch.float64, device="cuda")
            sl = torch.empty(max(1, int(off[1, -1])), dtype=torch.float64, device="cuda")
            rl = torch.empty((K, n_mine, 4), dtype=torch.float64, device="cuda")
            _lib.check(lib.psoap_farm_predict(self._farm, _lib.ptr(p_dev), _lib.ptr(dl), _lib.ptr(sl), _lib.ptr(rl),
                                              _lib.stream_ptr()))
            # each own chunk's proposals are contiguous in the attach layout: one copy per chunk and kind
            for k, i in enumerate(self.mine):
                nd, ns = K * q["M"][i], int(q["s0"][i + 1] - q["s0"][i])
                delta[q["d0"][i]:q["d0"][i] + nd].copy_(dl[off[0, k]:off[0, k] + nd])
                sig[q["s0"][i]:q["s0"][i] + ns].copy_(sl[off[1, k]:off[1, k] + ns])
            res.index_copy_(1, self._mine_idx, rl)
        if self.world_size > 1:
            self._allreduce(delta)
            self._allreduce(sig)
            self._allreduce(res)
        h = res.cpu().numpy()
        for k in range(K):
            for i in range(self.n_chunks):
                if q["m"][i] == 0:
                    continue
                if h[k, i, 3] != 0.0:
                    raise np.linalg.LinAlgError("proposal %d, chunk %d: %d-th leading minor of the data block is not "
                                                "positive definite" % (k, i, int(h[k, i, 3])))
                if h[k, i, 0] == -np.inf:
                    raise ValueError("proposal %d, chunk %d: a velocity reaches the speed of light or a GP parameter is "
                                     "negative" % (k, i))
        out = []
        for i in range(self.n_chunks):
            M, m = q["M"][i], q["m"][i]
            mu = delta[q["d0"][i]:q["d0"][i + 1]].view(K, M) + torch.from_numpy(np.repeat(mus, m)).cuda()
            s = sig[q["s0"][i]:q["s0"][i + 1]]
            out.append((mu, s.view(K, M, M) if q["mode"] == 0 else s.view(K, M)))
        return out

    def close(self):
        if self._farm:
            _lib.load().psoap_farm_destroy(self._farm)
            self._farm = _lib.vp(None)
        self._grad_farm_ws = None
        self._pred = None

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
