"""Row/column sharding of the alternating sweep across the GPUs of one box.

The reference has no distributed code; its per-row updates within a half-sweep are
independent (/root/reference/src/poismf.c:159-187, :296-321, :352-397: every row reads its
own CSR/CSC slice, the FULL opposite factor matrix and the k column sums, and writes its
own k numbers).  So:

  * users are split into contiguous CSR row ranges balanced by (cost-weighted) non-zeros, items
    into contiguous CSC column ranges likewise; rank r holds its two slices,
  * A and B are replicated on every rank,
  * after the B half-sweep every rank's freshly updated rows of B are exchanged
    (one exchange step per half-sweep), likewise A after the A half-sweep,
  * the column sums are recomputed locally from the replicated matrix (deterministic
    order, no collective), and tncg's early-stop count is summed over ranks.

One process per GPU (torchrun); torch.distributed is the plumbing (NCCL on GPUs, gloo in
the CPU tests, where the row solver is stood in by a caller-supplied function).
"""
from __future__ import annotations

import os

import numpy as np


def row_cost(nnz_per_row):
    """Relative device cost of solving a row with n non-zeros (measured on B200, r1 bins of config #2):
    ~10 non-zero-equivalents of fixed work per row, and non-zeros of long rows cost more — rows beyond
    one CTA's shared memory pay cluster barriers (x2), rows streamed from L2 more again (x3)."""
    n = np.asarray(nnz_per_row).astype(np.float64)
    spec = os.environ.get("POISMF_B200_ROW_COST")      # tuning: "fixed,b1:f1,b2:f2,..." = fixed + n * f_i for n > b_i
    if spec:
        parts = spec.split(",")
        c = n + float(parts[0])
        for item in parts[1:]:
            b, f = item.split(":")
            c += n * ((n > float(b)) * float(f))       # f = the factor ADDED above the break
        c[n <= 0] = 0.0
        return c
    c = n + 10.0                        # (in-place arithmetic: this runs inside every sharded load)
    c += n * (n > 1000)
    c += n * (n > 16000)
    c[n <= 0] = 0.0
    return c


def nnz_balanced_ranges(indptr, nparts, cost_aware=True):
    """Split rows 0..n into `nparts` contiguous ranges of ~equal work.

    Work is the non-zero count, or with `cost_aware` the device cost model of `row_cost` (power-law
    matrices put a few very long rows somewhere; their non-zeros are dearer than a short row's).
    Returns a list of (begin, end); ranges may be empty when nparts > rows."""
    indptr = np.asarray(indptr).astype(np.int64)
    n = indptr.shape[0] - 1
    if cost_aware:
        cum = np.zeros(n + 1)
        np.cumsum(row_cost(np.diff(indptr)), out=cum[1:])
    else:
        cum = (indptr - indptr[0]).astype(np.float64)
    total = float(cum[-1])
    cuts = [0]
    for p in range(1, nparts):
        target = total * p / nparts
        c = int(np.searchsorted(cum, target, side="left"))
        c = min(max(c, cuts[-1]), n)
        cuts.append(c)
    cuts.append(n)
    return [(cuts[i], cuts[i + 1]) for i in range(nparts)]


def slice_compressed(mat, begin, end):
    """Rows [begin, end) of a (values, indptr, indices) triple, indptr rebased to 0."""
    vals, ptr, ind = mat
    lo, hi = int(ptr[begin]), int(ptr[end])
    return (np.ascontiguousarray(vals[lo:hi]),
            np.ascontiguousarray(ptr[begin:end + 1] - ptr[begin]).astype(ptr.dtype),
            np.ascontiguousarray(ind[lo:hi]))


class ShardedSweep:
    """Drives sharded alternating sweeps; mirrors run_poismf's outer loop (src/poismf.c:506-608).

    backend: an object with
        half_sweep(side, params, step, cnst_div) -> n_unchanged   (updates the LOCAL rows in place)
        exchange(side)                                             (refresh the replicated matrix)
    `GpuBackend` below is the product one; tests inject a CPU stand-in.
    """

    def __init__(self, backend, dimA, dimB, dtype, world_allreduce_int=None):
        self.be = backend
        self.dimA, self.dimB = dimA, dimB
        self.dtype = np.dtype(dtype)
        # tncg's early stop compares the number of unchanged rows of the WHOLE matrix with its dimension
        # (src/poismf.c:393-403): the local counts are summed over ranks
        self.allreduce_int = world_allreduce_int or getattr(backend, "allreduce_int", None) or (lambda v: v)

    def run(self, params):
        from . import _lib
        real = self.dtype.type
        step = real(params.step_size)
        l2 = real(params.l2_reg)
        stopA = stopB = False
        is_tncg = params.method == _lib.METHODS["tncg"]
        is_pg = params.method == _lib.METHODS["pg"]
        for _ in range(params.numiter):
            cdiv = float(real(1. / (1. + 2. * float(l2) * float(step))))
            if not (is_tncg and stopB):
                n = self.be.half_sweep(_lib.SIDE_CSC, params, float(step), cdiv)
                self.be.exchange(_lib.SIDE_CSC)
                if is_tncg and params.early_stop:
                    stopB = (self.allreduce_int(n) / self.dimB) >= .95
            if is_pg:
                step = real(float(step) * 0.5)
            if not (is_tncg and stopA):
                n = self.be.half_sweep(_lib.SIDE_CSR, params, float(step), cdiv)
                self.be.exchange(_lib.SIDE_CSR)
                if is_tncg and params.early_stop:
                    stopA = (self.allreduce_int(n) / self.dimA) >= .95
            if stopA and stopB:
                break


class GpuBackend:
    """One rank's shard on one GPU.

    exchange="p2p"  (default): the handle owns the replicas of A and B; their CUDA IPC handles are
        all-gathered once, and from then on the row kernels store every solved row directly into
        all peers' replicas over NVLink (fused compute + exchange, include/poismf_b200.h).
        Completion is signalled on the device (epoch slots in peer memory, a one-warp wait kernel
        ahead of the next half-sweep): nothing is left for the host between half-sweeps, whole fits
        are enqueued asynchronously.  `exchange="p2p-host"` keeps the r1 behaviour (stream sync +
        process barrier after every half-sweep).
    exchange="nccl": replicas are torch tensors bound into the handle; after each half-sweep the
        owners' rows are broadcast in place (one NCCL broadcast per owner).
    """

    def __init__(self, csr, csc, A0, B0, rank, world, device_index, group=None, exchange="p2p"):
        import torch
        import torch.distributed as dist
        from .device import DeviceFit
        from . import _lib
        self.torch, self.dist, self.group = torch, dist, group
        self.rank, self.world = rank, world
        self.mode = exchange if world > 1 else "local"
        dimA, k = A0.shape
        dimB = B0.shape[0]
        self.k = k
        self.dev = torch.device("cuda", device_index)
        self.fit = DeviceFit(dimA, dimB, k, A0.dtype, device=device_index)
        ldf = self.fit.ldf
        self.stream = torch.cuda.current_stream(self.dev)
        self.fit.set_stream(self.stream.cuda_stream)
        if self.mode == "nccl":
            tdt = torch.float32 if A0.dtype == np.float32 else torch.float64
            self.A = torch.zeros((dimA, ldf), dtype=tdt, device=self.dev)
            self.B = torch.zeros((dimB, ldf), dtype=tdt, device=self.dev)
            self.fit.bind_factors(self.A.data_ptr(), self.B.data_ptr())
        if self.mode in ("p2p", "p2p-host"):
            for which in ((0, 1, 2) if self.mode == "p2p" else (0, 1)):
                mine = self.fit.ipc_export(which)
                allh = [None] * world
                dist.all_gather_object(allh, mine, group=group)
                self.fit.ipc_import(which, allh, rank)
        self.load(csr, csc, A0, B0)

    def load(self, csr, csc, A0, B0):
        """(Re-)upload this rank's row / column shard and the replicated factors from host memory; the
        handle, its peer mappings and the epoch slots persist (a second fit on the same backend)."""
        from . import _lib
        self.finish()
        world, rank = self.world, self.rank
        if csr is None or csc is None:      # factors only (ranking with a model fitted elsewhere)
            self.rangesA = self.rangesB = None
            self.local_nnz = 0
            self._set_factors(A0, B0)
            return
        self.rangesA = self._ranges(csr[1])
        self.rangesB = self._ranges(csc[1])
        a0, a1 = self.rangesA[rank]
        b0, b1 = self.rangesB[rank]
        lr = slice_compressed(csr, a0, a1)
        lc = slice_compressed(csc, b0, b1)
        self.local_nnz = int(lr[0].shape[0])
        self.fit.set_matrix(_lib.SIDE_CSR, *lr, row_begin=a0, n_rows=a1 - a0)
        self.fit.set_matrix(_lib.SIDE_CSC, *lc, row_begin=b0, n_rows=b1 - b0)
        self._set_factors(A0, B0)

    def _ranges(self, indptr):
        """Shard boundaries of one side, remembered per offsets array (address, length, a strided sample of
        its content) — a refit on the same matrix skips the cost model's passes over every row."""
        indptr = np.asarray(indptr)
        step = max(1, indptr.shape[0] // 1024)
        key = (indptr.__array_interface__["data"][0], indptr.shape[0], indptr.dtype.str, self.world,
               indptr[::step].tobytes(), int(indptr[-1]))
        cache = self.__dict__.setdefault("_ranges_cache", {})
        if key not in cache:
            if len(cache) > 8:
                cache.clear()
            cache[key] = nnz_balanced_ranges(indptr, self.world)
        return cache[key]

    def _set_factors(self, A0, B0):
        if self.mode == "nccl":
            self.A[:, :self.k].copy_(self.torch.from_numpy(A0))
            self.B[:, :self.k].copy_(self.torch.from_numpy(B0))
        elif self.mode in ("p2p", "p2p-host"):
            # every rank uploads 1/N of the rows and stores them into all replicas over NVLink: each factor
            # row crosses PCIe once per box, not once per GPU
            for which, M in ((0, A0), (1, B0)):
                lo, hi = user_ranges(M.shape[0], self.world)[self.rank]
                self.fit.set_factor_rows(which, np.ascontiguousarray(M[lo:hi]), lo)
        else:
            self.fit.set_factors(A0, B0)
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier(group=self.group)

    def reset(self, A0, B0):
        """Restore the initial factors on this rank's replica (bench warm-up)."""
        self.finish()           # nobody may still be storing rows into this replica
        self._set_factors(A0, B0)

    def half_sweep(self, side, params, step, cdiv):
        return self.fit.half_sweep(side, params, step, cdiv)

    def allreduce_int(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([int(v)], dtype=self.torch.int64, device=self.dev)
        self.dist.all_reduce(t, group=self.group)
        return int(t.item())

    def finish(self):
        """Wait for everything enqueued on this rank (and, through the epoch slots, on its peers)."""
        self.fit.sync()
        if self.world > 1:
            self.dist.barrier(group=self.group)

    def exchange(self, side):
        if self.mode in ("local", "p2p"):
            return      # p2p: the rows already sit in every replica, completion is signalled on the device
        if self.mode == "p2p-host":
            self.fit.sync()
            self.dist.barrier(group=self.group)
            return
        from . import _lib
        M, ranges = (self.A, self.rangesA) if side == _lib.SIDE_CSR else (self.B, self.rangesB)
        works = []
        for r, (lo, hi) in enumerate(ranges):
            if hi > lo:
                works.append(self.dist.broadcast(M[lo:hi], src=r, group=self.group, async_op=True))
        for w in works:
            w.wait()

    def factors(self, root=None, out=None):
        """The fitted factors as host arrays.  Every rank's replica holds the same bits; with `root` set only
        that rank reads them back (the others return None) — the process that asked for the fit."""
        self.finish()
        if root is not None and self.rank != root:
            return None
        if self.mode == "nccl":
            k = self.k
            return self.A[:, :k].cpu().numpy(), self.B[:, :k].cpu().numpy()
        return self.fit.get_factors(*(out or (None, None)))


    def topN(self, top_n, users=None, excl_ptr=None, excl_ix=None, output_score=False, gather=True, incl_ptr=None,
             incl_ix=None):
        """Batched top-N after the fit, users split across the ranks: every rank ranks its share against ITS
        replicas of A and B (resident: pmf_b200_topN_fitted, no factor leaves or enters a GPU) and the per-user
        lists are all-gathered: every rank returns the full (n_users x top_n) result.  With gather=False a
        rank returns the lists of its own share only (user_ranges(n_users, world)[rank]).  With `incl_ptr` /
        `incl_ix` user u ranks only its listed items (pmf_b200_topN_fitted_include)."""
        dimA, dimB, dt = self.fit.dimA, self.fit.dimB, self.fit.dtype

        def scorer(A_, B_, u_, p_, i_, n_, s_, include=False):
            if include:
                return self.fit.topN(users=u_, incl_ptr=p_, incl_ix=i_, top_n=n_, output_score=s_)
            return self.fit.topN(users=u_, excl_ptr=p_, excl_ix=i_, top_n=n_, output_score=s_)
        return topn_sharded(np.empty((dimA, 0), dt), np.empty((dimB, 0), dt), top_n, users=users, excl_ptr=excl_ptr,
                            excl_ix=excl_ix, output_score=output_score, rank=self.rank, world=self.world,
                            group=self.group, scorer=scorer, gather=gather, incl_ptr=incl_ptr, incl_ix=incl_ix)

    def topN_new(self, Xr_indptr, Xr_indices, Xr, top_n=10, excl_ptr=None, excl_ix=None, incl_ptr=None, incl_ix=None,
                 gather=True, **kw):
        """DeviceFit.topN_new with the new users split across the ranks (new_users_sharded): every rank folds in and
        ranks its share against ITS replicas; returns (ids, scores) or, with return_factors=True, (ids, scores, A)."""

        def fold(csr, p_, i_, include):
            lists = dict(incl_ptr=p_, incl_ix=i_) if include else dict(excl_ptr=p_, excl_ix=i_)
            return self.fit.topN_new(csr[1], csr[2], csr[0], top_n=top_n, **lists, **kw)
        return new_users_sharded((Xr, Xr_indptr, Xr_indices), fold, self.rank, self.world, self.group, excl_ptr,
                                 excl_ix, incl_ptr, incl_ix, gather)

    def transform(self, Xr_indptr, Xr_indices, Xr, gather=True, **kw):
        """DeviceFit.transform with the new users split across the ranks; returns their factors."""
        return new_users_sharded((Xr, Xr_indptr, Xr_indices),
                                 lambda csr, p_, i_, include: (self.fit.transform(csr[1], csr[2], csr[0], **kw),),
                                 self.rank, self.world, self.group, gather=gather)[0]


def user_ranges(n_users, nparts):
    """Contiguous, near-equal user ranges (topN work per user is the same: n items x k)."""
    cuts = [n_users * p // nparts for p in range(nparts + 1)]
    return [(cuts[i], cuts[i + 1]) for i in range(nparts)]


def _slice_lists(ptr, ix, lo, hi):
    """The per-user lists of users [lo, hi) as (offsets rebased to 0, ids), uint64; (None, None) without lists."""
    if ptr is None or ix is None:
        return None, None
    ep = np.asarray(ptr).astype(np.int64)
    return (np.ascontiguousarray(ep[lo:hi + 1] - ep[lo]).astype(np.uint64),
            np.ascontiguousarray(np.asarray(ix)[ep[lo]:ep[hi]]).astype(np.uint64))


def new_users_sharded(csr, fold, rank=0, world=1, group=None, excl_ptr=None, excl_ix=None, incl_ptr=None,
                      incl_ix=None, gather=True):
    """New users (CSR rows `csr` = (values, indptr, indices)) split across ranks: rank r folds in and ranks the
    contiguous range user_ranges(n_new, world)[r] against its own replicas, and the per-user results are all-gathered
    (with gather=False a rank returns its own range only).  Exclusion or include lists are sliced by the same range.
    `fold(csr_slice, list_ptr, list_ix, include) -> tuple of arrays with one row per user of the slice` does the
    work (GpuBackend.topN_new / transform pass the resident handle's; the CPU tests inject a stand-in)."""
    include = incl_ptr is not None or incl_ix is not None
    if include and (excl_ptr is not None or excl_ix is not None):
        raise ValueError("topN: include and exclude lists cannot be combined")
    lo, hi = user_ranges(csr[1].shape[0] - 1, world)[rank]
    p_loc, i_loc = _slice_lists(*((incl_ptr, incl_ix) if include else (excl_ptr, excl_ix)), lo, hi)
    out = tuple(fold(slice_compressed(csr, lo, hi), p_loc, i_loc, include))
    if world == 1 or not gather:
        return out
    import torch.distributed as dist
    parts = [None] * world
    dist.all_gather_object(parts, out, group=group)
    return tuple(np.concatenate([p[j] for p in parts], axis=0) for j in range(len(out)))


def topn_sharded(A, B, top_n, users=None, excl_ptr=None, excl_ix=None, output_score=False, rank=0, world=1,
                 group=None, scorer=None, gather=True, incl_ptr=None, incl_ix=None):
    """Batched topN with the USERS split across ranks (SURVEY.md 8e): B is replicated, every rank ranks
    its own contiguous range of users on its GPU, and the per-user lists are all-gathered — no exchange
    inside the scoring.  Every rank returns the full (n_users x top_n) result.  With `incl_ptr` / `incl_ix`
    user u ranks only the items incl_ix[incl_ptr[u]:incl_ptr[u+1]]; they are sliced by user range like the
    exclusion lists.

    `scorer(A, B, users, excl_ptr, excl_ix, top_n, output_score) -> (ids, scores)` defaults to the
    device path (c_funs._topN_batch); the CPU tests inject a stand-in.  With include lists it is called as
    `scorer(A, B, users, incl_ptr, incl_ix, top_n, output_score, include=True)`."""
    include = incl_ptr is not None or incl_ix is not None
    if include and (excl_ptr is not None or excl_ix is not None):
        raise ValueError("topN: include and exclude lists cannot be combined")
    if scorer is None:
        from . import c_funs

        def scorer(A_, B_, u_, p_, i_, n_, s_, include=False):
            if include:
                return c_funs._topN_batch(A_, B_, users=u_, incl_ptr=p_, incl_ix=i_, top_n=n_, output_score=s_)
            return c_funs._topN_batch(A_, B_, users=u_, excl_ptr=p_, excl_ix=i_, top_n=n_, output_score=s_)
    all_users = np.arange(A.shape[0], dtype=np.uint64) if users is None else np.ascontiguousarray(users, dtype=np.uint64)
    lo, hi = user_ranges(all_users.shape[0], world)[rank]
    mine = np.ascontiguousarray(all_users[lo:hi])
    p_loc, i_loc = _slice_lists(*((incl_ptr, incl_ix) if include else (excl_ptr, excl_ix)), lo, hi)
    if hi > lo:
        if include:
            ids, sc = scorer(A, B, mine, p_loc, i_loc, top_n, output_score, include=True)
        else:
            ids, sc = scorer(A, B, mine, p_loc, i_loc, top_n, output_score)
    else:
        ids = np.empty((0, top_n), np.uint64)
        sc = np.empty((0, top_n) if output_score else (0, 0), B.dtype)
    if world == 1 or not gather:
        return ids, sc
    import torch.distributed as dist
    parts = [None] * world
    dist.all_gather_object(parts, (ids, sc), group=group)
    ids = np.concatenate([p[0] for p in parts], axis=0)
    sc = np.concatenate([p[1] for p in parts], axis=0) if output_score else parts[0][1]
    return ids, sc

