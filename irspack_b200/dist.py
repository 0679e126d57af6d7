"""Row-sharded multi-GPU iALS: one process per GPU, ``torch.distributed`` plumbing.

The reference is single-process (SURVEY.md 8 e); its row solves are independent
within a half-epoch (every worker writes only its own ``target_factor`` rows,
/root/reference/cpp_source/als/IALSTrainer.hpp:193-265, 291-325), so users and
items are partitioned into ``world`` contiguous, nnz-balanced row ranges:

* rank r holds the CSR rows of X for its users, the CSR rows of X^T for its
  items and FULL replicas of both factor matrices;
* a half-epoch is  partial Gram of the rank's own rows of the other side
  -> all-reduce(sum) of the K x K buffer (NCCL; 64 KB at K=128)
  -> row solve of the rank's own rows;
* the all-gather of the freshly solved rows is FUSED INTO THE SOLVE KERNEL: the
  kernel stores every solved row into the local replica and, through CUDA-IPC
  mapped peer pointers, into every peer's replica over NVLink (no separate
  collective, the transfer overlaps the arithmetic row by row).  The Gram
  all-reduce of the next half-epoch is the only synchronisation point: it orders
  a rank's reads of a replica after every peer's writes to it.

Everything above the C ABI here is host logic (partitioning, the one-off
exchange of transposed shards, collectives); it runs on ``gloo`` without a GPU
for the world_size-2 CPU tests.
"""
from __future__ import annotations

import ctypes
import json
import os
import time
from typing import Any, List, Optional, Sequence, Tuple

import numpy as np
import scipy.sparse as sps

# ----------------------------------------------------------------------------
# host logic (no GPU needed)
# ----------------------------------------------------------------------------


def balanced_bounds(weights: np.ndarray, world: int) -> np.ndarray:
    """``world + 1`` non-decreasing boundaries cutting ``weights`` into contiguous
    ranges of (nearly) equal total weight -- nnz-balanced row shards, not equal
    row counts (power-law degrees).  Rows are weighted ``nnz + 1`` by callers so
    that empty rows still spread evenly."""
    weights = np.asarray(weights, dtype=np.float64)
    n = weights.shape[0]
    if world < 1:
        raise ValueError("world must be positive")
    csum = np.concatenate([[0.0], np.cumsum(weights)])
    targets = csum[-1] * np.arange(1, world, dtype=np.float64) / world
    cuts = np.searchsorted(csum, targets, side="left")
    bounds = np.concatenate([[0], cuts, [n]]).astype(np.int64)
    return np.maximum.accumulate(np.minimum(bounds, n))


def transposed_pieces(X_local: sps.csr_matrix, user_offset: int, item_bounds: Sequence[int]
                      ) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
    """Cut this rank's user block (rows = its users, columns = all items) into the
    pieces of X^T each rank needs: for destination d, items
    ``[item_bounds[d], item_bounds[d+1])`` as (per-item counts int64, global user
    ids int32 ascending within an item, values float32)."""
    Xc = sps.csc_matrix(X_local)
    Xc.sort_indices()
    indptr = Xc.indptr.astype(np.int64)
    out = []
    for d in range(len(item_bounds) - 1):
        b, e = int(item_bounds[d]), int(item_bounds[d + 1])
        s, t = indptr[b], indptr[e]
        counts = np.diff(indptr[b:e + 1]).astype(np.int64)
        users = (Xc.indices[s:t].astype(np.int64) + user_offset).astype(np.int32)
        out.append((counts, users, Xc.data[s:t].astype(np.float32)))
    return out


def assemble_transposed_shard(pieces: Sequence[Tuple[np.ndarray, np.ndarray, np.ndarray]],
                              n_users_global: int) -> sps.csr_matrix:
    """Merge the pieces received from ranks 0..world-1 (ascending user blocks) into
    this rank's rows of X^T (CSR: items x all users, user ids ascending)."""
    n_items = pieces[0][0].shape[0]
    counts = np.stack([p[0] for p in pieces])            # [world, n_items]
    total = counts.sum(axis=0)
    indptr = np.zeros(n_items + 1, dtype=np.int64)
    np.cumsum(total, out=indptr[1:])
    nnz = int(indptr[-1])
    indices = np.empty(nnz, dtype=np.int32)
    data = np.empty(nnz, dtype=np.float32)
    before = np.cumsum(counts, axis=0) - counts          # entries of earlier sources per item
    for s, (cnt, users, vals) in enumerate(pieces):
        if users.size == 0:
            continue
        start = indptr[:-1] + before[s]                  # destination of each item's run
        src_start = np.concatenate([[0], np.cumsum(cnt)[:-1]])
        pos = np.repeat(start - src_start, cnt) + np.arange(users.size, dtype=np.int64)
        indices[pos] = users
        data[pos] = vals
    M = sps.csr_matrix((data, indices, indptr), shape=(n_items, n_users_global))
    M.has_sorted_indices = True
    return M


def _p2p_exchange(send: List[Any], rank: int, world: int, device: Any) -> List[Any]:
    """All-to-all of one tensor per destination with point-to-point ops (works on
    both NCCL and gloo).  Sizes are exchanged first."""
    import torch
    import torch.distributed as dist

    sizes = torch.tensor([t.numel() for t in send], dtype=torch.int64, device=device)
    all_sizes = [torch.empty_like(sizes) for _ in range(world)]
    dist.all_gather(all_sizes, sizes)
    recv: List[Any] = [None] * world
    recv[rank] = send[rank]
    for k in range(1, world):
        dst, src = (rank + k) % world, (rank - k) % world
        n_in = int(all_sizes[src][rank].item())
        buf = torch.empty(n_in, dtype=send[dst].dtype, device=device)
        ops = []
        if send[dst].numel():
            ops.append(dist.P2POp(dist.isend, send[dst].contiguous(), dst))
        if n_in:
            ops.append(dist.P2POp(dist.irecv, buf, src))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        recv[src] = buf
    return recv


def exchange_transposed_shards(X_local: sps.csr_matrix, user_offset: int, n_users_global: int,
                               item_bounds: Sequence[int], device: Any = "cpu") -> sps.csr_matrix:
    """Collective: every rank contributes its user block and receives its rows of
    X^T (items ``[item_bounds[rank], item_bounds[rank+1])`` x all users)."""
    import torch
    import torch.distributed as dist

    rank, world = dist.get_rank(), dist.get_world_size()
    pieces = transposed_pieces(X_local, user_offset, item_bounds)
    got = []
    for field, dtype in ((0, torch.int64), (1, torch.int32), (2, torch.float32)):
        send = [torch.from_numpy(np.ascontiguousarray(p[field])).to(device=device, dtype=dtype)
                for p in pieces]
        got.append([t.cpu().numpy() for t in _p2p_exchange(send, rank, world, device)])
    merged = [(got[0][s], got[1][s], got[2][s]) for s in range(world)]
    return assemble_transposed_shard(merged, n_users_global)


def global_item_bounds(X_local: sps.csr_matrix, device: Any = "cpu") -> np.ndarray:
    """nnz-balanced item ranges from the global item degrees (all-reduce of bincounts)."""
    import torch
    import torch.distributed as dist

    cnt = torch.from_numpy(np.bincount(X_local.indices, minlength=X_local.shape[1]).astype(np.int64))
    cnt = cnt.to(device)
    dist.all_reduce(cnt)
    return balanced_bounds(cnt.cpu().numpy() + 1, dist.get_world_size())


# ----------------------------------------------------------------------------
# device-resident shard construction (1 B-interaction matrices: BASELINE configs[3], [4]).
# Same results as the scipy functions above, on torch tensors of any device: nothing of the
# matrix touches the host, so a 125 M-interaction shard per rank is built in seconds.
# ----------------------------------------------------------------------------


def synth_user_block_device(n_users_block: int, n_items: int, nnz_block: int, seed: int,
                            device: Any, item_seed: int = 0) -> Tuple[Any, Any, Any]:
    """This rank's rows of a synthetic power-law matrix (SURVEY.md 8 d) as a device CSR:
    ``(indptr int64 [n_users_block + 1], indices int32 ascending within a row, data float32
    ones)`` with exactly ``nnz_block`` distinct pairs.  User activity ~ lognormal(sigma = 1)
    from ``seed`` (rank-specific); item popularity ~ (rank + n_items/400)^-1 in a random item
    order drawn from ``item_seed`` -- the SAME on every rank, so that the stacked blocks share
    one popularity law (``synth.synth_csr`` is the host twin of this generator)."""
    import torch

    if nnz_block > n_users_block * n_items:
        raise ValueError("nnz exceeds the block size")
    g = torch.Generator(device=device).manual_seed(int(seed))
    gi = torch.Generator(device=device).manual_seed(int(item_seed))
    pu = torch.exp(torch.randn(n_users_block, generator=g, device=device, dtype=torch.float64))
    pi = 1.0 / (torch.arange(n_items, device=device, dtype=torch.float64) + max(n_items / 400.0, 1.0))
    pi = pi[torch.randperm(n_items, generator=gi, device=device)]
    cu = torch.cumsum(pu / pu.sum(), 0)
    ci = torch.cumsum(pi / pi.sum(), 0)
    cu[-1] = ci[-1] = 1.0
    keys = torch.empty(0, dtype=torch.int64, device=device)
    while keys.numel() < nnz_block:
        m = int((nnz_block - keys.numel()) * 1.25) + 1024
        rows = torch.searchsorted(cu, torch.rand(m, generator=g, device=device, dtype=torch.float64),
                                  right=True).clamp_(max=n_users_block - 1)
        cols = torch.searchsorted(ci, torch.rand(m, generator=g, device=device, dtype=torch.float64),
                                  right=True).clamp_(max=n_items - 1)
        keys = torch.unique(torch.cat([keys, rows * n_items + cols]))  # sorted, duplicate-free
    if keys.numel() > nnz_block:
        keep = torch.randperm(keys.numel(), generator=g, device=device)[:nnz_block]
        keys = keys[torch.sort(keep).values]
    rows = torch.div(keys, n_items, rounding_mode="floor")
    indices = (keys - rows * n_items).to(torch.int32)
    indptr = torch.zeros(n_users_block + 1, dtype=torch.int64, device=device)
    indptr[1:] = torch.cumsum(torch.bincount(rows, minlength=n_users_block), 0)
    return indptr, indices, torch.ones(nnz_block, dtype=torch.float32, device=device)


def global_item_bounds_device(indices: Any, n_items: int) -> np.ndarray:
    """``global_item_bounds`` for a device-resident block (all-reduce of the item degrees)."""
    import torch
    import torch.distributed as dist

    cnt = torch.bincount(indices.to(torch.int64), minlength=n_items)
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(cnt)
    world = dist.get_world_size() if dist.is_initialized() else 1
    return balanced_bounds(cnt.cpu().numpy() + 1, world)


def exchange_transposed_shards_device(indptr: Any, indices: Any, data: Any, user_offset: int,
                                      n_users_global: int, item_bounds: Sequence[int]
                                      ) -> Tuple[Any, Any, Any]:
    """``exchange_transposed_shards`` on device tensors: every rank contributes its user block
    (CSR, local rows) and receives its rows of X^T -- items
    ``[item_bounds[rank], item_bounds[rank + 1])`` x all users -- as a device CSR
    ``(indptr int64, indices int32 = global user ids ascending, data float32)``.

    One key per interaction, ``item * n_users_global + user``: sorting the keys IS the
    transposition; destinations are contiguous key ranges."""
    import torch
    import torch.distributed as dist

    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    device = indices.device
    n_rows = indptr.numel() - 1
    rows = torch.repeat_interleave(torch.arange(n_rows, device=device, dtype=torch.int64),
                                   indptr[1:] - indptr[:-1]) + int(user_offset)
    keys, order = torch.sort(indices.to(torch.int64) * int(n_users_global) + rows)
    vals = data[order]
    del rows, order
    bounds = torch.as_tensor(np.asarray(item_bounds, dtype=np.int64), device=device)
    cuts = torch.searchsorted(keys, bounds * int(n_users_global)).tolist()
    if world > 1:
        send_k = [keys[cuts[d]:cuts[d + 1]] for d in range(world)]
        send_v = [vals[cuts[d]:cuts[d + 1]] for d in range(world)]
        keys = torch.cat(_p2p_exchange(send_k, rank, world, device))
        vals = torch.cat(_p2p_exchange(send_v, rank, world, device))
        # sources own disjoint ascending user ranges: one more sort merges their runs
        keys, order = torch.sort(keys)
        vals = vals[order]
        del order
    b, e = int(item_bounds[rank]), int(item_bounds[rank + 1])
    items = torch.div(keys, int(n_users_global), rounding_mode="floor")
    users = (keys - items * int(n_users_global)).to(torch.int32)
    t_indptr = torch.zeros(e - b + 1, dtype=torch.int64, device=device)
    t_indptr[1:] = torch.cumsum(torch.bincount(items - b, minlength=e - b), 0)
    return t_indptr, users, vals.contiguous()


# ----------------------------------------------------------------------------
# the sharded trainer (needs the CUDA library)
# ----------------------------------------------------------------------------


class ShardedIALSTrainer:
    """One rank of the row-sharded trainer (``ials_trainer_create_sharded``).

    ``X_user_rows``: this rank's users x all items (CSR); ``Xt_item_rows``: this
    rank's items x all users (CSR) -- two scipy matrices, or two device CSR triples
    ``(indptr, indices, data)`` of torch tensors on this rank's GPU
    (``exchange_transposed_shards_device``).  ``user`` / ``item`` return the local full
    replicas, identical on every rank after ``sync()``.

    ``user_feature`` / ``item_feature`` (both or neither): this rank's rows of the feature
    matrices, dense or scipy sparse -- the feature-aware model of
    ``IALSTrainer(config, X, user_feature, item_feature)`` with the config's
    ``lambda_*_feature`` and ``feature_warmup_epochs``.  Each epoch then refits the feature
    weights from sums over all ranks; every rank holds the same weights."""

    def __init__(self, model_config: Any, X_user_rows: sps.csr_matrix, user_begin: int,
                 n_users: int, Xt_item_rows: sps.csr_matrix, item_begin: int, n_items: int,
                 init_on_device: bool = False, user_feature: Any = None, item_feature: Any = None) -> None:
        import torch
        import torch.distributed as dist

        from . import _ials_core as core
        from ._lib import check, lib

        if (user_feature is None) != (item_feature is None):
            raise TypeError("the feature-aware trainer takes both user_feature and item_feature; pass a "
                            "matrix with 0 columns for a side without features")
        self._core, self._lib, self._check = core, lib, check
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.n_users, self.n_items, self.K = int(n_users), int(n_items), int(model_config.K)
        self._device, stream = core._current_device_and_stream()
        on_device = isinstance(X_user_rows, (tuple, list))
        if on_device != isinstance(Xt_item_rows, (tuple, list)):
            raise ValueError("both shards must be scipy matrices or both device CSR triples")
        if on_device:
            # (indptr int64, indices int32, data float32) torch tensors on this rank's GPU
            # (exchange_transposed_shards_device); the library copies them (device to device)
            keep = []
            ptrs = []
            rows = []
            for triple in (X_user_rows, Xt_item_rows):
                ip, ix, dt = triple
                ip = ip.to(dtype=torch.int64).contiguous()
                ix = ix.to(dtype=torch.int32).contiguous()
                dt = dt.to(dtype=torch.float32).contiguous()
                for t in (ip, ix, dt):
                    if not t.is_cuda or t.device.index != self._device:
                        raise ValueError(f"device CSR arrays must live on cuda:{self._device}")
                if ix.numel() != dt.numel() or ip.numel() < 1:
                    raise ValueError("malformed device CSR")
                keep.append((ip, ix, dt))
                ptrs.append(tuple(ctypes.c_void_p(t.data_ptr()) for t in (ip, ix, dt)))
                rows.append(ip.numel() - 1)
            torch.cuda.current_stream(self._device).synchronize()  # the copies below are synchronous
            ua, ia = ptrs
            n_u_rows, n_i_rows = rows
            self.nnz_local = int(keep[0][1].numel())
        else:
            Xu = core._canonical_csr(X_user_rows)
            Xi = core._canonical_csr(Xt_item_rows)
            if Xu.shape[1] != n_items or Xi.shape[1] != n_users:
                raise ValueError("shard shapes do not match the global matrix")
            keep = [core._csr_arrays(Xu), core._csr_arrays(Xi)]
            ua, ia = (tuple(core._ptr(a) for a in arrs) for arrs in keep)
            n_u_rows, n_i_rows = Xu.shape[0], Xi.shape[0]
            self.nnz_local = int(Xu.nnz)
        self.user_range = (int(user_begin), int(user_begin) + n_u_rows)
        self.item_range = (int(item_begin), int(item_begin) + n_i_rows)
        cfg = model_config._as_struct()
        h = ctypes.c_void_p(0)
        check(lib.ials_trainer_create_sharded(
            ctypes.byref(cfg), self.n_users, self.n_items, self.user_range[0], self.user_range[1],
            ua[0], ua[1], ua[2], self.item_range[0], self.item_range[1], ia[0], ia[1], ia[2],
            int(on_device), int(bool(init_on_device)), self._device, ctypes.byref(h)))
        del keep
        self._handle = h
        check(lib.ials_trainer_set_stream(h, ctypes.c_void_p(stream)))
        self._torch = torch
        self._buffer_views: dict = {}
        # per side: does some rank's shard hold an empty row (the guard of step_with_prior needs the
        # OR over all ranks, so that every rank rejects an epoch alike)
        self._empty_row = (0, 0)
        self._feature_aware = user_feature is not None
        if user_feature is not None:
            self._set_features(model_config, (user_feature, item_feature))
        if self.world > 1:
            self._open_peers()

    def _set_features(self, model_config: Any, features: Tuple[Any, Any]) -> None:
        lams = (model_config.lambda_user_feature, model_config.lambda_item_feature)
        empty = [0, 0]
        err: Optional[BaseException] = None
        try:
            for side, F in enumerate(features):
                rows, cols, dense, ip, ix, dt = self._core._feature_arrays(F)
                flag = ctypes.c_int(0)
                p = self._core._ptr
                self._check(self._lib.ials_trainer_set_shard_features(
                    self._handle, side, rows, cols, p(dense), p(ip), p(ix), p(dt), ctypes.c_float(lams[side]),
                    int(model_config.feature_warmup_epochs), ctypes.byref(flag)))
                empty[side] = flag.value
        except (RuntimeError, ValueError, TypeError) as e:  # a shard of the wrong size may be one rank's
            err = e
        failed, *self._empty_row = self._max_over_ranks([1 if err is not None else 0] + empty)
        self._raise_agreed(err, failed)

    def _max_over_ranks(self, values: List[int]) -> List[int]:
        import torch.distributed as dist

        if self.world == 1:
            return list(values)
        dev = f"cuda:{self._device}" if dist.get_backend() == "nccl" else "cpu"
        t = self._torch.tensor(values, dtype=self._torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [int(v) for v in t.tolist()]

    @staticmethod
    def _raise_agreed(err: Optional[BaseException], failed: int) -> None:
        """Raise this rank's exception, or report a peer's failure, on every rank alike."""
        if err is not None:
            raise err
        if failed:
            raise RuntimeError("a peer rank failed (see that rank's exception)")

    @classmethod
    def from_global(cls, model_config: Any, X: sps.csr_matrix, rank: Optional[int] = None,
                    world: Optional[int] = None, user_feature: Any = None, item_feature: Any = None,
                    **kw: Any) -> "ShardedIALSTrainer":
        """Shard a matrix (and the feature matrices) every rank holds in full (tests, small problems)."""
        import torch.distributed as dist

        rank = dist.get_rank() if rank is None else rank
        world = dist.get_world_size() if world is None else world
        X = sps.csr_matrix(X)
        Xt = sps.csr_matrix(X.T)
        ub = balanced_bounds(np.diff(X.indptr) + 1, world)
        ib = balanced_bounds(np.diff(Xt.indptr) + 1, world)

        def rows(F: Any, b: int, e: int) -> Any:
            if F is None:
                return None
            return (sps.csr_matrix(F) if sps.issparse(F) else np.asarray(F))[b:e]

        return cls(model_config, X[ub[rank]:ub[rank + 1]], ub[rank], X.shape[0],
                   Xt[ib[rank]:ib[rank + 1]], ib[rank], X.shape[1],
                   user_feature=rows(user_feature, ub[rank], ub[rank + 1]),
                   item_feature=rows(item_feature, ib[rank], ib[rank + 1]), **kw)

    def __del__(self) -> None:
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            self._lib.ials_trainer_destroy(h)
            self._handle = ctypes.c_void_p(0)

    # -- peer replicas over CUDA IPC (NVLink P2P stores from the solve kernel) --
    def _open_peers(self) -> None:
        import torch.distributed as dist

        for side in (0, 1):
            buf = (ctypes.c_ubyte * 64)()
            self._check(self._lib.ials_trainer_ipc_handle(self._handle, side, buf))
            handles: List[Any] = [None] * self.world
            dist.all_gather_object(handles, bytes(buf))
            blob = np.frombuffer(b"".join(handles), dtype=np.uint8).copy()
            self._check(self._lib.ials_trainer_ipc_open_peers(
                self._handle, side, blob.ctypes.data_as(ctypes.c_void_p), self.world, self.rank))
        dist.barrier()

    def _use_current_stream(self) -> None:
        stream = self._core._stream_of(self._device)  # the trainer's own device, not torch's current one
        self._check(self._lib.ials_trainer_set_stream(self._handle, ctypes.c_void_p(stream)))

    def _buffer_view(self, ptr: ctypes.c_void_p, count: ctypes.c_int64) -> Any:
        """Zero-copy flat torch view of a trainer-owned float buffer (cached per buffer)."""
        key = (int(ptr.value), int(count.value))
        if key not in self._buffer_views:
            arr = self._core._DeviceArray(key[0], (key[1],), (4,))
            self._buffer_views[key] = self._torch.as_tensor(arr, device=f"cuda:{self._device}")
        return self._buffer_views[key]

    def _gram_partial(self, factor_side: int) -> Any:
        ptr, cnt = ctypes.c_void_p(0), ctypes.c_int64(0)
        self._check(self._lib.ials_trainer_gram_partial(self._handle, factor_side, ctypes.byref(ptr),
                                                        ctypes.byref(cnt)))
        return self._buffer_view(ptr, cnt)

    def _refit(self, side: int) -> None:
        """The feature-weight refit of ``side`` after its solve (IALSTrainer.hpp:777-778): this rank's
        F^T D F (first refit only) and F^T D X, all-reduced, then the same ridge solve on every rank.
        Nothing (and no collective, on any rank) when the solve used no prior."""
        bufs = [(ctypes.c_void_p(0), ctypes.c_int64(0)) for _ in range(2)]
        self._check(self._lib.ials_trainer_feature_partials(
            self._handle, side, ctypes.byref(bufs[0][0]), ctypes.byref(bufs[0][1]), ctypes.byref(bufs[1][0]),
            ctypes.byref(bufs[1][1])))
        for ptr, cnt in bufs:
            if cnt.value:
                self._all_reduce(self._buffer_view(ptr, cnt))
        self._check(self._lib.ials_trainer_feature_refit(self._handle, side))

    def _check_step(self, sc: Any) -> None:
        """The rejections of a feature-aware epoch, before its first collective and before any factor
        changes; decided from state every rank shares, so every rank raises alike."""
        self._check(self._lib.ials_trainer_check_shard_step(self._handle, ctypes.byref(sc), *self._empty_row))

    def _all_reduce_max(self, host: Any) -> None:
        """Element-wise MAX over ranks of a host tensor, in place."""
        import torch.distributed as dist

        if self.world == 1:
            return
        if dist.get_backend() == "nccl":
            dev = host.to(f"cuda:{self._device}")
            dist.all_reduce(dev, op=dist.ReduceOp.MAX)
            host.copy_(dev.cpu())
        else:
            dist.all_reduce(host, op=dist.ReduceOp.MAX)

    def _all_reduce(self, view: Any) -> None:
        import torch.distributed as dist

        if self.world == 1:
            return
        if dist.get_backend() == "nccl":
            dist.all_reduce(view)
        else:  # gloo control plane (several ranks on one GPU in the tests): stage through the host
            h = view.cpu()
            dist.all_reduce(h)
            view.copy_(h)

    def step_async(self, solver_config: Any, events: Optional[list] = None) -> None:
        """One epoch (IALSTrainer::step, IALSTrainer.hpp:758-789) across all ranks.  With
        ``events`` (a list) seven CUDA events are appended: start, then after the partial Gram,
        the Gram all-reduce and the row solve (with the feature-weight refit) of each side
        (``phase_ms`` turns them into ms)."""
        sc = self._core.IALSTrainer._solver(solver_config)
        self._check_step(sc)
        self._use_current_stream()

        def mark() -> None:
            if events is not None:
                e = self._torch.cuda.Event(enable_timing=True)
                e.record(self._torch.cuda.current_stream(self._device))
                events.append(e)

        mark()
        for side in (0, 1):
            view = self._gram_partial(1 - side)
            mark()
            self._all_reduce(view)
            mark()
            self._check(self._lib.ials_trainer_solve_shard(self._handle, side, ctypes.byref(sc)))
            self._refit(side)
            mark()

    PHASES = ("gram_item_partial", "gram_item_allreduce", "solve_users",
              "gram_user_partial", "gram_user_allreduce", "solve_items")

    @classmethod
    def phase_ms(cls, events: list) -> dict:
        """Per-phase milliseconds (averaged over the recorded epochs) of ``step_async(events=...)``."""
        n = len(events) // 7
        out = {k: 0.0 for k in cls.PHASES}
        for e in range(n):
            ev = events[7 * e: 7 * e + 7]
            for i, k in enumerate(cls.PHASES):
                out[k] += ev[i].elapsed_time(ev[i + 1]) / max(n, 1)
        return out

    def sync(self) -> None:
        """Wait for this rank's kernels, raise solver failures, and make every peer's
        stores into the local replicas complete (barrier)."""
        import torch.distributed as dist

        if self.world == 1:
            self._check(self._lib.ials_trainer_sync(self._handle))
            return
        # a solver failure on ONE rank (singular CG system, failed Cholesky) must not leave the
        # others blocked in the barrier: agree on the status first, then raise everywhere
        err: Optional[BaseException] = None
        try:
            self._check(self._lib.ials_trainer_sync(self._handle))
        except (RuntimeError, ValueError) as e:  # the exception types `check` maps status codes to
            err = e
        flag = self._torch.tensor([1 if err is not None else 0], dtype=self._torch.int32,
                                  device=f"cuda:{self._device}" if dist.get_backend() == "nccl" else "cpu")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        dist.barrier()
        if err is not None:
            raise err
        if int(flag.item()):
            raise RuntimeError("a peer rank's row solver failed (see that rank's exception)")

    def step(self, solver_config: Any) -> None:
        self.step_async(solver_config)
        self.sync()

    def compute_loss(self, solver_config: Any) -> float:
        """IALSTrainer::compute_loss (IALSTrainer.hpp:836-940) of the sharded model, the same float
        on every rank: every rank sums the terms of its own rows, rank 0 adds the Gram and the
        feature-weight terms, and the float64 partials are all-reduced.  Call it after ``step`` /
        ``sync`` (it reads the full replicas)."""
        import torch.distributed as dist

        sc = self._core.IALSTrainer._solver(solver_config)
        self._use_current_stream()
        out = ctypes.c_double(0.0)
        self._check(self._lib.ials_trainer_compute_loss_shard(self._handle, ctypes.byref(sc),
                                                              int(self.rank == 0), ctypes.byref(out)))
        total = out.value
        if self.world > 1:
            dev = f"cuda:{self._device}" if dist.get_backend() == "nccl" else "cpu"
            t = self._torch.tensor([total], dtype=self._torch.float64, device=dev)
            dist.all_reduce(t)
            total = float(t.item())
        return float(np.float32(total))  # the reference returns a float (IALSTrainer.hpp:836)

    def _get_feature_weight(self, side: int) -> np.ndarray:
        n = ctypes.c_int64(0)
        self._check(self._lib.ials_trainer_feature_weight_rows(self._handle, side, ctypes.byref(n)))
        out = np.zeros((int(n.value), self.K), dtype=np.float32)
        if n.value:
            self._use_current_stream()
            self._check(self._lib.ials_trainer_get_feature_weight(self._handle, side, self._core._ptr(out)))
        return out

    def _set_feature_weight(self, side: int, value: np.ndarray) -> None:
        """Collective: every rank calls it; rank 0's matrix becomes every rank's weight."""
        import torch.distributed as dist

        if self.world > 1:
            box = [np.ascontiguousarray(value, dtype=np.float32)]
            dist.broadcast_object_list(box, src=0)
            value = box[0]
        value = np.ascontiguousarray(value, dtype=np.float32)
        if value.ndim != 2 or (value.shape[0] and value.shape[1] != self.K):
            raise ValueError(f"expected an (n, {self.K}) matrix, got {value.shape}")
        self._use_current_stream()
        self._check(self._lib.ials_trainer_set_feature_weight(self._handle, side, int(value.shape[0]),
                                                              self._core._ptr(value)))

    user_feature_weight = property(lambda s: s._get_feature_weight(0), lambda s, v: s._set_feature_weight(0, v))
    item_feature_weight = property(lambda s: s._get_feature_weight(1), lambda s, v: s._set_feature_weight(1, v))

    def _get(self, side: int) -> np.ndarray:
        n = self.n_users if side == 0 else self.n_items
        out = np.empty((n, self.K), dtype=np.float32)
        self._use_current_stream()
        self._check(self._lib.ials_trainer_get_factors(self._handle, side, self._core._ptr(out)))
        return out

    def _set(self, side: int, value: np.ndarray) -> None:
        n = self.n_users if side == 0 else self.n_items
        value = np.ascontiguousarray(value, dtype=np.float32)
        if value.shape != (n, self.K):
            raise ValueError(f"expected a ({n}, {self.K}) matrix, got {value.shape}")
        self._use_current_stream()
        self._check(self._lib.ials_trainer_set_factors(self._handle, side, self._core._ptr(value)))

    user = property(lambda s: s._get(0), lambda s, v: s._set(0, v))
    item = property(lambda s: s._get(1), lambda s, v: s._set(1, v))

    def get_factors_into(self, side: int, out: np.ndarray) -> None:
        self._use_current_stream()
        self._check(self._lib.ials_trainer_get_factors(self._handle, side, self._core._ptr(out)))

    def shard_range(self, side: int) -> Tuple[int, int]:
        return self.user_range if side == 0 else self.item_range

    def set_shard_rows(self, side: int, rows: np.ndarray, push_to_peers: bool = True) -> None:
        """Upload THIS rank's rows of a factor matrix from a (pinned) host buffer and copy them
        into every peer's replica over NVLink (``ials_trainer_set_factor_rows``): together the
        ranks bring each matrix down exactly once.  Asynchronous; the next epoch's Gram
        all-reduce orders every rank's solve after all ranks' copies.  ``push_to_peers=False``
        keeps the rows local (warm starts that the peers never read)."""
        b, e = self.shard_range(side)
        if rows.dtype != np.float32 or rows.shape != (e - b, self.K) or not rows.flags.c_contiguous:
            raise ValueError("rows must be C-contiguous float32 of shape (shard rows, K)")
        self._use_current_stream()
        self._check(self._lib.ials_trainer_set_factor_rows(self._handle, side, b, e - b,
                                                           self._core._ptr(rows), int(bool(push_to_peers))))

    def get_shard_rows(self, side: int, out: np.ndarray) -> None:
        """Read this rank's own (authoritative) rows back into a host buffer."""
        b, e = self.shard_range(side)
        if out.dtype != np.float32 or out.shape != (e - b, self.K) or not out.flags.c_contiguous:
            raise ValueError("out must be C-contiguous float32 of shape (shard rows, K)")
        self._use_current_stream()
        self._check(self._lib.ials_trainer_get_factor_rows(self._handle, side, b, e - b,
                                                           self._core._ptr(out)))

    def _factors_view(self, side: int) -> Any:
        """Zero-copy torch view ([n, ld]) of this rank's replica of a factor matrix."""
        p, n, K, ld = ctypes.c_void_p(0), ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
        self._check(self._lib.ials_trainer_factors_device(self._handle, side, ctypes.byref(p), ctypes.byref(n),
                                                          ctypes.byref(K), ctypes.byref(ld)))
        arr = self._core._DeviceArray(int(p.value), (int(n.value), int(ld.value)), (int(ld.value) * 4, 4))
        return self._torch.as_tensor(arr, device=f"cuda:{self._device}")

    def step_io(self, solver_config: Any, user_rows: Any, item_rows: Any) -> None:
        """One epoch on HOST-resident shards, in place (the row-sharded twin of
        ``IALSTrainer.step_io``): every rank uploads ITS OWN user and item rows from pinned host
        tensors (pushed to the peers' replicas over NVLink), the epoch runs, and the rank's own
        fresh rows come back -- the user rows on a second stream while the item half-epoch runs.
        ``user_rows`` / ``item_rows``: pinned float32 torch tensors of shape (shard rows, K)."""
        torch = self._torch
        sc = self._core.IALSTrainer._solver(solver_config)
        self._check_step(sc)  # before the uploads: a rejected call leaves the factors as they were
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=self._device)
            self._views = [self._factors_view(0), self._factors_view(1)]
        self.set_shard_rows(1, item_rows.numpy())  # item first: the user half-epoch starts with Gram(item)
        # the user rows are only the warm starts of this rank's solves: the peers' copies of them are
        # first read in the item half-epoch, after the solve kernels have stored the new values there;
        # they arrive in flagged chunks while the user half-epoch runs (ials_trainer_set_user_rows_flagged)
        ub, ue = self.user_range
        un = user_rows.numpy()
        if un.dtype != np.float32 or un.shape != (ue - ub, self.K) or not un.flags.c_contiguous:
            raise ValueError("user_rows must be C-contiguous float32 of shape (shard rows, K)")
        self._use_current_stream()
        self._check(self._lib.ials_trainer_set_user_rows_flagged(self._handle, ub, ue - ub, self._core._ptr(un)))
        main = torch.cuda.current_stream(self._device)
        for side in (0, 1):
            self._all_reduce(self._gram_partial(1 - side))
            self._check(self._lib.ials_trainer_solve_shard(self._handle, side, ctypes.byref(sc)))
            if side == 0:  # the rank's new user rows are final: they travel back during the item half
                done = torch.cuda.Event()
                done.record(main)
                b, e = self.user_range
                with torch.cuda.stream(self._copy_stream):
                    self._copy_stream.wait_event(done)
                    user_rows.copy_(self._views[0][b:e, : self.K], non_blocking=True)
            self._refit(side)
        b, e = self.item_range
        item_rows.copy_(self._views[1][b:e, : self.K], non_blocking=True)
        self._copy_stream.synchronize()
        self.sync()

    def recommend(self, begin: int, end: int, cutoff: int, idx: Optional[np.ndarray] = None,
                  cnt: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Fused score + seen-mask (training rows) + top-``cutoff`` for users ``[begin, end)`` of
        this rank's shard (the item factors are replicated: no collective, SURVEY.md 8 e)."""
        rows = int(end) - int(begin)
        if idx is None:
            idx = np.empty((rows, cutoff), dtype=np.int32)
        if cnt is None:
            cnt = np.empty((rows,), dtype=np.int32)
        p = self._core._ptr
        self._use_current_stream()
        self._check(self._lib.ials_trainer_recommend(self._handle, int(begin), int(end), int(cutoff), 0,
                                                     p(None), p(None), p(idx), p(None), p(cnt)))
        return idx, cnt

    # -- validation-based early stopping (BaseRecommenderWithEarlyStopping, base_earlystop.py:106-149) --
    def save_state(self, state: Optional[dict] = None) -> dict:
        """This rank's own rows of both factor matrices (into pinned host buffers: ``state`` from an
        earlier call is reused) and, for the feature-aware model, the feature weights."""
        if state is None:
            state = {side: self._torch.empty((e - b, self.K), dtype=self._torch.float32, pin_memory=True)
                     for side, (b, e) in enumerate((self.user_range, self.item_range))}
        for side in (0, 1):
            self.get_shard_rows(side, state[side].numpy())
        if self._feature_aware:
            state["weights"] = (self.user_feature_weight, self.item_feature_weight)
        return state

    def load_state(self, state: dict) -> None:
        """Collective: every rank uploads its saved rows and copies them into the peers' replicas, the
        weights are set on every rank, and ``sync`` leaves every replica on every rank identical."""
        for side in (0, 1):
            self.set_shard_rows(side, state[side].numpy(), push_to_peers=True)
        if "weights" in state:
            self.user_feature_weight, self.item_feature_weight = state["weights"]
        self.sync()

    def learn_with_optimizer(self, solver_config: Any, evaluator: Any = None, max_epoch: int = 128,
                             validate_epoch: int = 5, score_degradation_max: int = 5) -> int:
        """Collective epoch loop with validation-based early stopping (``IALSRecommender.
        learn_with_optimizer``, base_earlystop.py:106-149).  ``evaluator``: a ``ShardedEvaluator`` of
        this trainer; its score is the same on every rank, so is every decision.  Returns the number
        of epochs of the model left in the trainer: the best validated one (``max_epoch`` without an
        evaluator)."""
        best_score = -float("inf")
        best_epoch = 0
        n_score_degradation = 0
        state = None
        for epoch in range(max_epoch):
            self.step(solver_config)
            if (epoch + 1) % validate_epoch or evaluator is None:
                continue
            target_score = evaluator.get_target_score(self)
            if target_score > best_score:
                best_score = target_score
                state = self.save_state(state)
                best_epoch = epoch + 1
                n_score_degradation = 0
            else:
                n_score_degradation += 1
                if n_score_degradation >= score_degradation_max:
                    break
        if evaluator is None:
            return max_epoch
        if state is None:
            raise RuntimeError("'load_state' called before achieving any results.")
        self.load_state(state)
        return best_epoch

    def set_profiling(self, enabled: bool) -> None:
        self._check(self._lib.ials_trainer_set_profiling(self._handle, int(bool(enabled))))

    def plan_stats(self, side: int) -> dict:
        """Row schedule of this rank's shard of ``side`` (see ``IALSTrainer.plan_stats``)."""
        out = (ctypes.c_int64 * 8)()
        self._check(self._lib.ials_trainer_plan_stats(self._handle, side, out))
        keys = ("rows", "nnz", "heavy_rows", "heavy_nnz", "jobs", "max_degree", "has_negative",
                "reserved")
        return dict(zip(keys, (int(v) for v in out)))


class ShardedEvaluator:
    """The ``Evaluator`` of a row-sharded model, one per rank.

    ``ground_truth`` holds THIS rank's user rows only (``trainer.user_range``), shape
    ``(user_end - user_begin, n_items)``: a scipy matrix, or a device CSR triple ``(indptr, indices,
    data)`` of torch tensors on the trainer's GPU (only the indices are read, stored zeros included, as
    the ``Evaluator`` reads them).  ``per_user_recommendable_items`` and ``masked_interactions`` hold
    the same rows; the other arguments are the ``Evaluator``'s.  ``from_global`` slices matrices every
    rank holds in full.

    ``get_score`` / ``get_scores`` / ``get_target_score`` are collective and return, on every rank,
    what ``Evaluator`` returns for the gathered model.  Each rank scores and judges its own users on the
    device (``ials_trainer_evaluate``: the fused lists of ``max(cutoffs)``, then the metrics of every
    cutoff, no list leaves the device), the per-cutoff sums, counts and item histograms are
    all-reduced, and the diversity metrics are reduced from the merged histograms on the device.
    ``catalog_coverage`` divides by the number of recommendable items over ALL ranks' lists."""

    def __init__(self, trainer: "ShardedIALSTrainer", ground_truth: Any, cutoff: int = 10,
                 target_metric: str = "ndcg", recommendable_items: Optional[List[int]] = None,
                 per_user_recommendable_items: Any = None, masked_interactions: Any = None,
                 recall_with_cutoff: bool = False) -> None:
        import torch

        from .evaluation import Evaluator

        self._trainer = trainer
        self._sets: dict = {}
        self._gt_device = None
        self._lists = recommendable_items is not None or per_user_recommendable_items is not None
        self.last_timings: dict = {}
        ub, ue = trainer.user_range
        err: Optional[BaseException] = None
        try:
            gt = ground_truth
            if isinstance(gt, (tuple, list)):  # device CSR: rows sorted here, on the device
                ip = gt[0].to(torch.int64)
                ix = gt[1].to(torch.int64)
                n_rows = ip.numel() - 1
                if ip.device != torch.device(f"cuda:{trainer._device}") or ix.device != ip.device:
                    raise ValueError(f"device CSR arrays must live on cuda:{trainer._device}")
                rows = torch.repeat_interleave(torch.arange(n_rows, device=ip.device), ip[1:] - ip[:-1])
                keys = torch.sort(rows * trainer.n_items + ix).values
                self._gt_device = ((ip - ip[0]).contiguous(),
                                   (keys - rows * trainer.n_items).to(torch.int32).contiguous())
                gt = sps.csr_matrix((n_rows, trainer.n_items))
            if gt.shape[1] != trainer.n_items:
                raise ValueError("The model and evaluator assume different n_items.")
            if gt.shape[0] != ue - ub:
                raise ValueError(f"ground_truth must hold this rank's {ue - ub} user rows "
                                 f"[{ub}, {ue}), got {gt.shape[0]}.")
            self._ev = Evaluator(gt, offset=ub, cutoff=cutoff, target_metric=target_metric,
                                 recommendable_items=recommendable_items,
                                 per_user_recommendable_items=per_user_recommendable_items,
                                 masked_interactions=masked_interactions, recall_with_cutoff=recall_with_cutoff)
        except (ValueError, TypeError, KeyError, RuntimeError) as e:
            err = e
        failed, = trainer._max_over_ranks([1 if err is not None else 0])
        trainer._raise_agreed(err, failed)
        if recommendable_items is None and per_user_recommendable_items is not None:
            # the union of every rank's lists: one OR of the catalogue bitmaps
            seen = torch.zeros(trainer.n_items, dtype=torch.int32)
            seen[torch.from_numpy(self._ev._allow_sorted_flat.astype(np.int64))] = 1
            trainer._all_reduce_max(seen)
            self._ev.n_recommendable_items = int(seen.sum())

    @classmethod
    def from_global(cls, trainer: "ShardedIALSTrainer", ground_truth: Any,
                    per_user_recommendable_items: Any = None, masked_interactions: Any = None,
                    **kw: Any) -> "ShardedEvaluator":
        """Slice matrices (and per-user lists) that every rank holds in full by ``trainer.user_range``."""
        ub, ue = trainer.user_range

        def rows(m: Any) -> Any:
            if m is None:
                return None
            return sps.csr_matrix(m)[ub:ue] if sps.issparse(m) else m[ub:ue]

        return cls(trainer, rows(sps.csr_matrix(ground_truth)), per_user_recommendable_items=rows(
            per_user_recommendable_items), masked_interactions=rows(masked_interactions), **kw)

    def __del__(self) -> None:
        from ._lib import lib

        for h in getattr(self, "_sets", {}).values():
            lib.ials_eval_set_destroy(h)
        self._sets = {}

    @property
    def cutoff(self) -> int:
        return self._ev.cutoff

    @property
    def target_metric_name(self) -> str:
        return self._ev.target_metric_name

    def get_target_score(self, trainer: "ShardedIALSTrainer") -> float:
        return self.get_score(trainer)[self._ev.target_metric.name]

    def get_score(self, trainer: "ShardedIALSTrainer") -> dict:
        return self._get_scores_as_list(trainer, [self._ev.cutoff])[0]

    def get_scores(self, trainer: "ShardedIALSTrainer", cutoffs: List[int]) -> dict:
        return self._ev._flatten(cutoffs, self._get_scores_as_list(trainer, cutoffs))

    def _set_for(self, trainer: "ShardedIALSTrainer", cutoffs: Tuple[int, ...]) -> ctypes.c_void_p:
        from . import _ials_core as core
        from .evaluation import _mask_csr
        from ._lib import check, lib

        h = self._sets.get(cutoffs)
        if h is not None:
            return h
        ev, p = self._ev, core._ptr
        ub, ue = trainer.user_range
        if self._gt_device is not None:
            gi, gx = self._gt_device
            g_ptrs, on_device = (ctypes.c_void_p(gi.data_ptr()), ctypes.c_void_p(gx.data_ptr())), 1
        else:
            gi = np.ascontiguousarray(ev.ground_truth.indptr, dtype=np.int64)
            gx = np.ascontiguousarray(ev.ground_truth.indices, dtype=np.int32)
            g_ptrs, on_device = (p(gi), p(gx)), 0
        mi = mx = None
        if ev.masked_interactions is not None:
            mi, mx = _mask_csr(ev.masked_interactions)
        n_lists, ai, ax = ev._allowed_for(0, ue - ub, canonical=True) or (0, None, None)
        cut = np.ascontiguousarray(cutoffs, dtype=np.int64)
        h = ctypes.c_void_p(0)
        trainer._use_current_stream()
        check(lib.ials_eval_set_create(trainer._handle, ub, ue - ub, g_ptrs[0], g_ptrs[1], on_device, p(mi),
                                       p(mx), int(n_lists), p(ai), p(ax), p(cut), len(cutoffs),
                                       int(bool(ev.recall_with_cutoff)), ctypes.byref(h)))
        self._sets[cutoffs] = h
        return h

    def _views(self, h: ctypes.c_void_p) -> Tuple[Any, Any, Any]:
        """Zero-copy torch views of the set's sums (float64), counts and histograms (int64)."""
        from . import _ials_core as core
        from ._lib import check, lib

        ptrs = [ctypes.c_void_p(0) for _ in range(3)]
        n_cut, n_items = ctypes.c_int64(0), ctypes.c_int64(0)
        check(lib.ials_eval_set_buffers(h, *(ctypes.byref(x) for x in ptrs), ctypes.byref(n_cut),
                                        ctypes.byref(n_items)))
        dev = f"cuda:{self._trainer._device}"
        out = []
        for ptr, n, typ in zip(ptrs, (5 * n_cut.value, 2 * n_cut.value, n_cut.value * n_items.value),
                               ("<f8", "<i8", "<i8")):
            out.append(self._trainer._torch.as_tensor(core._DeviceArray(int(ptr.value), (n,), (8,), typ),
                                                      device=dev))
        return out[0], out[1], out[2]

    def _get_scores_as_list(self, trainer: "ShardedIALSTrainer", cutoffs: List[int]) -> List[dict]:
        from .evaluation import Metrics
        from ._lib import check, lib

        ev = self._ev
        cutoffs = [int(c) for c in cutoffs]
        ev._check_cutoffs(cutoffs)  # the same cutoffs and n_items on every rank: every rank raises alike
        if self._lists and max(cutoffs) > 128:
            raise NotImplementedError("allow-lists need the fused tensor-core kernel (cutoff <= 128)")
        torch = trainer._torch
        timings = {}
        err: Optional[BaseException] = None
        t0 = time.perf_counter()
        try:
            if trainer is not self._trainer:
                raise ValueError("the ShardedEvaluator was built for another trainer")
            h = self._set_for(trainer, tuple(cutoffs))
            stream = trainer._core._stream_of(trainer._device)
            check(lib.ials_eval_set_reset(h, ctypes.c_void_p(stream)))
            trainer._use_current_stream()
            ub, ue = trainer.user_range
            check(lib.ials_trainer_evaluate(trainer._handle, h, ub, ue))
        except (ValueError, RuntimeError, NotImplementedError) as e:
            err = e
        failed, = trainer._max_over_ranks([1 if err is not None else 0])
        trainer._raise_agreed(err, failed)
        t1 = time.perf_counter()
        sums, counts, hist = self._views(h)
        for view in (sums, counts, hist):
            trainer._all_reduce(view)
        torch.cuda.current_stream(trainer._device).synchronize()
        t2 = time.perf_counter()
        div = np.empty((len(cutoffs), 3), dtype=np.float64)
        check(lib.ials_eval_set_diversity(h, ctypes.c_void_p(stream), div.ctypes.data_as(ctypes.c_void_p)))
        t3 = time.perf_counter()
        s_host, c_host = sums.cpu().numpy().reshape(-1, 5), counts.cpu().numpy()
        self.last_timings = {"evaluate_s": t1 - t0, "allreduce_s": t2 - t1, "diversity_s": t3 - t2}
        out = []
        n_cut = len(cutoffs)
        for c in range(n_cut):
            m = Metrics(ev.n_items)
            m.hit, m.recall, m.ndcg, m.map, m.precision = (float(v) for v in s_host[c])
            m.valid_user, m.total_user = int(c_host[c]), int(c_host[n_cut + c])
            out.append(ev._metrics_as_dict(m, tuple(float(v) for v in div[c])))
        return out


# ----------------------------------------------------------------------------
# BASELINE configs[3] + [4]: the 1 B-interaction power-law matrix, row-sharded (bench.py --gpus N)
# ----------------------------------------------------------------------------


def c4_shape(scale: float, world: int) -> Tuple[int, int, int, int]:
    from .synth import SHAPES

    U0, I0, nnz0, K = SHAPES["powerlaw1b"]
    return (max(int(U0 * scale), world), max(int(I0 * scale), 128), int(nnz0 * scale), K)


def run_c4(hyper: dict, steps: int, warmup: int, scale: float = 1.0, e2e_steps: int = 3,
           score_users_per_rank: int = 100_000, score_block: int = 16384, topk: int = 100,
           shape: Optional[Tuple[int, int, int, int]] = None, solver: str = "CG",
           parity_sample: int = 64, parity_check: Any = None) -> Optional[dict]:
    """configs[3]: ``steps`` epochs of iALS K=128 CG on the synthetic power-law matrix (10 M x 2 M,
    1 B interactions at ``scale`` 1), row-sharded over the ranks of the initialised process group
    (or one GPU), STRONG scaling: the matrix is fixed, every rank draws its user block on the
    device and the rows of X^T are exchanged device to device.  configs[4]: top-``topk`` with the
    seen-item mask for a bounded sample of each rank's users.  Timing: CUDA events on the
    launching stream around exactly ``steps`` epochs, barrier + synchronize on both sides, MAX
    over ranks.  Returns the result dict on rank 0 (None elsewhere).  ``parity_check`` (optional, the
    same on every rank): a callable that re-solves rank 0's ``parity_sample`` sampled user rows with
    an independent implementation and returns a dict for the result's ``parity_sample`` key.

    ``shape`` = (users, items, interactions, K) and ``solver`` ("CG" | "CHOLESKY") run another
    configuration through the same code: configs[2] (Netflix shape, K = 256, Cholesky) on N GPUs
    is ``tools/time_c3_sharded.py``."""
    import torch
    import torch.distributed as dist

    from . import _ials_core as core
    from ._lib import lib

    multi = dist.is_initialized() and dist.get_world_size() > 1
    rank = dist.get_rank() if multi else 0
    world = dist.get_world_size() if multi else 1
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    U, I, nnz, K = c4_shape(scale, world) if shape is None else shape

    def barrier() -> None:
        if multi:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if not multi:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: int) -> int:
        if not multi:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        return int(t.item())

    # user blocks of equal row count and equal nnz (the generator draws exactly nnz/world pairs
    # per block): nnz-balanced by construction; items are cut by their global degrees
    ub = np.linspace(0, U, world + 1).astype(np.int64)
    nb = np.linspace(0, nnz, world + 1).astype(np.int64)
    n_rows, n_nnz = int(ub[rank + 1] - ub[rank]), int(nb[rank + 1] - nb[rank])
    t0 = time.perf_counter()
    ip, ix, dt = synth_user_block_device(n_rows, I, n_nnz, seed=1004 + rank, device=dev, item_seed=1004)
    item_bounds = global_item_bounds_device(ix, I)
    t_ip, t_ix, t_dt = exchange_transposed_shards_device(ip, ix, dt, int(ub[rank]), U, item_bounds)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(hyper["alpha0"]).set_reg(hyper["reg"])
           .set_nu(hyper["nu"]).build())
    sc = (core.IALSSolverConfigBuilder().set_solver_type(getattr(core.SolverType, solver))
          .set_max_cg_steps(hyper["max_cg_steps"]).build())
    # a sample of rank 0's user rows for the row-wise oracle check after the timed region: random rows
    # and the longest ones, their neighbour lists copied out of the device CSR
    parity_rows = None
    if rank == 0 and parity_check is not None and parity_sample > 0 and n_rows > 0:
        grng = torch.Generator(device="cpu").manual_seed(7)
        deg = (ip[1:] - ip[:-1])
        pick = torch.unique(torch.cat([torch.randint(0, n_rows, (parity_sample,), generator=grng),
                                       torch.topk(deg, min(4, n_rows)).indices.cpu()])).tolist()
        lens = [int(ip[r + 1] - ip[r]) for r in pick]
        sub_ip = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        sub_ix = torch.cat([ix[int(ip[r]):int(ip[r + 1])] for r in pick]).cpu().numpy() if sum(lens) else np.zeros(0, np.int32)
        sub_dt = torch.cat([dt[int(ip[r]):int(ip[r + 1])] for r in pick]).cpu().numpy() if sum(lens) else np.zeros(0, np.float32)
        parity_rows = (pick, sps.csr_matrix((sub_dt, sub_ix, sub_ip), shape=(len(pick), I)))
    t0 = time.perf_counter()
    tr = ShardedIALSTrainer(cfg, (ip, ix, dt), int(ub[rank]), U, (t_ip, t_ix, t_dt),
                            int(item_bounds[rank]), I, init_on_device=True)
    del ip, ix, dt, t_ip, t_ix, t_dt
    torch.cuda.empty_cache()
    t_plan = time.perf_counter() - t0

    # ---- device-resident epochs ----
    for _ in range(warmup):
        tr.step_async(sc)
    tr.sync()
    events: list = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = lib.ials_kernel_launch_count()
    barrier()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        tr.step_async(sc, events)
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    tr.sync()  # raises if a solver flagged a failure
    launches = lib.ials_kernel_launch_count() - n0
    ms = max_over_ranks(ev0.elapsed_time(ev1)) / steps
    phases_local = ShardedIALSTrainer.phase_ms(events)
    phases = {k: max_over_ranks(v) for k, v in phases_local.items()}
    phases_min = {k: -max_over_ranks(-v) for k, v in phases_local.items()}

    # ---- end to end with host buffers: own rows down (+ NVLink copies to the peers), one epoch,
    # own rows back ----
    e2e = None
    if e2e_steps > 0:
        host = []
        for side in (0, 1):
            b, e = tr.shard_range(side)
            pin = torch.empty((e - b, K), dtype=torch.float32, pin_memory=True)
            host.append((pin, pin.numpy()))
            tr.get_shard_rows(side, host[side][1])

        def e2e_step() -> None:
            tr.step_io(sc, host[0][0], host[1][0])

        e2e_step()
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        barrier()
        e2e_dt = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": nnz * e2e_steps / e2e_dt, "ms_per_step": 1e3 * e2e_dt / e2e_steps, "steps": e2e_steps,
               "h2d_bytes_per_step": (U + I) * K * 4, "d2h_bytes_per_step": (U + I) * K * 4,
               "what": "ShardedIALSTrainer.step_io on every rank: its OWN user+item rows from pinned host "
                       "(ials_trainer_set_factor_rows; the item rows are pushed to the peers' replicas over "
                       "NVLink, the user rows -- warm starts only -- stay local), one sharded "
                       "epoch, its own rows back (user rows during the item half-epoch); bytes are the sum "
                       "over ranks = each matrix once per direction"}

    # ---- configs[4]: score + seen mask + top-k of a bounded sample of each rank's users ----
    score = None
    n_score = min(score_users_per_rank, n_rows) if score_users_per_rank >= 0 else n_rows
    if n_score > 0:
        k = min(topk, I)
        b0 = int(ub[rank])
        idx = np.empty((score_block, k), dtype=np.int32)
        cnt = np.empty((score_block,), dtype=np.int32)
        m = min(score_block, n_score)
        tr.recommend(b0, b0 + m, k, idx[:m], cnt[:m])  # warm-up (scratch allocation)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in range(b0, b0 + n_score, score_block):
            m = min(score_block, b0 + n_score - b)
            tr.recommend(b, b + m, k, idx[:m], cnt[:m])
        torch.cuda.synchronize()
        dt_score = max_over_ranks(time.perf_counter() - t0)
        scored = sum_over_ranks(n_score)
        score = {"users_scored": scored, "k": k, "n_items": I, "seconds": dt_score,
                 "users_per_s": scored / dt_score,
                 "algorithmic_tflops": 2.0 * scored * I * K / dt_score / 1e12,
                 "full_config_seconds_extrapolated": U / (scored / dt_score),
                 "what": f"ials_trainer_recommend(mask='train', k={k}) over {n_score} of each rank's own users "
                         f"in blocks of {score_block}; host wall clock incl. the D2H of k indices per user, "
                         "max over ranks; users are row-sharded, item factors replicated: no collective"}

    # ---- parity at this size: one more user half-epoch on every rank; rank 0 hands its sampled rows
    # (values before and after, their neighbour lists, the item factors) to ``parity_check`` -- the
    # caller's checker (bench.py / the tools re-solve them with the CPU oracle; this package never
    # imports it).  Collective: every rank passes the same ``parity_check is not None``. ----
    parity = None
    if parity_check is not None and parity_sample > 0:
        import ctypes as _ct

        b0 = int(ub[rank])
        views = [tr._factors_view(0), tr._factors_view(1)]
        before = items_host = gidx = None
        if parity_rows is not None:
            gidx = torch.tensor([b0 + r for r in parity_rows[0]], device=dev)
            before = views[0][gidx, :K].cpu().numpy()
            items_host = views[1][:, :K].cpu().numpy()
        tr._use_current_stream()
        tr._all_reduce(tr._gram_partial(1))
        tr._check(tr._lib.ials_trainer_solve_shard(tr._handle, 0, _ct.byref(core.IALSTrainer._solver(sc))))
        tr.sync()
        if parity_rows is not None:
            after = views[0][gidx, :K].cpu().numpy()
            parity = parity_check(before=before, after=after, other=items_host, rows=parity_rows[1], solver=solver,
                                  hyper=hyper)
    stats = [tr.plan_stats(0), tr.plan_stats(1)] if hasattr(tr, "plan_stats") else None
    del tr
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    algo = 2 * nnz * (4 * K + 8) + (U + I) * 8 * K + (U + I + 2) * 8 + (U + I) * 4 * K
    return {"n_users": U, "n_items": I, "nnz": nnz, "K": K, "world": world, "scale": scale, "solver": solver,
            "ms_per_epoch": ms, "interactions_per_s": nnz / (ms / 1e3), "epochs_per_s": 1e3 / ms,
            "algorithmic_bytes_per_epoch": algo, "achieved_gbs": algo / (ms / 1e3) / 1e9,
            "phases_ms_max_over_ranks": phases, "phases_ms_min_over_ranks": phases_min,
            "nvlink_bytes_per_epoch_per_rank": (U + I) * K * 4 // world * (world - 1) + 2 * K * K * 4 * (world > 1),
            "gpu_launches": int(launches), "build_s": round(t_build, 2), "plan_s": round(t_plan, 2),
            "e2e": e2e, "score_topk": score, "parity_sample": parity, "schedule": stats}


def c4_config_dict(world: int, scale: float = 1.0) -> dict:
    U, I, nnz, K = c4_shape(scale, world)
    return {
        "workload": f"BASELINE configs[3]: iALS epoch on a synthetic power-law matrix {U}x{I}, {nnz} nnz, "
                    f"K={K}, CG max_cg_steps=3, alpha0=0.1, reg=0.001, loss_type=IALSPP, row-sharded "
                    f"across {world} B200 (strong scaling: the matrix is fixed)",
        "n_users": U, "n_items": I, "nnz": nnz, "K": K, "solver": "CG",
        "parallelism": f"row-sharded x{world}: nnz-balanced user/item ranges, full factor replicas, "
                       "solve kernels store solved rows into the peers' replicas (CUDA IPC / NVLink), "
                       "K x K Gram all-reduce (NCCL)",
        "l2": "factor replicas (5.1 + 1.0 GB) and the CSR shards exceed the 126 MB L2; no explicit flush",
    }


def bench_main(args: Any, metric: str, unit: str, hyper: dict, parity_check: Any = None) -> None:
    """``bench.py --gpus N`` for N > 1: BASELINE configs[3] (1 B interactions, 10 M x 2 M, K=128)
    row-sharded over the N GPUs, strong scaling, plus the configs[4] top-100 sample."""
    import torch
    import torch.distributed as dist

    from bench import ClockSampler, measured_peaks

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    scale = float(os.environ.get("IALS_BENCH_C4_SCALE", "1.0"))
    with ClockSampler(local_rank) as clocks:
        res = run_c4(hyper, steps=args.steps, warmup=args.warmup, scale=scale,
                     e2e_steps=max(2, min(args.steps, 3)), parity_check=parity_check)
    if rank == 0:
        peak, peak_kind = measured_peaks()
        e2e = res.pop("e2e")
        line = {
            "metric": metric, "value": res["interactions_per_s"], "unit": unit, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_epoch"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "epochs_per_sec": res["epochs_per_s"],
            "config": c4_config_dict(world, scale), "clocks": clocks.summary(),
            "e2e": {"value": e2e["value"], "unit": unit, "h2d_bytes_per_step": e2e["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": e2e["d2h_bytes_per_step"], "ms_per_step": e2e["ms_per_step"],
                    "steps": e2e["steps"], "what": e2e["what"]},
            "gpu_launches": res["gpu_launches"],
            "roofline": {"bound": "hbm", "kernel": "whole epoch (Gram partials + CG row solves), all ranks",
                         "achieved": res["achieved_gbs"], "peak": peak * world, "peak_kind": peak_kind,
                         "unit": "GB/s", "frac": res["achieved_gbs"] / (peak * world), "traffic": None,
                         "algorithmic_bytes_per_epoch": res["algorithmic_bytes_per_epoch"]},
            "phases_ms_per_epoch": {"max_over_ranks": res["phases_ms_max_over_ranks"],
                                    "min_over_ranks": res["phases_ms_min_over_ranks"]},
            "nvlink_bytes_per_epoch_per_rank": res["nvlink_bytes_per_epoch_per_rank"],
            "parity_sample": res.get("parity_sample"),
            "topk_configs4": res["score_topk"],
            "setup_s": {"build_shards": res["build_s"], "plan": res["plan_s"]},
        }
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()
