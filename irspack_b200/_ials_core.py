"""B200-native stand-in for ``irspack.recommenders._ials_core``.

Same names, argument meaning and error behaviour as the reference's nanobind
module (/root/reference/cpp_source/als/wrapper.cpp:17-182; type stubs in
src/irspack/recommenders/_ials_core.pyi), but every operation runs in
hand-written sm_100a CUDA behind the C ABI of ``include/ials_b200.h``.
Factors live on the GPU; the ``user`` / ``item`` properties return host copies.

The feature-aware overloads (wrapper.cpp:133-136, 144-155, 160-161) run on the generic device
kernels (csrc/feature.cu, cg.cu, cholesky_tile.cu).  Not implemented (``NotImplementedError``):
``SolverType.IALSPP`` with subspace blocks of more than 256 dimensions.
"""
from __future__ import annotations

import ctypes
import enum
import os
import types
from typing import Any, NamedTuple, Optional, Tuple

import numpy as np
import scipy.sparse as sps

from . import _lib
from ._lib import ModelConfigStruct, SolverConfigStruct, check, lib


class LossType(enum.Enum):  # wrapper.cpp:25-27
    ORIGINAL = 0
    IALSPP = 1


class SolverType(enum.Enum):  # wrapper.cpp:29-32
    CHOLESKY = 0
    CG = 1
    IALSPP = 2


# legacy module-level aliases, wrapper.cpp:37-40 (IALSPP resolves to SolverType.IALSPP)
ORIGINAL = LossType.ORIGINAL
CHOLESKY = SolverType.CHOLESKY
CG = SolverType.CG
IALSPP = SolverType.IALSPP


class IALSModelConfig:  # wrapper.cpp:42-71
    def __init__(self, K: int, alpha0: float, reg: float, nu: float, init_stdev: float,
                 random_seed: int, loss_type: LossType, lambda_user_feature: float = 0.0,
                 lambda_item_feature: float = 0.0, feature_warmup_epochs: int = 0) -> None:
        if not isinstance(loss_type, LossType):
            raise TypeError("loss_type must be a LossType")
        if int(K) < 0 or int(feature_warmup_epochs) < 0:
            raise TypeError("K and feature_warmup_epochs are unsigned")  # size_t in the reference
        self.K = int(K)
        self.alpha0 = float(alpha0)
        self.reg = float(reg)
        self.nu = float(nu)
        self.init_stdev = float(init_stdev)
        self.random_seed = int(random_seed)
        self.loss_type = loss_type
        self.lambda_user_feature = float(lambda_user_feature)
        self.lambda_item_feature = float(lambda_item_feature)
        self.feature_warmup_epochs = int(feature_warmup_epochs)

    def __getstate__(self) -> Tuple[Any, ...]:
        return (self.K, self.alpha0, self.reg, self.nu, self.init_stdev, self.random_seed,
                self.loss_type, self.lambda_user_feature, self.lambda_item_feature,
                self.feature_warmup_epochs)

    def __setstate__(self, state: Tuple[Any, ...]) -> None:
        self.__init__(*state)  # type: ignore[misc]

    def _as_struct(self) -> ModelConfigStruct:
        return ModelConfigStruct(self.K, self.alpha0, self.reg, self.nu, self.init_stdev,
                                 self.random_seed, self.loss_type.value)


class IALSModelConfigBuilder:  # wrapper.cpp:72-90, defaults IALSLearningConfig.hpp:33-43
    def __init__(self) -> None:
        self.reg = 0.1
        self.alpha0 = 0.1
        self.nu = 1.0
        self.init_stdev = 0.1
        self.K = 16
        self.random_seed = 42
        self.loss_type = LossType.IALSPP
        self.lambda_user_feature = 0.0
        self.lambda_item_feature = 0.0
        self.feature_warmup_epochs = 0

    def build(self) -> IALSModelConfig:
        return IALSModelConfig(self.K, self.alpha0, self.reg, self.nu, self.init_stdev,
                               self.random_seed, self.loss_type, self.lambda_user_feature,
                               self.lambda_item_feature, self.feature_warmup_epochs)

    def set_K(self, K: int) -> "IALSModelConfigBuilder":
        self.K = K
        return self

    def set_alpha0(self, alpha0: float) -> "IALSModelConfigBuilder":
        self.alpha0 = alpha0
        return self

    def set_reg(self, reg: float) -> "IALSModelConfigBuilder":
        self.reg = reg
        return self

    def set_nu(self, nu: float) -> "IALSModelConfigBuilder":
        self.nu = nu
        return self

    def set_init_stdev(self, init_stdev: float) -> "IALSModelConfigBuilder":
        self.init_stdev = init_stdev
        return self

    def set_random_seed(self, random_seed: int) -> "IALSModelConfigBuilder":
        self.random_seed = random_seed
        return self

    def set_loss_type(self, loss_type: LossType) -> "IALSModelConfigBuilder":
        self.loss_type = loss_type
        return self

    def set_lambda_user_feature(self, value: float) -> "IALSModelConfigBuilder":
        self.lambda_user_feature = value
        return self

    def set_lambda_item_feature(self, value: float) -> "IALSModelConfigBuilder":
        self.lambda_item_feature = value
        return self

    def set_feature_warmup_epochs(self, value: int) -> "IALSModelConfigBuilder":
        self.feature_warmup_epochs = value
        return self


class IALSSolverConfig:  # wrapper.cpp:92-115
    def __init__(self, n_threads: int, solver_type: SolverType, max_cg_steps: int,
                 ialspp_subspace_dimension: int, ialspp_iteration: int) -> None:
        if not isinstance(solver_type, SolverType):
            raise TypeError("solver_type must be a SolverType")
        for v in (n_threads, max_cg_steps, ialspp_subspace_dimension, ialspp_iteration):
            if int(v) < 0:
                raise TypeError("solver config fields are unsigned (size_t in the reference)")
        self.n_threads = int(n_threads)
        self.solver_type = solver_type
        self.max_cg_steps = int(max_cg_steps)
        self.ialspp_subspace_dimension = int(ialspp_subspace_dimension)
        self.ialspp_iteration = int(ialspp_iteration)

    def __getstate__(self) -> Tuple[Any, ...]:
        return (self.n_threads, self.solver_type, self.max_cg_steps,
                self.ialspp_subspace_dimension, self.ialspp_iteration)

    def __setstate__(self, state: Tuple[Any, ...]) -> None:
        self.__init__(*state)  # type: ignore[misc]

    def _as_struct(self) -> SolverConfigStruct:
        return SolverConfigStruct(self.n_threads, self.solver_type.value, 0, self.max_cg_steps,
                                  self.ialspp_subspace_dimension, self.ialspp_iteration)


class IALSSolverConfigBuilder:  # wrapper.cpp:117-128, defaults IALSLearningConfig.hpp:114-120
    def __init__(self) -> None:
        self.n_threads = 1
        self.solver_type = SolverType.CG
        self.max_cg_steps = 3
        self.ialspp_subspace_dimension = 64
        self.ialspp_iteration = 1

    def build(self) -> IALSSolverConfig:
        return IALSSolverConfig(self.n_threads, self.solver_type, self.max_cg_steps,
                                self.ialspp_subspace_dimension, self.ialspp_iteration)

    def set_n_threads(self, n_threads: int) -> "IALSSolverConfigBuilder":
        self.n_threads = n_threads
        return self

    def set_solver_type(self, solver_type: SolverType) -> "IALSSolverConfigBuilder":
        self.solver_type = solver_type
        return self

    def set_max_cg_steps(self, max_cg_steps: int) -> "IALSSolverConfigBuilder":
        self.max_cg_steps = max_cg_steps
        return self

    def set_ialspp_subspace_dimension(self, v: int) -> "IALSSolverConfigBuilder":
        self.ialspp_subspace_dimension = v
        return self

    def set_ialspp_iteration(self, v: int) -> "IALSSolverConfigBuilder":
        self.ialspp_iteration = v
        return self


def _ptr(a: Optional[np.ndarray]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0) if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _canonical_csr(X: Any) -> sps.csr_matrix:
    """float32 CSR with sorted, duplicate-free indices (what Eigen receives)."""
    if not sps.issparse(X):
        raise TypeError("interaction must be a scipy sparse matrix")
    X = sps.csr_matrix(X, dtype=np.float32, copy=True)
    X.sum_duplicates()
    X.sort_indices()
    return X


def _csr_arrays(X: sps.csr_matrix) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    return (np.ascontiguousarray(X.indptr, dtype=np.int64),
            np.ascontiguousarray(X.indices, dtype=np.int32),
            np.ascontiguousarray(X.data, dtype=np.float32))


def _feature_arrays(F: Any) -> Tuple[int, int, Optional[np.ndarray], Optional[np.ndarray],
                                     Optional[np.ndarray], Optional[np.ndarray]]:
    """(rows, cols, dense, indptr, indices, data) of a FeatureMatrix (dense float32 row-major
    or CSR; the reference's std::variant<SparseMatrix, DenseMatrix>, IALSTrainer.hpp:684-702)."""
    if sps.issparse(F):
        C = sps.csr_matrix(F, dtype=np.float32, copy=True)
        C.sum_duplicates()
        C.sort_indices()
        ip, ix, dt = _csr_arrays(C)
        return int(C.shape[0]), int(C.shape[1]), None, ip, ix, dt
    D = np.ascontiguousarray(F, dtype=np.float32)
    if D.ndim != 2:
        raise TypeError("a feature matrix must be 2-dimensional")
    return int(D.shape[0]), int(D.shape[1]), D, None, None, None


def _current_device_and_stream() -> Tuple[int, int]:
    """Device / stream the work goes to: torch's current ones when torch drives
    the process (PyTorch is the device-memory and stream plumbing), else
    ``$IALS_B200_DEVICE`` (default 0) and the legacy default stream."""
    env = os.environ.get("IALS_B200_DEVICE")
    try:
        import torch

        if torch.cuda.is_available():
            dev = int(env) if env is not None else torch.cuda.current_device()
            return dev, int(torch.cuda.current_stream(dev).cuda_stream)
    except ImportError:  # pragma: no cover
        pass
    return (int(env) if env is not None else 0), 0


def _stream_of(device: int) -> int:
    """torch's current stream ON ``device`` (0 = the legacy default stream without torch)."""
    try:
        import torch

        if torch.cuda.is_available():
            return int(torch.cuda.current_stream(device).cuda_stream)
    except ImportError:  # pragma: no cover
        pass
    return 0


def _device_view(ptr: int, shape: Tuple[int, ...], strides: Tuple[int, ...], device: int,
                 typestr: str = "<f4") -> Any:
    """Zero-copy torch view of library-owned memory on ``cuda:device`` (``strides`` in bytes)."""
    import torch

    carrier = types.SimpleNamespace(__cuda_array_interface__={
        "shape": shape, "typestr": typestr, "data": (ptr, False), "version": 3, "strides": strides})
    return torch.as_tensor(carrier, device=f"cuda:{device}")


def _transform(handle: ctypes.c_void_p, K: int, device: int, side: int, interaction: Any,
               sc: SolverConfigStruct) -> np.ndarray:
    """``ials_trainer_transform`` of a trainer (or a row-sharded trainer's replicas) on its device's
    current stream: the fold-in of a host CSR, returned as host rows [n_new, K]."""
    X = _canonical_csr(interaction)
    indptr, indices, data = _csr_arrays(X)
    n_new = X.shape[0] if side == 0 else X.shape[1]
    out = np.empty((n_new, K), dtype=np.float32)
    check(lib.ials_trainer_set_stream(handle, ctypes.c_void_p(_stream_of(device))))
    check(lib.ials_trainer_transform(handle, side, X.shape[0], X.shape[1], _ptr(indptr), _ptr(indices),
                                     _ptr(data), ctypes.byref(sc), _ptr(out)))
    return out


_SIMILARITY_METRICS = {"dot": 0, "cosine": 1}  # IALS_SIMILARITY_DOT / IALS_SIMILARITY_COSINE


def _allowed_arrays(allowed: Any) -> Tuple[int, Optional[np.ndarray], Optional[np.ndarray]]:
    """``(n_lists, indptr, indices)`` allow-lists as the C ABI takes them (``None``: no list)."""
    if allowed is None:
        return 0, None, None
    n_lists, a_indptr, a_indices = allowed
    ai = np.ascontiguousarray(a_indptr, dtype=np.int64)
    ax = np.ascontiguousarray(a_indices, dtype=np.int32)
    if ai.shape != (int(n_lists) + 1,) or (ai.size and int(ai[-1]) != ax.size):
        raise ValueError("allowed = (n_lists, indptr[n_lists + 1], indices[indptr[-1]])")
    return int(n_lists), ai, ax


def _similar(handle: ctypes.c_void_p, device: int, n_side: int, side: int, indices: Any, cutoff: int,
             metric: str, exclude_self: bool, forbidden: Any, allowed: Any, return_scores: bool):
    """``ials_trainer_similar`` of a trainer (or a row-sharded trainer's replicas) on its device's current
    stream.  ``indices``: None (every row of the side), a ``range`` of step 1, or row indices."""
    if side not in (0, 1):
        raise ValueError("side must be 0 or 1")
    if metric not in _SIMILARITY_METRICS:
        raise ValueError("metric must be 'cosine' or 'dot'")
    cutoff = int(cutoff)
    if not 1 <= cutoff <= n_side:
        raise ValueError("cutoff must be in [1, rows of the side]")
    q = None
    if indices is None:
        begin, end = 0, n_side
    elif isinstance(indices, range):
        if indices.step != 1 or not 0 <= indices.start <= indices.stop <= n_side:
            raise ValueError("bad query block")
        begin, end = indices.start, indices.stop
    else:
        q = np.ascontiguousarray(indices, dtype=np.int64).reshape(-1)
        begin, end = 0, q.size
    rows = end - begin
    fi = fx = None
    if forbidden is not None:
        f = sps.csr_matrix(forbidden, copy=True)
        if f.shape != (rows, n_side):
            raise ValueError("forbidden has the wrong shape")
        f.eliminate_zeros()  # a stored zero forbids nothing, as in the recommend masks
        fi = np.ascontiguousarray(f.indptr, dtype=np.int64)
        fx = np.ascontiguousarray(f.indices, dtype=np.int32)
    n_lists, ai, ax = _allowed_arrays(allowed)
    idx = np.empty((rows, cutoff), dtype=np.int32)
    cnt = np.empty((rows,), dtype=np.int32)
    sc = np.empty((rows, cutoff), dtype=np.float32) if return_scores else None
    check(lib.ials_trainer_set_stream(handle, ctypes.c_void_p(_stream_of(device))))
    check(lib.ials_trainer_similar(handle, side, _ptr(q), begin, end, cutoff, _SIMILARITY_METRICS[metric],
                                   int(bool(exclude_self)), _ptr(fi), _ptr(fx), n_lists, _ptr(ai), _ptr(ax),
                                   _ptr(idx), _ptr(sc), _ptr(cnt)))
    return (idx, cnt, sc) if return_scores else (idx, cnt)


def _mask_arrays(mask: Any, rows: int, n_items: int) -> Tuple[int, Optional[np.ndarray], Optional[np.ndarray]]:
    """``(mask_mode, indptr, indices)`` of a list request's mask: "train" (0), None (1) or a sparse matrix
    with one row per query (2; stored zeros dropped, as scipy's ``.nonzero()`` drops them, evaluator.py:432)."""
    if isinstance(mask, str):
        if mask != "train":
            raise ValueError("mask must be 'train', None or a sparse matrix")
        return 0, None, None
    if mask is None:
        return 1, None, None
    m = sps.csr_matrix(mask)
    if m.shape != (rows, n_items):
        raise ValueError("mask has the wrong shape")
    m = sps.csr_matrix(m, copy=True)
    m.eliminate_zeros()
    m.sort_indices()
    return 2, np.ascontiguousarray(m.indptr, dtype=np.int64), np.ascontiguousarray(m.indices, dtype=np.int32)


def _candidate_lists(candidates: Any, rows: int, n_items: int,
                     rank: bool = True) -> Tuple[int, np.ndarray, np.ndarray]:
    """``(n_lists, indptr, indices)`` of candidate items given as ``(n_lists, indptr, indices)`` (the
    format of ``allowed``) or as a sequence of index lists: one list shared by every query row or one
    per row.  Ids must lie in ``[0, n_items)``.  ``rank``: each list is sorted and its repeats dropped
    (the strictly ascending lists the ranking takes); otherwise the lists are kept as given."""
    if isinstance(candidates, tuple) and len(candidates) == 3 and np.isscalar(candidates[0]):
        n_lists = int(candidates[0])
        ip = np.ascontiguousarray(candidates[1], dtype=np.int64).reshape(-1)
        ix = np.asarray(candidates[2]).reshape(-1)
        if (ip.shape != (n_lists + 1,) or ip[0] != 0 or np.any(np.diff(ip) < 0) or int(ip[-1]) != ix.size):
            raise ValueError("candidates = (n_lists, indptr[n_lists + 1], indices[indptr[-1]])")
    else:
        lists = [np.asarray(x).reshape(-1) for x in candidates]
        n_lists = len(lists)
        ip = np.zeros(n_lists + 1, dtype=np.int64)
        np.cumsum([x.size for x in lists], out=ip[1:])
        ix = np.concatenate([x for x in lists if x.size]) if ip[-1] else np.empty(0, dtype=np.int64)
    if n_lists != rows and n_lists != 1:
        raise ValueError("candidates: one shared list or one list per row")
    if ix.size and not np.issubdtype(ix.dtype, np.integer):
        raise ValueError("candidate item ids must be integers")
    # int32 lists to be ranked are range-checked by their first and last ids once sorted (one id per
    # list instead of every id); anything else before the cast, which could wrap
    full_check = ix.dtype != np.int32 or not rank
    if full_check and ix.size and (ix.min() < 0 or ix.max() >= n_items):
        raise ValueError("candidate item out of range")
    ix = np.ascontiguousarray(ix, dtype=np.int32)
    if rank and ix.size > 1:
        ascending = ix[1:] > ix[:-1]
        starts = ip[1:-1]
        ascending[starts[(starts > 0) & (starts < ix.size)] - 1] = True  # a list's first id follows another list
        if not ascending.all():
            row = np.repeat(np.arange(n_lists, dtype=np.int64), np.diff(ip))
            order = np.lexsort((ix, row))
            ix, row = ix[order], row[order]
            keep = np.ones(ix.size, dtype=bool)
            keep[1:] = (ix[1:] != ix[:-1]) | (row[1:] != row[:-1])
            ix, row = np.ascontiguousarray(ix[keep]), row[keep]
            ip = np.zeros(n_lists + 1, dtype=np.int64)
            np.cumsum(np.bincount(row, minlength=n_lists), out=ip[1:])
    if not full_check and ix.size:
        filled = ip[1:] > ip[:-1]
        if ix[ip[:-1][filled]].min() < 0 or ix[ip[1:][filled] - 1].max() >= n_items:
            raise ValueError("candidate item out of range")
    return n_lists, ip, ix


def _query_block(users: Any, n_users: int) -> Tuple[Optional[np.ndarray], int, int]:
    """``(user_idx, begin, end)`` of users given as a ``range`` of step 1 or as indices."""
    if isinstance(users, range):
        if users.step != 1 or not 0 <= users.start <= users.stop <= n_users:
            raise ValueError("bad user block")
        return None, users.start, users.stop
    u = np.ascontiguousarray(users, dtype=np.int64).reshape(-1)
    return u, 0, u.size


def _rank_candidates(handle: ctypes.c_void_p, device: int, n_users: int, n_items: int, K: int, users: Any,
                     embeddings: Any, candidates: Any, cutoff: int, mask: Any, return_scores: bool):
    """``ials_trainer_rank_candidates`` of a trainer (or a row-sharded trainer's replicas) on its device's
    current stream.  Queries: ``users`` (a step-1 ``range`` or indices) or, when it is None, the host rows
    ``embeddings`` [n, K]."""
    cutoff = int(cutoff)
    if not 1 <= cutoff <= min(1024, n_items):
        raise ValueError("cutoff must be in [1, min(1024, n_items)]")
    emb = None
    if users is None:
        emb = np.ascontiguousarray(embeddings, dtype=np.float32)
        if emb.ndim != 2 or emb.shape[1] != K:
            raise ValueError("embedding must be (n, n_components)")
        if isinstance(mask, str):
            raise ValueError("embeddings have no training rows: mask must be None or a sparse matrix")
        q, begin, end = None, 0, emb.shape[0]
    else:
        q, begin, end = _query_block(users, n_users)
    rows = end - begin
    mode, mi, mx = _mask_arrays(mask, rows, n_items)
    n_lists, ci, cx = _candidate_lists(candidates, rows, n_items)
    idx = np.empty((rows, cutoff), dtype=np.int32)
    cnt = np.empty((rows,), dtype=np.int32)
    sc = np.empty((rows, cutoff), dtype=np.float32) if return_scores else None
    check(lib.ials_trainer_set_stream(handle, ctypes.c_void_p(_stream_of(device))))
    check(lib.ials_trainer_rank_candidates(handle, _ptr(q), _ptr(emb), begin, end, cutoff, mode, _ptr(mi), _ptr(mx),
                                           n_lists, _ptr(ci), _ptr(cx), _ptr(idx), _ptr(sc), _ptr(cnt)))
    return (idx, cnt, sc) if return_scores else (idx, cnt)


def _candidate_scores(handle: ctypes.c_void_p, device: int, n_users: int, n_items: int, users: Any,
                      candidates: Any) -> np.ndarray:
    """``ials_trainer_candidate_scores``: the scores of every (row, candidate) pair, float32 in the order
    of the candidate lists (a shared list counts once per row)."""
    q, begin, end = _query_block(users, n_users)
    rows = end - begin
    n_lists, ci, cx = _candidate_lists(candidates, rows, n_items, rank=False)
    if n_lists != rows:  # one shared list: repeated for every row
        ci = np.arange(rows + 1, dtype=np.int64) * cx.size
        cx = np.tile(cx, rows)
    out = np.empty(cx.size, dtype=np.float32)
    check(lib.ials_trainer_set_stream(handle, ctypes.c_void_p(_stream_of(device))))
    check(lib.ials_trainer_candidate_scores(handle, _ptr(q), None, begin, end, _ptr(ci), _ptr(cx), _ptr(out)))
    return out


class Explanation(NamedTuple):
    """Explanations of (query row, target) pairs, pairs in target-list order: the pairs of query row r
    are ``indptr[r]:indptr[r + 1]``.  Per pair: ``score`` = y_t . x_u, ``prior`` = reg_u w_t . prior_u
    (0 without a feature prior), the best history entries as column ids ``indices`` [pairs, n_top]
    (padded with -1) and their ``contributions`` (bias + c_j) w_t . y_j (padded with -inf), ordered by
    (-contribution, column id), and ``counts`` = min(n_top, history length).  With every entry listed,
    the contributions plus the prior add up to the score."""
    indptr: np.ndarray
    score: np.ndarray
    prior: np.ndarray
    indices: np.ndarray
    contributions: np.ndarray
    counts: np.ndarray


def _target_lists(targets: Any, rows: int, n_other: int) -> Tuple[np.ndarray, np.ndarray]:
    """``(indptr, indices)`` of one target list per query row, given as a tuple of two arrays
    ``(indptr, indices)`` or as a sequence of index lists (any order, repeats allowed)."""
    if isinstance(targets, tuple) and len(targets) == 2 and all(isinstance(x, np.ndarray) for x in targets):
        ip = np.ascontiguousarray(targets[0], dtype=np.int64).reshape(-1)
        ix = np.asarray(targets[1]).reshape(-1)
        if ip.shape != (rows + 1,) or ip[0] != 0 or np.any(np.diff(ip) < 0) or int(ip[-1]) != ix.size:
            raise ValueError("targets = (indptr[rows + 1], indices[indptr[-1]])")
    else:
        lists = [np.asarray(x).reshape(-1) for x in targets]
        if len(lists) != rows:
            raise ValueError("targets: one list per query row")
        ip = np.zeros(rows + 1, dtype=np.int64)
        np.cumsum([x.size for x in lists], out=ip[1:])
        ix = np.concatenate([x for x in lists if x.size]) if ip[-1] else np.empty(0, dtype=np.int64)
    if ix.size and not np.issubdtype(ix.dtype, np.integer):
        raise ValueError("target ids must be integers")
    if ix.size and (ix.min() < 0 or ix.max() >= n_other):
        raise ValueError("target id out of range")
    return ip, np.ascontiguousarray(ix, dtype=np.int32)


def _explain(handle: ctypes.c_void_p, device: int, n_rows: Tuple[int, int], side: int, indices: Any, X: Any,
             targets: Any, n_top: int) -> Explanation:
    """``ials_trainer_explain`` of a trainer (or a row-sharded trainer's replicas) on its device's current
    stream.  Queries: ``indices`` (a step-1 ``range`` or row indices of ``side``) or, when ``X`` is given,
    its rows as cold histories over the other side (every stored entry counts, as given)."""
    if side not in (0, 1):
        raise ValueError("side must be 0 or 1")
    n_side, n_other = n_rows[side], n_rows[1 - side]
    n_top = int(n_top)
    if not 1 <= n_top <= 1024:
        raise ValueError("n_top must be in [1, 1024]")
    hi = hx = hd = None
    if X is None:
        q, begin, end = _query_block(indices, n_side)
    else:
        if not sps.issparse(X):
            raise TypeError("X must be a scipy sparse matrix")
        Xc = sps.csr_matrix(X)
        if Xc.shape[1] != n_other:
            raise ValueError("X must have one column per row of the other side")
        hi, hx, hd = _csr_arrays(Xc)
        q, begin, end = None, 0, Xc.shape[0]
    rows = end - begin
    ip, ix = _target_lists(targets, rows, n_other)
    pairs = ix.size
    score = np.empty(pairs, dtype=np.float32)
    prior = np.empty(pairs, dtype=np.float32)
    idx = np.empty((pairs, n_top), dtype=np.int32)
    contrib = np.empty((pairs, n_top), dtype=np.float32)
    cnt = np.empty(pairs, dtype=np.int32)
    check(lib.ials_trainer_set_stream(handle, ctypes.c_void_p(_stream_of(device))))
    check(lib.ials_trainer_explain(handle, side, _ptr(q), begin, end, _ptr(hi), _ptr(hx), _ptr(hd), _ptr(ip),
                                   _ptr(ix), n_top, _ptr(score), _ptr(prior), _ptr(idx), _ptr(contrib),
                                   _ptr(cnt)))
    return Explanation(ip, score, prior, idx, contrib, cnt)


def _factors_device(handle: ctypes.c_void_p, side: int, device: int) -> Any:
    """Zero-copy view ([n, K], row stride ld) of a trainer's factor matrix (or replica) of ``side``."""
    import torch

    p, n, K, ld = ctypes.c_void_p(0), ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
    check(lib.ials_trainer_factors_device(handle, side, ctypes.byref(p), ctypes.byref(n), ctypes.byref(K),
                                          ctypes.byref(ld)))
    if n.value == 0:
        return torch.empty((0, K.value), dtype=torch.float32, device=f"cuda:{device}")
    return _device_view(int(p.value), (int(n.value), int(ld.value)), (int(ld.value) * 4, 4), device)[:, : K.value]


class IALSTrainer:
    """``_ials_core.IALSTrainer`` (wrapper.cpp:130-181) on one B200."""

    def __init__(self, model_config: IALSModelConfig, interaction: Any,
                 user_feature: Any = None, item_feature: Any = None) -> None:
        if (user_feature is None) != (item_feature is None):
            raise TypeError("the feature-aware constructor takes both user_feature and item_feature "
                            "(wrapper.cpp:133-136); pass a matrix with 0 columns for a side without features")
        if not isinstance(model_config, IALSModelConfig):
            raise TypeError("model_config must be an IALSModelConfig")
        X = _canonical_csr(interaction)
        self._config = model_config
        self._handle = ctypes.c_void_p(0)
        self._cache: dict = {}
        self.n_users, self.n_items = int(X.shape[0]), int(X.shape[1])
        self.K = model_config.K
        self._device, stream = _current_device_and_stream()
        indptr, indices, data = _csr_arrays(X)
        cfg = model_config._as_struct()
        h = ctypes.c_void_p(0)
        check(lib.ials_trainer_create(ctypes.byref(cfg), self.n_users, self.n_items, _ptr(indptr),
                                      _ptr(indices), _ptr(data), self._device, ctypes.byref(h)))
        self._handle = h
        check(lib.ials_trainer_set_stream(self._handle, ctypes.c_void_p(stream)))
        if user_feature is not None:  # feature-aware model, IALSTrainer.hpp:722-743
            lams = (model_config.lambda_user_feature, model_config.lambda_item_feature)
            for side, F in enumerate((user_feature, item_feature)):
                rows, cols, dense, ip, ix, dt = _feature_arrays(F)
                check(lib.ials_trainer_set_features(self._handle, side, rows, cols, _ptr(dense), _ptr(ip),
                                                    _ptr(ix), _ptr(dt), ctypes.c_float(lams[side]),
                                                    int(model_config.feature_warmup_epochs)))

    # -- construction from pickled state (IALSTrainer.hpp:745-756) --
    @classmethod
    def _from_factors(cls, config: IALSModelConfig, user: np.ndarray, item: np.ndarray) -> "IALSTrainer":
        self = cls.__new__(cls)
        self._config = config
        self._handle = ctypes.c_void_p(0)
        self._cache = {}
        user = np.ascontiguousarray(user, dtype=np.float32)
        item = np.ascontiguousarray(item, dtype=np.float32)
        if user.ndim != 2 or item.ndim != 2 or user.shape[1] != item.shape[1]:
            raise ValueError("inconsistent factor shapes")
        self.n_users, self.n_items, self.K = user.shape[0], item.shape[0], user.shape[1]
        cfg = config._as_struct()
        cfg.K = self.K
        self._device, stream = _current_device_and_stream()
        h = ctypes.c_void_p(0)
        check(lib.ials_trainer_create_from_factors(ctypes.byref(cfg), self.n_users, self.n_items,
                                                   _ptr(user), _ptr(item), self._device,
                                                   ctypes.byref(h)))
        self._handle = h
        check(lib.ials_trainer_set_stream(self._handle, ctypes.c_void_p(stream)))
        return self

    def __del__(self) -> None:
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            lib.ials_trainer_destroy(h)
            self._handle = ctypes.c_void_p(0)

    def _use_current_stream(self) -> None:
        # the stream must belong to the trainer's OWN device: torch's current device (or
        # $IALS_B200_DEVICE) may be another GPU in a process that drives several
        check(lib.ials_trainer_set_stream(self._handle, ctypes.c_void_p(_stream_of(self._device))))

    @staticmethod
    def _solver(solver_config: IALSSolverConfig) -> SolverConfigStruct:
        if not isinstance(solver_config, IALSSolverConfig):
            raise TypeError("solver_config must be an IALSSolverConfig")
        return solver_config._as_struct()

    # -- reference API --
    def step(self, solver_config: IALSSolverConfig) -> None:  # wrapper.cpp:137
        sc = self._solver(solver_config)
        self._cache.clear()
        self._use_current_stream()
        check(lib.ials_trainer_step(self._handle, ctypes.byref(sc)))

    def user_scores(self, begin: int, end: int, solver_config: IALSSolverConfig) -> np.ndarray:
        sc = self._solver(solver_config)  # wrapper.cpp:138-139
        if begin < 0 or end < 0:
            raise TypeError("begin / end are unsigned (size_t in the reference)")
        rows = max(int(end) - int(begin), 0)
        out = np.empty((rows, self.n_items), dtype=np.float32)
        self._use_current_stream()
        check(lib.ials_trainer_user_scores(self._handle, int(begin), int(end), ctypes.byref(sc),
                                           _ptr(out)))
        return out

    def _transform(self, side: int, interaction: Any, solver_config: IALSSolverConfig) -> np.ndarray:
        return _transform(self._handle, self.K, self._device, side, interaction, self._solver(solver_config))

    def transform_user(self, interaction: Any, solver_config: IALSSolverConfig) -> np.ndarray:
        return self._transform(0, interaction, solver_config)  # wrapper.cpp:140-141

    def transform_item(self, interaction: Any, solver_config: IALSSolverConfig) -> np.ndarray:
        return self._transform(1, interaction, solver_config)  # wrapper.cpp:142-143

    def _transform_with_feature(self, side: int, interaction: Any, feature: Any,
                                solver_config: IALSSolverConfig) -> np.ndarray:
        sc = self._solver(solver_config)
        X = _canonical_csr(interaction)
        indptr, indices, data = _csr_arrays(X)
        rows, cols, dense, ip, ix, dt = _feature_arrays(feature)
        n_new = X.shape[0] if side == 0 else X.shape[1]
        out = np.empty((n_new, self.K), dtype=np.float32)
        self._use_current_stream()
        check(lib.ials_trainer_transform_with_feature(
            self._handle, side, X.shape[0], X.shape[1], _ptr(indptr), _ptr(indices), _ptr(data), rows, cols,
            _ptr(dense), _ptr(ip), _ptr(ix), _ptr(dt), ctypes.byref(sc), _ptr(out)))
        return out

    def transform_user_with_feature(self, interaction: Any, feature: Any,
                                    solver_config: IALSSolverConfig) -> np.ndarray:  # wrapper.cpp:144-147
        return self._transform_with_feature(0, interaction, feature, solver_config)

    def transform_item_with_feature(self, interaction: Any, feature: Any,
                                    solver_config: IALSSolverConfig) -> np.ndarray:  # wrapper.cpp:148-151
        return self._transform_with_feature(1, interaction, feature, solver_config)

    def _transform_feature(self, side: int, feature: Any) -> np.ndarray:
        rows, cols, dense, ip, ix, dt = _feature_arrays(feature)
        out = np.empty((rows, self.K), dtype=np.float32)
        self._use_current_stream()
        check(lib.ials_trainer_transform_feature(self._handle, side, rows, cols, _ptr(dense), _ptr(ip),
                                                 _ptr(ix), _ptr(dt), _ptr(out)))
        return out

    def transform_user_feature(self, feature: Any) -> np.ndarray:  # wrapper.cpp:152-153
        return self._transform_feature(0, feature)

    def transform_item_feature(self, feature: Any) -> np.ndarray:  # wrapper.cpp:154-155
        return self._transform_feature(1, feature)

    def compute_loss(self, solver_config: IALSSolverConfig) -> float:  # wrapper.cpp:156-157
        sc = self._solver(solver_config)
        out = ctypes.c_float(0)
        self._use_current_stream()
        check(lib.ials_trainer_compute_loss(self._handle, ctypes.byref(sc), ctypes.byref(out)))
        return float(out.value)

    def _get(self, side: int) -> np.ndarray:
        if side not in self._cache:
            n = self.n_users if side == 0 else self.n_items
            out = np.empty((n, self.K), dtype=np.float32)
            self._use_current_stream()
            check(lib.ials_trainer_get_factors(self._handle, side, _ptr(out)))
            # a host copy of device-resident factors: in-place edits would silently diverge from
            # the device, so they fail loudly -- assign through the setter instead
            out.flags.writeable = False
            self._cache[side] = out
        return self._cache[side]

    def _set(self, side: int, value: np.ndarray) -> None:
        n = self.n_users if side == 0 else self.n_items
        value = np.ascontiguousarray(value, dtype=np.float32)
        if value.shape != (n, self.K):
            raise ValueError(f"expected a ({n}, {self.K}) matrix, got {value.shape}")
        self._cache.pop(side, None)
        self._use_current_stream()
        check(lib.ials_trainer_set_factors(self._handle, side, _ptr(value)))

    @property
    def user(self) -> np.ndarray:  # wrapper.cpp:158
        return self._get(0)

    @user.setter
    def user(self, value: np.ndarray) -> None:
        self._set(0, value)

    @property
    def item(self) -> np.ndarray:  # wrapper.cpp:159
        return self._get(1)

    @item.setter
    def item(self, value: np.ndarray) -> None:
        self._set(1, value)

    def _get_feature_weight(self, side: int) -> np.ndarray:
        n = ctypes.c_int64(0)
        check(lib.ials_trainer_feature_weight_rows(self._handle, side, ctypes.byref(n)))
        out = np.zeros((int(n.value), self.K), dtype=np.float32)
        if n.value:
            self._use_current_stream()
            check(lib.ials_trainer_get_feature_weight(self._handle, side, _ptr(out)))
        return out

    def _set_feature_weight(self, side: int, value: np.ndarray) -> None:
        value = np.ascontiguousarray(value, dtype=np.float32)
        if value.ndim != 2 or (value.shape[0] and value.shape[1] != self.K):
            raise ValueError(f"expected an (n, {self.K}) matrix, got {value.shape}")
        self._use_current_stream()
        check(lib.ials_trainer_set_feature_weight(self._handle, side, int(value.shape[0]), _ptr(value)))

    @property
    def user_feature_weight(self) -> np.ndarray:  # wrapper.cpp:160 (no features: 0 x K)
        return self._get_feature_weight(0)

    @user_feature_weight.setter
    def user_feature_weight(self, value: np.ndarray) -> None:
        self._set_feature_weight(0, value)

    @property
    def item_feature_weight(self) -> np.ndarray:  # wrapper.cpp:161
        return self._get_feature_weight(1)

    @item_feature_weight.setter
    def item_feature_weight(self, value: np.ndarray) -> None:
        self._set_feature_weight(1, value)

    def __getstate__(self) -> Tuple[Any, ...]:  # wrapper.cpp:162-166
        return (self._config, self.user.copy(), self.item.copy(), self.user_feature_weight,
                self.item_feature_weight)

    def __setstate__(self, state: Tuple[Any, ...]) -> None:  # wrapper.cpp:167-181
        if len(state) not in (3, 5):
            raise RuntimeError("Invalid IALSTrainer pickle state.")
        other = IALSTrainer._from_factors(state[0], state[1], state[2])
        self.__dict__.update(other.__dict__)
        other._handle = ctypes.c_void_p(0)
        if len(state) == 5:  # wrapper.cpp:174-179
            self.user_feature_weight = state[3]
            self.item_feature_weight = state[4]

    # -- B200 extensions (not in the reference module) --
    def step_async(self, solver_config: IALSSolverConfig) -> None:
        """Enqueue one epoch without synchronising (see ``sync``)."""
        sc = self._solver(solver_config)
        self._cache.clear()
        self._use_current_stream()
        check(lib.ials_trainer_step_async(self._handle, ctypes.byref(sc)))

    def sync(self) -> None:
        check(lib.ials_trainer_sync(self._handle))

    def step_io(self, solver_config: IALSSolverConfig, user: np.ndarray, item: np.ndarray) -> None:
        """One epoch on HOST-resident factors, in place: the same as
        ``self.user = user; self.item = item; self.step(cfg); user[:] = self.user; item[:] = self.item``
        (wrapper.cpp:137, 158-159) as one call; the user matrix is read back while the item
        half-epoch runs.  Pinned arrays (``torch.empty(..., pin_memory=True).numpy()``) make
        the copies asynchronous."""
        sc = self._solver(solver_config)
        for a, n in ((user, self.n_users), (item, self.n_items)):
            if a.dtype != np.float32 or a.shape != (n, self.K) or not a.flags.c_contiguous:
                raise ValueError("factors must be C-contiguous float32 of shape (n, K)")
        self._cache.clear()
        self._use_current_stream()
        check(lib.ials_trainer_step_io(self._handle, ctypes.byref(sc), _ptr(user), _ptr(item),
                                       _ptr(user), _ptr(item)))

    def half_step(self, side: int, solver_config: IALSSolverConfig) -> None:
        sc = self._solver(solver_config)
        self._cache.clear()
        self._use_current_stream()
        check(lib.ials_trainer_half_step(self._handle, side, ctypes.byref(sc)))

    def gram(self, side: int) -> np.ndarray:
        """``Solver::prepare_p`` result of the solver of ``side`` (0: alpha0 item^T item)."""
        out = np.empty((self.K, self.K), dtype=np.float32)
        self._use_current_stream()
        check(lib.ials_trainer_gram(self._handle, side, _ptr(out)))
        return out

    def recommend(self, begin: int, end: int, cutoff: int, mask: Any = "train",
                  return_scores: bool = False, allowed: Any = None):
        """Fused score + seen-mask + top-``cutoff`` for users ``[begin, end)``.

        ``mask``: "train" (rows of the training matrix), None, or a scipy sparse
        matrix with ``end - begin`` rows.  ``allowed``: None, or ``(n_lists, indptr,
        indices)`` with one shared list (``n_lists == 1``) or one list per row of the
        block, every list strictly ascending (the Evaluator's recommendable items,
        evaluator.cpp:168-180); items outside a row's list are never returned.
        Returns (indices int32 [rows, cutoff] padded with -1, counts int32 [rows]
        [, scores float32 [rows, cutoff]]).
        """
        rows = max(int(end) - int(begin), 0)
        return self._recommend(None, int(begin), int(end), rows, cutoff, mask, return_scores, allowed)

    def recommend_users(self, user_indices: Any, cutoff: int, mask: Any = "train",
                        return_scores: bool = False, allowed: Any = None):
        """``recommend`` for users picked by index (any order, repeats allowed): their factor rows
        are gathered on the device, nothing but the lists comes back (the serving path of
        ``IDMapper.recommend_for_known_user_batch``, utils/id_mapping.py:418-453).  ``mask`` and
        ``allowed`` have one row / list per listed user."""
        u = np.ascontiguousarray(user_indices, dtype=np.int64).reshape(-1)
        return self._recommend(u, 0, u.size, u.size, cutoff, mask, return_scores, allowed)

    def recommend_embeddings(self, user_embedding: Any, cutoff: int, mask: Any = None,
                             return_scores: bool = False, allowed: Any = None):
        """``recommend`` for embeddings that are not rows of the model (fold-in results): scored
        against the item factors where they lie on the device.  ``mask``: None or one sparse row
        per embedding."""
        emb = np.ascontiguousarray(user_embedding, dtype=np.float32)
        if emb.ndim != 2 or emb.shape[1] != self.K:
            raise ValueError("embedding must be (n, n_components)")
        if isinstance(mask, str):
            raise ValueError("embeddings have no training rows: mask must be None or a sparse matrix")
        return self._recommend(emb, 0, emb.shape[0], emb.shape[0], cutoff, mask, return_scores, allowed)

    def _recommend(self, users, begin, end, rows, cutoff, mask, return_scores, allowed):
        idx = np.empty((rows, cutoff), dtype=np.int32)
        cnt = np.empty((rows,), dtype=np.int32)
        sc = np.empty((rows, cutoff), dtype=np.float32) if return_scores else None
        mode, mi, mx = _mask_arrays(mask, rows, self.n_items)
        n_lists, ai, ax = _allowed_arrays(allowed)
        self._use_current_stream()
        if users is not None and users.dtype == np.float32:
            check(lib.ials_trainer_recommend_embeddings(
                self._handle, _ptr(users), rows, int(cutoff), mode, _ptr(mi), _ptr(mx),
                int(n_lists), _ptr(ai), _ptr(ax), _ptr(idx), _ptr(sc), _ptr(cnt)))
        elif users is not None:
            check(lib.ials_trainer_recommend_users(
                self._handle, _ptr(users), rows, int(cutoff), mode, _ptr(mi), _ptr(mx),
                int(n_lists), _ptr(ai), _ptr(ax), _ptr(idx), _ptr(sc), _ptr(cnt)))
        elif allowed is None:
            check(lib.ials_trainer_recommend(self._handle, begin, end, int(cutoff), mode,
                                             _ptr(mi), _ptr(mx), _ptr(idx), _ptr(sc), _ptr(cnt)))
        else:
            check(lib.ials_trainer_recommend_allowed(
                self._handle, begin, end, int(cutoff), mode, _ptr(mi), _ptr(mx),
                int(n_lists), _ptr(ai), _ptr(ax), _ptr(idx), _ptr(sc), _ptr(cnt)))
        return (idx, cnt, sc) if return_scores else (idx, cnt)

    def similar(self, side: int, indices: Any = None, cutoff: int = 10, metric: str = "cosine",
                exclude_self: bool = True, forbidden: Any = None, allowed: Any = None,
                return_scores: bool = True):
        """Nearest neighbours within one side (0: similar users, 1: similar items): for each query row,
        the best ``cutoff`` rows of the same side by ``metric`` ("cosine": q.y / (|q| |y|), 0 when
        either row is zero; "dot": q.y), ordered by (-score, index).

        ``indices``: None (every row of the side), a ``range`` of step 1, or row indices (any order,
        repeats allowed).  ``exclude_self`` hides each query row itself; ``forbidden``: None or a
        sparse matrix with one row per query whose non-zeros are hidden as well; ``allowed`` as in
        ``recommend`` (allow-lists need ``cutoff <= 128``).  Returns (indices int32 [n, cutoff]
        padded with -1, counts int32 [n] [, scores float32 [n, cutoff]]).  No trainer state changes."""
        return _similar(self._handle, self._device, self.n_users if side == 0 else self.n_items, side, indices,
                        cutoff, metric, exclude_self, forbidden, allowed, return_scores)

    def rank_candidates(self, user_indices: Any, candidates: Any, cutoff: int, mask: Any = "train",
                        return_scores: bool = True):
        """Ranks each user's own candidate items: the best ``cutoff`` of them by score, ordered by
        (-score, index), at a cost that follows the number of (user, candidate) pairs, not the catalogue.

        ``user_indices``: a ``range`` of step 1 or user indices (any order, repeats allowed).
        ``candidates``: ``(n_lists, indptr, indices)`` as ``allowed`` takes it, or a sequence of index
        lists; one list shared by every user or one per user.  Lists are sorted and their repeats dropped
        here.  ``mask``: "train" (each user's training row), None, or a sparse matrix with one row per
        user; masked candidates are dropped.  ``1 <= cutoff <= min(1024, n_items)``.  Returns (indices
        int32 [n, cutoff] padded with -1, counts int32 [n] [, scores float32 [n, cutoff]]).  No trainer
        state changes."""
        return _rank_candidates(self._handle, self._device, self.n_users, self.n_items, self.K, user_indices,
                                None, candidates, cutoff, mask, return_scores)

    def rank_candidates_embeddings(self, user_embedding: Any, candidates: Any, cutoff: int, mask: Any = None,
                                   return_scores: bool = True):
        """``rank_candidates`` for embeddings that are not rows of the model (fold-in results).
        ``mask``: None or one sparse row per embedding."""
        return _rank_candidates(self._handle, self._device, self.n_users, self.n_items, self.K, None,
                                user_embedding, candidates, cutoff, mask, return_scores)

    def candidate_scores(self, user_indices: Any, candidates: Any) -> np.ndarray:
        """The score of every (user, candidate) pair, float32, in the order of the candidate lists
        (any order, repeats allowed; a shared list counts once per user)."""
        return _candidate_scores(self._handle, self._device, self.n_users, self.n_items, user_indices, candidates)

    def explain(self, side: int, indices: Any, targets: Any, n_top: int = 10) -> Explanation:
        """Why rows of ``side`` (0: users) score their targets (rows of the other side): each score split
        into the contributions of the row's training history, exactly (Hu, Koren and Volinsky, ICDM 2008,
        section 5; ``implicit``'s ``ALS.explain``), solved on the device against the current factors.

        ``indices``: a ``range`` of step 1 or row indices (any order, repeats allowed).  ``targets``: one
        list of target ids per query row, as a sequence of lists or ``(indptr, indices)`` arrays.
        ``1 <= n_top <= 1024`` history entries are kept per pair.  Past the feature warm-up the stored
        feature prior enters as ``prior``.  The factors do not change."""
        return _explain(self._handle, self._device, (self.n_users, self.n_items), side, indices, None, targets,
                        n_top)

    def explain_history(self, side: int, X: Any, targets: Any, n_top: int = 10) -> Explanation:
        """``explain`` for rows that are not in the model: the rows of the sparse matrix ``X`` (one column
        per row of the other side) are the histories, every stored entry counting as given (zeros and
        repeated columns included), without a feature prior."""
        return _explain(self._handle, self._device, (self.n_users, self.n_items), side, None, X, targets, n_top)

    def get_factors_into(self, side: int, out: np.ndarray) -> None:
        """Device -> host copy into a caller-owned (e.g. pinned) C-contiguous buffer."""
        n = self.n_users if side == 0 else self.n_items
        if out.dtype != np.float32 or out.shape != (n, self.K) or not out.flags.c_contiguous:
            raise ValueError("output buffer must be C-contiguous float32 of the factor shape")
        self._use_current_stream()
        check(lib.ials_trainer_get_factors(self._handle, side, _ptr(out)))

    def set_profiling(self, enabled: bool) -> None:
        check(lib.ials_trainer_set_profiling(self._handle, int(bool(enabled))))

    def plan_stats(self, side: int) -> dict:
        """Row schedule of ``side``: rows, nnz, heavy rows (tensor-core path), their nnz, jobs,
        the longest row, and whether a stored value is negative (then every row is light)."""
        out = (ctypes.c_int64 * 8)()
        check(lib.ials_trainer_plan_stats(self._handle, side, out))
        keys = ("rows", "nnz", "heavy_rows", "heavy_nnz", "jobs", "max_degree", "has_negative",
                "reserved")
        return dict(zip(keys, (int(v) for v in out)))

    def get_timings(self):
        """(ms[8], n_epochs) since the last call: Gram(item), users {heavy Gram, heavy dense CG,
        other rows}, Gram(user), items {same three}."""
        ms = (ctypes.c_double * 8)()
        n = ctypes.c_int64(0)
        check(lib.ials_trainer_get_timings(self._handle, ms, ctypes.byref(n)))
        return [float(v) for v in ms], int(n.value)

    def factors_device(self, side: int):
        """Zero-copy ``torch`` view ([n, K], row stride ld) of a factor matrix."""
        return _factors_device(self._handle, side, self._device)
