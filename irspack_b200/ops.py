"""Stand-alone operators of the B200 iALS library (host buffers in and out).

``weighted_gram`` is the tensor-core contraction behind ``Solver::prepare_p``
(/root/reference/cpp_source/als/IALSTrainer.hpp:78-115) and the rank updates of
``Solver::step_cholesky`` (:37-58, 301-308); see ``include/ials_b200.h``.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import numpy as np

from ._ials_core import _current_device_and_stream, _ptr
from ._lib import check, lib


def weighted_gram(Y: np.ndarray, idx: Optional[np.ndarray] = None, w: Optional[np.ndarray] = None,
                  n_jobs: int = 8, bias: float = 0.0) -> Tuple[np.ndarray, np.ndarray]:
    """``G = sum_t w[t] * Y[idx[t]] Y[idx[t]]^T`` and ``b = sum_t (bias + w[t]) * Y[idx[t]]``
    computed by ``tcgen05.mma`` (error-compensated TF32, fp32-level accuracy)."""
    Y = np.ascontiguousarray(Y, dtype=np.float32)
    if Y.ndim != 2:
        raise ValueError("Y must be 2-D")
    n, K = Y.shape
    m = n
    if idx is not None:
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        m = idx.shape[0]
    if w is not None:
        w = np.ascontiguousarray(w, dtype=np.float32)
        if w.shape[0] != m:
            raise ValueError("w must have one entry per gathered row")
    G = np.empty((K, K), dtype=np.float32)
    b = np.empty((K,), dtype=np.float32)
    dev, _ = _current_device_and_stream()
    check(lib.ials_weighted_gram(_ptr(Y), n, K, _ptr(idx), _ptr(w), m, int(n_jobs),
                                 ctypes.c_float(bias), dev, _ptr(G), _ptr(b)))
    return G, b


def weighted_gram256(Y: np.ndarray, idx: np.ndarray, w: Optional[np.ndarray] = None,
                     n_jobs: int = 1, bias: float = 0.0) -> Tuple[np.ndarray, np.ndarray]:
    """The same contraction for 128 < K <= 256 (rank updates of the K = 256 Cholesky solver,
    ``BatchedRankUpdater`` :37-58): two symmetric 128 x 128 blocks and the cross block on the
    tensor cores (``ials_weighted_gram256``)."""
    Y = np.ascontiguousarray(Y, dtype=np.float32)
    n, K = Y.shape
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    m = idx.shape[0]
    if w is not None:
        w = np.ascontiguousarray(w, dtype=np.float32)
        if w.shape[0] != m:
            raise ValueError("w must have one entry per gathered row")
    G = np.empty((K, K), dtype=np.float32)
    b = np.empty((K,), dtype=np.float32)
    dev, _ = _current_device_and_stream()
    check(lib.ials_weighted_gram256(_ptr(Y), n, K, _ptr(idx), _ptr(w), m, int(n_jobs),
                                    ctypes.c_float(bias), dev, _ptr(G), _ptr(b)))
    return G, b


def weighted_gram_jobs(Y: np.ndarray, job_begin: np.ndarray, job_end: np.ndarray,
                       idx: Optional[np.ndarray] = None, w: Optional[np.ndarray] = None,
                       bias: float = 0.0) -> Tuple[np.ndarray, np.ndarray]:
    """Each job's own block, for K <= 256: ``G[j] = sum_{t in [job_begin[j], job_end[j])} w[t] *
    Y[idx[t]] Y[idx[t]]^T`` and ``b[j] = sum_t (bias + w[t]) * Y[idx[t]]`` from one launch of the
    tensor-core Gram (``ials_weighted_gram_jobs``).  Returns G [n_jobs, K, K], b [n_jobs, K]."""
    Y = np.ascontiguousarray(Y, dtype=np.float32)
    if Y.ndim != 2:
        raise ValueError("Y must be 2-D")
    n, K = Y.shape
    m = n
    if idx is not None:
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        m = idx.shape[0]
    if w is not None:
        w = np.ascontiguousarray(w, dtype=np.float32)
        if w.shape[0] != m:
            raise ValueError("w must have one entry per gathered row")
    jb = np.ascontiguousarray(job_begin, dtype=np.int64)
    je = np.ascontiguousarray(job_end, dtype=np.int64)
    if jb.ndim != 1 or jb.shape != je.shape:
        raise ValueError("job_begin and job_end must be 1-D of the same length")
    G = np.empty((jb.shape[0], K, K), dtype=np.float32)
    b = np.empty((jb.shape[0], K), dtype=np.float32)
    dev, _ = _current_device_and_stream()
    check(lib.ials_weighted_gram_jobs(_ptr(Y), n, K, _ptr(idx), _ptr(w), m, _ptr(jb), _ptr(je), jb.shape[0],
                                      ctypes.c_float(bias), dev, _ptr(G), _ptr(b)))
    return G, b
