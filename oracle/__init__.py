"""CPU oracle for the iALS hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes front-end of ``oracle/ials_oracle.cpp`` (see that file's header for the
parity status: pinned to the reference's own sources -- ``oracle/_ref``, compiled
from /root/reference where it lies against the stand-ins of ``oracle/ref_shim`` --
at the algorithm level, unpinned at bit level) and of ``oracle/_ref`` itself
(``RefTrainer``, ``ref_evaluator_metrics``).  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import this package.  ``irspack_b200`` never does.

The library is compiled for the host it runs on (``-march=native``): it is
rebuilt automatically when the source is newer than the binary or when the
binary was built on a CPU with a different flag set (the GPU box's host is not
this container's host).
"""
from __future__ import annotations

import ctypes
import hashlib
import math
import os
import shutil
import stat
import subprocess
import tempfile
from typing import Dict, List, Optional, Tuple

import numpy as np
import scipy.sparse as sps

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ials_oracle.cpp")
_SRC_RNG = os.path.join(_HERE, "ials_oracle_rng.cpp")
_BUILD = os.path.join(_HERE, "_build")
_SO = os.path.join(_BUILD, "libials_oracle.so")
# A toolchain that links libstdc++ statically (this image's /opt/gcc wrapper) must keep that copy
# private: a Python process already holds another libstdc++, and a half-interposed static one
# crashes on the first throw.  Harmless with a dynamic libstdc++.
_PRIVATE_RUNTIME = "-Wl,--exclude-libs,ALL"

STATUS_OK, STATUS_INVALID, STATUS_CG_SINGULAR, STATUS_CHOL_DECOMP, STATUS_CHOL_SOLVE = range(5)
LOSS_ORIGINAL, LOSS_IALSPP = 0, 1
SOLVER_CHOLESKY, SOLVER_CG, SOLVER_IALSPP = 0, 1, 2

# messages of the reference's exceptions (IALSTrainer.hpp:252-253, 318, 322)
_MESSAGES = {
    STATUS_CG_SINGULAR: "Conjugate-gradient solver encountered a singular system.",
    STATUS_CHOL_DECOMP: "Cholesky decomposition failed.",
    STATUS_CHOL_SOLVE: "Cholesky solve failed.",
}


def _cpu_stamp() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return hashlib.sha1(line.encode()).hexdigest()
    except OSError:
        pass
    return "unknown"


def _fresh(build_dir: str) -> bool:
    """The library in ``build_dir`` is newer than both sources and was built for this CPU."""
    so, stamp = os.path.join(build_dir, "libials_oracle.so"), os.path.join(build_dir, "cpu.stamp")
    if not (os.path.exists(so) and os.path.exists(stamp)):
        return False
    if any(os.path.getmtime(so) < os.path.getmtime(p) for p in (_SRC, _SRC_RNG)):
        return False
    with open(stamp) as f:
        return f.read().strip() == _cpu_stamp()


def _private_build_dir() -> str:
    """Where a read-only checkout builds the oracle: one directory per user under the system's
    temporary directory, reused by that user's later processes."""
    d = os.path.join(tempfile.gettempdir(), f"ials_oracle_{os.getuid()}")
    os.makedirs(d, mode=0o700, exist_ok=True)
    st = os.lstat(d)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or st.st_mode & 0o077:
        raise RuntimeError(f"{d} is not a directory private to this user; not loading a library from it")
    return d


def build(force: bool = False) -> str:
    """Compile the oracle with g++ -O3 (a few seconds): ``ials_oracle.cpp`` for this host
    (``-march=native``), ``ials_oracle_rng.cpp`` -- the libstdc++ random-number helpers -- for the
    x86-64 baseline without FMA contraction, like the reference's portable wheels.  A read-only
    checkout whose ``oracle/_build`` is missing or stale builds into ``_private_build_dir()``."""
    if not force and _fresh(_BUILD):
        return _SO
    writable = os.access(_BUILD if os.path.isdir(_BUILD) else _HERE, os.W_OK)
    out = _BUILD if writable else _private_build_dir()
    so = os.path.join(out, "libials_oracle.so")
    if not force and _fresh(out):
        return so
    os.makedirs(out, exist_ok=True)
    # objects and library are made in a scratch directory and the library moved into place, so that
    # processes building at the same time never load a half-written file
    work = tempfile.mkdtemp(dir=out)
    try:
        cxx = os.environ.get("CXX", "g++")
        common = ["-O3", "-std=c++17", "-fPIC", "-pthread", "-fvisibility=hidden"]
        obj, obj_rng = os.path.join(work, "ials_oracle.o"), os.path.join(work, "ials_oracle_rng.o")
        subprocess.run([cxx, *common, "-march=native", "-c", _SRC, "-o", obj], check=True)
        subprocess.run([cxx, *common, "-ffp-contract=off", "-c", _SRC_RNG, "-o", obj_rng], check=True)
        subprocess.run([cxx, "-shared", "-pthread", _PRIVATE_RUNTIME, "-o", os.path.join(work, "lib.so"),
                        obj, obj_rng], check=True)
        os.replace(os.path.join(work, "lib.so"), so)
    finally:
        shutil.rmtree(work, ignore_errors=True)
    with open(os.path.join(out, "cpu.stamp"), "w") as f:
        f.write(_cpu_stamp())
    return so


# ---- oracle/_ref: the reference's own sources, compiled where they lie ----
_REF_DIR = os.path.join(_HERE, "_ref")
_REF_EVAL_SO = os.path.join(_REF_DIR, "libref_evaluator.so")
_REF_SOURCES = "/root/reference/cpp_source"


def build_ref(force: bool = False) -> Optional[str]:
    """Compile the reference's evaluator (/root/reference/cpp_source/evaluator.cpp, unmodified,
    where it lies) against the container stand-ins of ``oracle/ref_shim`` into
    ``oracle/_ref/libref_evaluator.so``.  Only possible where /root/reference exists (the build
    container); elsewhere the prebuilt file, if it travelled, is used.  Returns its path or None."""
    src = os.path.join(_REF_SOURCES, "evaluator.cpp")
    capi = os.path.join(_HERE, "ref_evaluator_capi.cpp")
    if os.path.exists(src):
        shim = [os.path.join(_HERE, "ref_shim", "Eigen", f) for f in ("Core", "Sparse")]
        stale = force or not os.path.exists(_REF_EVAL_SO) or os.path.getmtime(_REF_EVAL_SO) < max(
            os.path.getmtime(p) for p in [capi, src] + shim)
        if stale:
            os.makedirs(_REF_DIR, exist_ok=True)
            subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread",
                            "-fvisibility=hidden", _PRIVATE_RUNTIME, "-I", os.path.join(_HERE, "ref_shim"),
                            "-I", _REF_SOURCES,
                            capi, "-o", _REF_EVAL_SO], check=True)
    return _REF_EVAL_SO if os.path.exists(_REF_EVAL_SO) else None


_REF_TRAINER_SO = os.path.join(_REF_DIR, "libref_trainer.so")


def build_ref_trainer(force: bool = False) -> Optional[str]:
    """Compile the reference's trainer (/root/reference/cpp_source/als/IALSTrainer.hpp with its
    config headers, unmodified, where they lie) against the Eigen stand-in of ``oracle/ref_shim``
    into ``oracle/_ref/libref_trainer.so``.  Returns its path, or None where neither
    /root/reference nor a prebuilt file exists."""
    src = os.path.join(_REF_SOURCES, "als", "IALSTrainer.hpp")
    capi = os.path.join(_HERE, "ref_trainer_capi.cpp")
    shim = [os.path.join(_HERE, "ref_shim", "Eigen", f) for f in ("Core", "Sparse", "Cholesky")]
    if os.path.exists(src):
        newest = max(os.path.getmtime(p) for p in [capi, src] + shim)
        if force or not os.path.exists(_REF_TRAINER_SO) or os.path.getmtime(_REF_TRAINER_SO) < newest:
            os.makedirs(_REF_DIR, exist_ok=True)
            subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread",
                            "-fvisibility=hidden", _PRIVATE_RUNTIME, "-I", os.path.join(_HERE, "ref_shim"),
                            "-I", _REF_SOURCES,
                            capi, "-o", _REF_TRAINER_SO], check=True)
    return _REF_TRAINER_SO if os.path.exists(_REF_TRAINER_SO) else None


class RefTrainer:
    """The REFERENCE'S OWN ``IALSTrainer`` (``oracle/_ref``: IALSTrainer.hpp compiled where it lies
    against the Eigen stand-in), with the interface of ``OracleTrainer``.  Test infrastructure."""

    _so: Optional[ctypes.CDLL] = None

    @classmethod
    def available(cls) -> bool:
        return build_ref_trainer() is not None

    def __init__(self, X, K, alpha0=0.1, reg=0.1, nu=1.0, loss_type=1, init_stdev=0.1, random_seed=42,
                 user_features=None, item_features=None, lambda_user_feature=0.0, lambda_item_feature=0.0,
                 feature_warmup_epochs=0):
        if RefTrainer._so is None:
            path = build_ref_trainer()
            if path is None:
                raise FileNotFoundError("oracle/_ref/libref_trainer.so is not built (needs /root/reference)")
            RefTrainer._so = ctypes.CDLL(path)
            RefTrainer._so.ref_trainer_last_error.restype = ctypes.c_char_p
        X = sps.csr_matrix(X, dtype=np.float32)
        X.sort_indices()
        self.n_users, self.n_items, self.K = X.shape[0], X.shape[1], int(K)
        ip = np.ascontiguousarray(X.indptr, dtype=np.int64)
        ix = np.ascontiguousarray(X.indices, dtype=np.int32)
        dt = np.ascontiguousarray(X.data, dtype=np.float32)
        h = ctypes.c_void_p(0)
        cf = ctypes.c_float
        self._h = None
        if user_features is None and item_features is None:
            self._chk(self._so.ref_trainer_create(
                ctypes.c_int64(K), cf(alpha0), cf(reg), cf(nu), cf(init_stdev), ctypes.c_int32(random_seed),
                ctypes.c_int(int(loss_type)), ctypes.c_int64(X.shape[0]), ctypes.c_int64(X.shape[1]), _p(ip), _p(ix),
                _p(dt), ctypes.byref(h)))
        else:  # IALSTrainer(config, X, user_features, item_features), IALSTrainer.hpp:722-743
            self._so.ref_trainer_feature_weight_rows.restype = ctypes.c_int64
            fa = [self._features(F, n) for F, n in ((user_features, X.shape[0]), (item_features, X.shape[1]))]
            self._chk(self._so.ref_trainer_create_features(
                ctypes.c_int64(K), cf(alpha0), cf(reg), cf(nu), cf(init_stdev), ctypes.c_int32(random_seed),
                ctypes.c_int(int(loss_type)), cf(lambda_user_feature), cf(lambda_item_feature),
                ctypes.c_int64(feature_warmup_epochs), ctypes.c_int64(X.shape[0]), ctypes.c_int64(X.shape[1]),
                _p(ip), _p(ix), _p(dt), *fa[0][1:], *fa[1][1:], ctypes.byref(h)))
        self._h = h

    @staticmethod
    def _features(F, n_rows):
        """(keep-alive arrays, cols, dense, indptr, indices, data) for ref_trainer_create_features."""
        null = ctypes.c_void_p(0)
        if F is None:
            F = np.zeros((n_rows, 0), np.float32)
        if sps.issparse(F):
            C = sps.csr_matrix(F, dtype=np.float32)
            C.sort_indices()
            a = (np.ascontiguousarray(C.indptr, dtype=np.int64), np.ascontiguousarray(C.indices, dtype=np.int32),
                 np.ascontiguousarray(C.data, dtype=np.float32))
            return (a, ctypes.c_int64(C.shape[1]), null, _p(a[0]), _p(a[1]), _p(a[2]))
        D = np.ascontiguousarray(F, dtype=np.float32)
        return ((D,), ctypes.c_int64(D.shape[1]), _p(D), null, null, null)

    def _feature_weight(self, side):
        n = int(self._so.ref_trainer_feature_weight_rows(self._h, side))
        out = np.zeros((n, self.K), dtype=np.float32)
        if n:
            self._chk(self._so.ref_trainer_get_feature_weight(self._h, side, _p(out)))
        return out

    user_feature_weight = property(lambda s: s._feature_weight(0))
    item_feature_weight = property(lambda s: s._feature_weight(1))

    def transform_with_feature(self, side, X, features, solver_type=1, max_cg_steps=5, n_threads=1):
        X = sps.csr_matrix(X, dtype=np.float32)
        X.sort_indices()
        ip = np.ascontiguousarray(X.indptr, dtype=np.int64)
        ix = np.ascontiguousarray(X.indices, dtype=np.int32)
        dt = np.ascontiguousarray(X.data, dtype=np.float32)
        F = np.ascontiguousarray(features.toarray() if sps.issparse(features) else features, dtype=np.float32)
        out = np.empty((X.shape[0] if side == 0 else X.shape[1], self.K), dtype=np.float32)
        self._chk(self._so.ref_trainer_transform_with_feature(
            self._h, side, ctypes.c_int64(X.shape[0]), ctypes.c_int64(X.shape[1]), _p(ip), _p(ix), _p(dt),
            ctypes.c_int64(F.shape[0]), ctypes.c_int64(F.shape[1]), _p(F), ctypes.c_int64(n_threads),
            ctypes.c_int(solver_type), ctypes.c_int64(max_cg_steps), _p(out)))
        return out

    def __del__(self):
        if getattr(self, "_h", None):
            self._so.ref_trainer_destroy(self._h)
            self._h = None

    def _chk(self, st: int) -> None:
        if st != 0:
            msg = self._so.ref_trainer_last_error().decode()
            raise (ValueError if st == 1 else RuntimeError)(msg)

    def _get(self, side):
        out = np.empty((self.n_users if side == 0 else self.n_items, self.K), dtype=np.float32)
        self._chk(self._so.ref_trainer_get(self._h, side, _p(out)))
        return out

    def _set(self, side, v):
        v = np.ascontiguousarray(v, dtype=np.float32)
        assert v.shape == ((self.n_users if side == 0 else self.n_items), self.K)
        self._chk(self._so.ref_trainer_set(self._h, side, _p(v)))

    user = property(lambda s: s._get(0), lambda s, v: s._set(0, v))
    item = property(lambda s: s._get(1), lambda s, v: s._set(1, v))

    # solver_type as in the product's C ABI / wrapper.cpp:29-32: 0 CHOLESKY, 1 CG, 2 IALSPP
    def step(self, solver_type=1, max_cg_steps=3, n_threads=1, subspace_dim=64, iterations=1):
        self._chk(self._so.ref_trainer_step(self._h, ctypes.c_int64(n_threads), ctypes.c_int(solver_type),
                                            ctypes.c_int64(max_cg_steps), ctypes.c_int64(subspace_dim),
                                            ctypes.c_int64(iterations)))

    def gram(self, side, n_threads=1):
        out = np.empty((self.K, self.K), dtype=np.float32)
        self._chk(self._so.ref_trainer_gram(self._h, side, ctypes.c_int64(n_threads), _p(out)))
        return out

    def transform(self, side, X, solver_type=1, max_cg_steps=5, n_threads=1, subspace_dim=64, iterations=1):
        X = sps.csr_matrix(X, dtype=np.float32)
        X.sort_indices()
        ip = np.ascontiguousarray(X.indptr, dtype=np.int64)
        ix = np.ascontiguousarray(X.indices, dtype=np.int32)
        dt = np.ascontiguousarray(X.data, dtype=np.float32)
        out = np.empty((X.shape[0] if side == 0 else X.shape[1], self.K), dtype=np.float32)
        self._chk(self._so.ref_trainer_transform(
            self._h, side, ctypes.c_int64(X.shape[0]), ctypes.c_int64(X.shape[1]), _p(ip), _p(ix), _p(dt),
            ctypes.c_int64(n_threads), ctypes.c_int(solver_type), ctypes.c_int64(max_cg_steps),
            ctypes.c_int64(subspace_dim), ctypes.c_int64(iterations), _p(out)))
        return out

    def compute_loss(self, n_threads=1) -> float:
        out = ctypes.c_float(0)
        self._chk(self._so.ref_trainer_compute_loss(self._h, ctypes.c_int64(n_threads), ctypes.byref(out)))
        return float(out.value)

    def user_scores(self, begin, end, n_threads=1):
        out = np.empty((max(end - begin, 0), self.n_items), dtype=np.float32)
        self._chk(self._so.ref_trainer_user_scores(self._h, ctypes.c_int64(begin), ctypes.c_int64(end),
                                                   ctypes.c_int64(n_threads), _p(out)))
        return out


_ref_eval: Optional[ctypes.CDLL] = None


def ref_evaluator_metrics(scores: np.ndarray, ground_truth, cutoff: int, offset: int = 0, n_threads: int = 1,
                          recall_with_cutoff: bool = False, recommendable=None) -> Dict[str, float]:
    """``EvaluatorCore(ground_truth, recommendable).get_metrics_f32/f64(scores, cutoff, offset,
    n_threads, recall_with_cutoff).as_dict()`` computed by the REFERENCE'S OWN evaluator.cpp
    (``oracle/_ref``).  Raises FileNotFoundError when it is not built (no /root/reference)."""
    global _ref_eval
    if _ref_eval is None:
        path = build_ref()
        if path is None:
            raise FileNotFoundError("oracle/_ref/libref_evaluator.so is not built (needs /root/reference)")
        _ref_eval = ctypes.CDLL(path)
        _ref_eval.ref_evaluator_last_error.restype = ctypes.c_char_p
    scores = np.ascontiguousarray(scores)
    if scores.dtype not in (np.dtype("float32"), np.dtype("float64")):
        raise ValueError("scores must be float32 or float64")
    gt = sps.csr_matrix(ground_truth)
    gt.sort_indices()
    gi = np.ascontiguousarray(gt.indptr, dtype=np.int64)
    gx = np.ascontiguousarray(gt.indices, dtype=np.int32)
    lists = [] if recommendable is None else [np.asarray(l, dtype=np.int64) for l in recommendable]
    rip = np.zeros(len(lists) + 1, dtype=np.int64)
    if lists:
        rip[1:] = np.cumsum([len(l) for l in lists])
    rix = np.concatenate(lists).astype(np.int64) if lists else np.zeros(0, np.int64)
    out = np.zeros(11, dtype=np.float64)
    st = _ref_eval.ref_evaluator_metrics(
        ctypes.c_int(int(scores.dtype == np.float64)), _p(scores), ctypes.c_int64(scores.shape[0]),
        ctypes.c_int64(gt.shape[0]), ctypes.c_int64(gt.shape[1]), _p(gi), _p(gx), ctypes.c_int64(len(lists)),
        _p(rip), _p(rix), ctypes.c_int64(cutoff), ctypes.c_int64(offset), ctypes.c_int64(n_threads),
        ctypes.c_int(int(recall_with_cutoff)), _p(out))
    if st != 0:
        msg = _ref_eval.ref_evaluator_last_error().decode()
        raise (ValueError if st == 1 else RuntimeError)(msg)
    keys = ("total_user", "valid_user", "n_items", "hit", "ndcg", "recall", "map", "precision",
            "appeared_item", "entropy", "gini_index")
    return dict(zip(keys, (float(v) for v in out)))


_lib: Optional[ctypes.CDLL] = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def hardware_threads() -> int:
    return int(lib().oracle_hardware_threads())


def _sfx(dtype) -> Tuple[str, type]:
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        return "f32", ctypes.c_float
    if dtype == np.float64:
        return "f64", ctypes.c_double
    raise ValueError("oracle supports float32 and float64 only")


def _p(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def _check(status: int) -> None:
    if status == STATUS_OK:
        return
    if status == STATUS_INVALID:
        raise ValueError("invalid argument")
    raise RuntimeError(_MESSAGES.get(status, f"oracle status {status}"))


def _csr_parts(X: sps.csr_matrix, dtype) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    X = sps.csr_matrix(X)
    if not X.has_sorted_indices:
        X = X.sorted_indices()
    return (
        np.ascontiguousarray(X.indptr, dtype=np.int64),
        np.ascontiguousarray(X.indices, dtype=np.int32),
        np.ascontiguousarray(X.data, dtype=dtype),
    )


def gram(Y: np.ndarray, alpha0: float, n_threads: int = 1) -> np.ndarray:
    """P = alpha0 * Y^T Y  (IALSTrainer.hpp:78-115)."""
    Y = np.ascontiguousarray(Y)
    sfx, cf = _sfx(Y.dtype)
    n, K = Y.shape
    P = np.empty((K, K), dtype=Y.dtype)
    _check(getattr(lib(), f"oracle_gram_{sfx}")(
        _p(Y), ctypes.c_int64(n), ctypes.c_int64(K), cf(alpha0), ctypes.c_int(n_threads), _p(P)))
    return P


def step_cg(target, X, other, P, alpha0, reg, nu, loss_type, max_cg_steps, n_threads=1, prior=None):
    """In-place CG half-epoch on ``target`` (IALSTrainer.hpp:170-271).  ``prior`` (same shape
    as ``target``): the feature-aware variant, ``b += reg_u * prior_u`` and rows without
    interactions are solved too (:207-215)."""
    sfx, cf = _sfx(target.dtype)
    assert target.flags.c_contiguous and other.flags.c_contiguous and P.flags.c_contiguous
    indptr, indices, data = _csr_parts(X, target.dtype)
    n_rows, K = target.shape
    args = [_p(target), ctypes.c_int64(n_rows), _p(indptr), _p(indices), _p(data), _p(other),
            ctypes.c_int64(other.shape[0]), ctypes.c_int64(K), _p(P), cf(alpha0), cf(reg), cf(nu),
            ctypes.c_int(loss_type), ctypes.c_int(max_cg_steps), ctypes.c_int(n_threads)]
    if prior is None:
        _check(getattr(lib(), f"oracle_step_cg_{sfx}")(*args))
    else:
        prior = _prior_like(prior, target)
        _check(getattr(lib(), f"oracle_step_cg_prior_{sfx}")(*args, _p(prior)))


def step_cholesky(target, X, other, P, alpha0, reg, nu, loss_type, n_threads=1, prior=None):
    """In-place Cholesky half-epoch on ``target`` (IALSTrainer.hpp:273-331; with ``prior``:
    step_cholesky_with_prior, :333-385)."""
    sfx, cf = _sfx(target.dtype)
    assert target.flags.c_contiguous and other.flags.c_contiguous and P.flags.c_contiguous
    indptr, indices, data = _csr_parts(X, target.dtype)
    n_rows, K = target.shape
    args = [_p(target), ctypes.c_int64(n_rows), _p(indptr), _p(indices), _p(data), _p(other),
            ctypes.c_int64(other.shape[0]), ctypes.c_int64(K), _p(P), cf(alpha0), cf(reg), cf(nu),
            ctypes.c_int(loss_type), ctypes.c_int(n_threads)]
    if prior is None:
        _check(getattr(lib(), f"oracle_step_cholesky_{sfx}")(*args))
    else:
        prior = _prior_like(prior, target)
        _check(getattr(lib(), f"oracle_step_cholesky_prior_{sfx}")(*args, _p(prior)))


def _prior_like(prior, target):
    prior = np.ascontiguousarray(prior, dtype=target.dtype)
    if prior.shape != target.shape:
        raise ValueError("Feature prior shape does not match factor.")  # :176-178, :338-341
    return prior


def compute_reg(nnz, n_other, alpha0, reg, nu, dtype):
    """``Solver::compute_reg`` (:117-120) for an array of row counts, in ``dtype`` arithmetic."""
    dt = np.dtype(dtype).type
    return dt(reg) * np.power(dt(alpha0) * dt(n_other) + np.asarray(nnz).astype(dtype), dt(nu))


def feature_ridge(features, factor, row_weights, lam):
    """``update_feature_weight`` (:1095-1209): W = (F^T D F + lam I)^-1 F^T D factor with
    D = diag(row_weights) -- the weighted ridge regression of the factors on the features,
    solved through the Cholesky factor of the Gram the reference caches.  Sparse features are
    densified: this is the checker, sizes are small."""
    F = np.asarray(features.todense() if sps.issparse(features) else features, dtype=factor.dtype)
    if F.shape[1] == 0:
        return np.zeros((0, factor.shape[1]), dtype=factor.dtype)
    w = np.asarray(row_weights, dtype=factor.dtype)
    Fw = F * np.sqrt(w)[:, None]
    G = Fw.T @ Fw
    G[np.diag_indices_from(G)] += factor.dtype.type(lam)
    try:
        L = np.linalg.cholesky(G)
    except np.linalg.LinAlgError:
        raise RuntimeError("Feature ridge Cholesky decomposition failed.")  # :1103-1104
    rhs = F.T @ (factor * w[:, None])
    sol = np.linalg.solve(L.T, np.linalg.solve(L, rhs)).astype(factor.dtype)
    if not np.isfinite(sol).all():
        raise RuntimeError("Feature ridge solve failed.")
    return sol


def step_ialspp(target, X, other, P, alpha0, reg, nu, loss_type, subspace_dim=64, iterations=1,
                n_threads=1):
    """In-place iALS++ half-epoch on ``target`` (IALSTrainer.hpp:387-535)."""
    sfx, cf = _sfx(target.dtype)
    assert target.flags.c_contiguous and other.flags.c_contiguous and P.flags.c_contiguous
    indptr, indices, data = _csr_parts(X, target.dtype)
    n_rows, K = target.shape
    _check(getattr(lib(), f"oracle_step_ialspp_{sfx}")(
        _p(target), ctypes.c_int64(n_rows), _p(indptr), _p(indices), _p(data), _p(other),
        ctypes.c_int64(other.shape[0]), ctypes.c_int64(K), _p(P), cf(alpha0), cf(reg), cf(nu),
        ctypes.c_int(loss_type), ctypes.c_int64(subspace_dim), ctypes.c_int64(iterations),
        ctypes.c_int(n_threads)))


def user_scores(user, item, begin, end, n_threads=1):
    """S = user[begin:end] @ item.T  (IALSTrainer.hpp:942-984)."""
    user = np.ascontiguousarray(user)
    item = np.ascontiguousarray(item)
    sfx, _ = _sfx(user.dtype)
    if end < begin or end > user.shape[0] or begin < 0:
        raise ValueError("bad user block")
    out = np.empty((end - begin, item.shape[0]), dtype=user.dtype)
    _check(getattr(lib(), f"oracle_user_scores_{sfx}")(
        _p(user), _p(item), ctypes.c_int64(user.shape[0]), ctypes.c_int64(item.shape[0]),
        ctypes.c_int64(user.shape[1]), ctypes.c_int64(begin), ctypes.c_int64(end),
        ctypes.c_int(n_threads), _p(out)))
    return out


class Metrics:
    """Restatement of ``Metrics`` (cpp_source/evaluator.cpp:49-179)."""

    def __init__(self, n_item: int):
        self.n_item = n_item
        self.acc = np.zeros(7, dtype=np.float64)
        self.item_cnt = np.zeros(n_item, dtype=np.int64)

    def merge(self, other: "Metrics") -> None:  # :76-85
        self.acc += other.acc
        self.item_cnt += other.item_cnt

    def as_dict(self) -> Dict[str, float]:  # :87-123
        cnt = np.sort(self.item_cnt)
        total = float(cnt.sum())
        appeared, entropy, gini = 0.0, 0.0, 0.0
        n = len(cnt)
        for i, c in enumerate(cnt):
            if c == 0:
                continue
            p = c / total
            appeared += 1
            entropy += -math.log(p) * p
            gini += (2 * i - n + 1) * float(c)
        if total > 0:
            gini /= n * total
        valid, total_user, hit, recall, ndcg, precision, map_ = self.acc
        den = valid if valid > 0 else 1.0
        return {
            "total_user": total_user, "valid_user": valid, "n_items": float(self.n_item),
            "hit": hit / den, "ndcg": ndcg / den, "recall": recall / den, "map": map_ / den,
            "precision": precision / den, "appeared_item": appeared, "entropy": entropy,
            "gini_index": gini,
        }


def topk_metrics(scores, ground_truth, cutoff, offset=0, recall_with_cutoff=False):
    """``EvaluatorCore.get_metrics`` for one score block (evaluator.cpp:256-367).

    Returns (Metrics, rec[int32 rows x cutoff, -1 padded], n_rec[int32 rows]).
    """
    scores = np.ascontiguousarray(scores)
    sfx, _ = _sfx(scores.dtype)
    rows, n_items = scores.shape
    gt = sps.csr_matrix(ground_truth)
    gt.sort_indices()
    if gt.shape[1] != n_items or offset + rows > gt.shape[0]:
        raise ValueError("shape mismatch")
    gi = np.ascontiguousarray(gt.indptr, dtype=np.int64)
    gx = np.ascontiguousarray(gt.indices, dtype=np.int32)
    m = Metrics(n_items)
    rec = np.empty((rows, cutoff), dtype=np.int32)
    cnt = np.empty(rows, dtype=np.int32)
    _check(getattr(lib(), f"oracle_topk_metrics_{sfx}")(
        _p(scores), ctypes.c_int64(rows), ctypes.c_int64(n_items), _p(gi), _p(gx),
        ctypes.c_int64(offset), ctypes.c_int64(cutoff), ctypes.c_int(int(recall_with_cutoff)),
        _p(m.acc), _p(m.item_cnt), _p(rec), _p(cnt)))
    return m, rec, cnt


class OracleTrainer:
    """CPU twin of ``_ials_core.IALSTrainer`` (IALSTrainer.hpp:709-984) for tests.

    Factors are set explicitly (``user`` / ``item`` attributes), which is how the
    parity runs bypass ``Solver::initialize`` (SURVEY.md section 8 a2).
    """

    def __init__(self, X, K, alpha0=0.1, reg=0.1, nu=1.0, loss_type=LOSS_IALSPP,
                 dtype=np.float32, init_stdev=0.1, seed=42, user_features=None, item_features=None,
                 lambda_user_feature=0.0, lambda_item_feature=0.0, feature_warmup_epochs=0):
        self.dtype = np.dtype(dtype)
        X = sps.csr_matrix(X).astype(self.dtype)
        X.sort_indices()
        self.X = X
        self.X_t = sps.csr_matrix(X.T)  # IALSTrainer.hpp:713
        self.X_t.sort_indices()
        self.K, self.alpha0, self.reg, self.nu, self.loss_type = K, alpha0, reg, nu, loss_type
        U, I = X.shape
        rng = np.random.default_rng(seed)
        scale = init_stdev / math.sqrt(K)
        self.user = (rng.standard_normal((U, K)) * scale).astype(self.dtype)
        self.item = (rng.standard_normal((I, K)) * scale).astype(self.dtype)
        # feature-aware model (IALSTrainer.hpp:722-743, initialize_feature_aware :1001-1014)
        self.feature_aware = user_features is not None or item_features is not None
        self.epoch = 0
        self.feature_warmup_epochs = feature_warmup_epochs
        self.lambda_feature = [lambda_user_feature, lambda_item_feature]
        self.features = [None, None]
        self.feature_weight = [np.zeros((0, K), self.dtype), np.zeros((0, K), self.dtype)]
        if self.feature_aware:
            for side, (F, n) in enumerate(((user_features, U), (item_features, I))):
                if F is None:  # ials.py:64-66: the other side gets an n x 0 matrix
                    F = sps.csr_matrix((n, 0), dtype=self.dtype)
                F = sps.csr_matrix(F, dtype=self.dtype) if sps.issparse(F) else np.asarray(F, self.dtype)
                if F.shape[0] != n:
                    raise ValueError("Feature matrix row count mismatch.")
                if F.shape[1] and not self.lambda_feature[side] > 0:
                    raise ValueError("Feature weight regularization must be positive.")
                self.features[side] = F
                self.feature_weight[side] = np.zeros((F.shape[1], K), self.dtype)

    user_feature_weight = property(lambda s: s.feature_weight[0])
    item_feature_weight = property(lambda s: s.feature_weight[1])

    def _row_reg(self, side):
        """compute_reg of every row of ``side`` (0 users, 1 items)."""
        X = self.X if side == 0 else self.X_t
        return compute_reg(np.diff(X.indptr), X.shape[1], self.alpha0, self.reg, self.nu, self.dtype)

    def _prior(self, side, features=None):
        """feature_times_weight (:696-702): ``features @ feature_weight`` of ``side``."""
        F = self.features[side] if features is None else features
        W = self.feature_weight[side]
        if F.shape[1] != W.shape[0]:
            who = "user" if side == 0 else "item"
            raise ValueError(f"Shape mismatch: {who} feature matrix has {F.shape[1]} columns but "
                             f"{who}_feature_weight has {W.shape[0]} rows.")  # :1016-1042
        out = F @ W
        return np.ascontiguousarray(np.asarray(out), dtype=self.dtype)

    def _solve_with_prior(self, target, X, other, prior, solver_type, max_cg_steps, n_threads):
        """Solver::step_with_prior (:634-662)."""
        if self.alpha0 == 0:
            empty_reg = compute_reg(np.zeros(1), other.shape[0], self.alpha0, self.reg, self.nu, self.dtype)[0]
            if (not empty_reg > 0 or not np.isfinite(empty_reg)) and (np.diff(X.indptr) == 0).any():
                raise ValueError("Feature-prior embedding is not uniquely defined for an empty "
                                 "interaction row when alpha0 and its regularization are zero.")
        P = gram(other, self.alpha0, n_threads)
        if solver_type == SOLVER_CG:
            step_cg(target, X, other, P, self.alpha0, self.reg, self.nu, self.loss_type,
                    max_cg_steps, n_threads, prior=prior)
        elif solver_type == SOLVER_CHOLESKY:
            step_cholesky(target, X, other, P, self.alpha0, self.reg, self.nu, self.loss_type,
                          n_threads, prior=prior)
        else:
            raise ValueError("Feature-aware iALS does not support IALSPP.")

    # iALS++ settings (IALSSolverConfig: ialspp_subspace_dimension, ialspp_iteration)
    ialspp_subspace_dimension = 64
    ialspp_iteration = 1

    def _solve(self, target, X, other, solver_type, max_cg_steps, n_threads):
        P = gram(other, self.alpha0, n_threads)
        if solver_type == SOLVER_CG:
            step_cg(target, X, other, P, self.alpha0, self.reg, self.nu, self.loss_type,
                    max_cg_steps, n_threads)
        elif solver_type == SOLVER_IALSPP:
            step_ialspp(target, X, other, P, self.alpha0, self.reg, self.nu, self.loss_type,
                        self.ialspp_subspace_dimension, self.ialspp_iteration, n_threads)
        else:
            step_cholesky(target, X, other, P, self.alpha0, self.reg, self.nu, self.loss_type,
                          n_threads)

    def step(self, solver_type=SOLVER_CG, max_cg_steps=3, n_threads=1):  # :758-789
        if self.feature_aware and solver_type == SOLVER_IALSPP:
            raise ValueError("Feature-aware iALS does not support IALSPP.")
        with_features = self.feature_aware and self.epoch >= self.feature_warmup_epochs
        sides = ((0, self.user, self.X, self.item), (1, self.item, self.X_t, self.user))
        for side, target, X, other in sides:
            if with_features and self.feature_weight[side].shape[0]:
                # solve against the prior of the CURRENT weights, then refit the weights (:765-769)
                self._solve_with_prior(target, X, other, self._prior(side), solver_type, max_cg_steps,
                                       n_threads)
                self.feature_weight[side] = feature_ridge(self.features[side], target,
                                                          self._row_reg(side), self.lambda_feature[side])
            else:
                self._solve(target, X, other, solver_type, max_cg_steps, n_threads)
        self.epoch += 1

    def transform_user_feature(self, features):  # :820-824
        return self._prior(0, self._as_features(features))

    def transform_item_feature(self, features):  # :826-830
        return self._prior(1, self._as_features(features))

    def _as_features(self, F):
        return sps.csr_matrix(F, dtype=self.dtype) if sps.issparse(F) else np.asarray(F, self.dtype)

    def transform_user_with_feature(self, X, features, solver_type=SOLVER_CG, max_cg_steps=5,
                                    n_threads=1):  # :804-811, X_to_vector_with_prior :143-167
        X = sps.csr_matrix(X).astype(self.dtype)
        if X.shape[1] != self.item.shape[0]:
            raise ValueError("Shape mismatch")
        prior = self.transform_user_feature(features)
        if prior.shape != (X.shape[0], self.K):
            raise ValueError("Feature prior shape does not match X.")
        out = prior.copy()
        self._solve_with_prior(out, X, self.item, prior, solver_type, max_cg_steps, n_threads)
        return out

    def transform_item_with_feature(self, X, features, solver_type=SOLVER_CG, max_cg_steps=5,
                                    n_threads=1):  # :813-818
        Xt = sps.csr_matrix(sps.csr_matrix(X).T).astype(self.dtype)
        if Xt.shape[1] != self.user.shape[0]:
            raise ValueError("Shape mismatch")
        prior = self.transform_item_feature(features)
        if prior.shape != (Xt.shape[0], self.K):
            raise ValueError("Feature prior shape does not match X.")
        out = prior.copy()
        self._solve_with_prior(out, Xt, self.user, prior, solver_type, max_cg_steps, n_threads)
        return out

    def transform_user(self, X, solver_type=SOLVER_CG, max_cg_steps=5, n_threads=1):  # :791-795
        X = sps.csr_matrix(X).astype(self.dtype)
        if X.shape[1] != self.item.shape[0]:
            raise ValueError("Shape mismatch")
        out = np.zeros((X.shape[0], self.K), dtype=self.dtype)
        self._solve(out, X, self.item, solver_type, max_cg_steps, n_threads)
        return out

    def transform_item(self, X, solver_type=SOLVER_CG, max_cg_steps=5, n_threads=1):  # :797-802
        X = sps.csr_matrix(X).astype(self.dtype)
        if X.shape[0] != self.user.shape[0]:
            raise ValueError("Shape mismatch")
        Xt = sps.csr_matrix(X.T)
        out = np.zeros((Xt.shape[0], self.K), dtype=self.dtype)
        self._solve(out, Xt, self.user, solver_type, max_cg_steps, n_threads)
        return out

    def user_scores(self, begin, end, n_threads=1):
        return user_scores(self.user, self.item, begin, end, n_threads)

    def compute_loss(self, n_threads=1) -> float:  # :836-940
        if self.feature_aware:
            return self._compute_loss_feature_aware()
        sfx, cf = _sfx(self.dtype)
        indptr, indices, data = _csr_parts(self.X, self.dtype)
        indptr_t = np.ascontiguousarray(self.X_t.indptr, dtype=np.int64)
        out = np.zeros(1, dtype=self.dtype)
        U, I = self.X.shape
        _check(getattr(lib(), f"oracle_compute_loss_{sfx}")(
            _p(self.user), _p(self.item), ctypes.c_int64(U), ctypes.c_int64(I),
            ctypes.c_int64(self.K), _p(indptr), _p(indices), _p(data), _p(indptr_t),
            cf(self.alpha0), cf(self.reg), cf(self.nu), ctypes.c_int(self.loss_type),
            ctypes.c_int(n_threads), _p(out)))
        return float(out[0])

    def _compute_loss_feature_aware(self) -> float:
        """:836-940 with feature_aware_: a side that has features is regularised towards its
        prior (reg_u |x_u - f_u W|^2 + lambda |W|^2) instead of towards zero."""
        dt = self.dtype.type
        bias = dt(0) if self.loss_type == LOSS_IALSPP else dt(self.alpha0)
        loss = dt(0)
        if self.alpha0 != 0:
            loss = (gram(self.item, self.alpha0) * gram(self.user, self.alpha0)).sum(dtype=self.dtype) / dt(self.alpha0)
        rows = np.repeat(np.arange(self.X.shape[0]), np.diff(self.X.indptr))
        pred = np.einsum("ij,ij->i", self.user[rows], self.item[self.X.indices]).astype(self.dtype)
        c = self.X.data
        loss += (c * pred * pred - 2 * (c + bias) * pred + c + bias).sum(dtype=self.dtype)
        for side, factor in ((0, self.user), (1, self.item)):
            reg = self._row_reg(side)
            W = self.feature_weight[side]
            if W.shape[0]:
                resid = factor - self._prior(side)
                loss += (reg * (resid * resid).sum(axis=1)).sum(dtype=self.dtype)
                loss += dt(self.lambda_feature[side]) * (W * W).sum(dtype=self.dtype)
            else:
                loss += (reg * (factor * factor).sum(axis=1)).sum(dtype=self.dtype)
        return float(loss / dt(2))

    def epoch_native(self, solver_type=SOLVER_CG, max_cg_steps=3, n_threads=1) -> None:
        """One epoch entirely inside the C++ library (what bench.py times)."""
        sfx, cf = _sfx(self.dtype)
        a = _csr_parts(self.X, self.dtype)
        b = _csr_parts(self.X_t, self.dtype)
        U, I = self.X.shape
        _check(getattr(lib(), f"oracle_epoch_{sfx}")(
            _p(self.user), _p(self.item), ctypes.c_int64(U), ctypes.c_int64(I),
            ctypes.c_int64(self.K), _p(a[0]), _p(a[1]), _p(a[2]), _p(b[0]), _p(b[1]), _p(b[2]),
            cf(self.alpha0), cf(self.reg), cf(self.nu), ctypes.c_int(self.loss_type),
            ctypes.c_int(solver_type), ctypes.c_int(max_cg_steps), ctypes.c_int(n_threads)))


def evaluate(score_block_fn, X_train, ground_truth, cutoff=10, mb_size=128, offset=0,
             recall_with_cutoff=False) -> Tuple[Dict[str, float], np.ndarray]:
    """``Evaluator._get_scores_as_list`` (src/irspack/evaluation/evaluator.py:400-441)
    for one cutoff: chunk loop, seen mask ``scores[mask.nonzero()] = -inf`` (:426-432),
    per-chunk metrics merged.  Returns (metrics dict, top lists int32 n_users x cutoff)."""
    gt = sps.csr_matrix(ground_truth)
    n_users, n_items = gt.shape
    X_train = sps.csr_matrix(X_train)
    total = Metrics(n_items)
    recs: List[np.ndarray] = []
    for b in range(offset, offset + n_users, mb_size):
        e = min(b + mb_size, offset + n_users)
        scores = score_block_fn(b, e)
        mask = X_train[b:e]
        scores[mask.nonzero()] = -np.inf
        m, rec, _ = topk_metrics(scores, gt, cutoff, b - offset, recall_with_cutoff)
        total.merge(m)
        recs.append(rec)
    d = total.as_dict()
    return d, np.concatenate(recs, axis=0) if recs else np.empty((0, cutoff), np.int32)


def retrieve_recommend_from_score(score: np.ndarray, allowed_indices: List[List[int]], cutoff: int
                                  ) -> List[List[Tuple[int, float]]]:
    """numpy restatement of ``retrieve_recommend_from_score<Real>``
    (/root/reference/cpp_source/util.hpp:426-504): per row, candidates = all items or the
    in-range entries of the row's (or the shared) allow-list (:458-478), best ``cutoff`` by
    descending score (:479-485), stop at the first ``-inf`` (:489-491).  The reference's
    comparator leaves the order of equal scores open; this oracle -- like the CUDA path --
    breaks ties by ascending index and counts a repeated allowed index once."""
    score = np.asarray(score)
    rows, n_items = score.shape
    if len(allowed_indices) not in (0, 1, rows):
        raise ValueError("allowed_indices, if not empty, must have a size equal to X.rows()")
    out: List[List[Tuple[int, float]]] = []
    for r in range(rows):
        if allowed_indices:
            src = allowed_indices[0] if len(allowed_indices) == 1 else allowed_indices[r]
            cand = np.unique(np.asarray([i for i in src if 0 <= i < n_items], dtype=np.int64))
        else:
            cand = np.arange(n_items, dtype=np.int64)
        v = score[r, cand]
        keep = v != -np.inf
        cand, v = cand[keep], v[keep]
        order = np.lexsort((cand, -v))[:cutoff]
        out.append([(int(cand[j]), float(v[j])) for j in order])
    return out
