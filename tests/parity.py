"""Shared pieces of the GPU parity suites (test_gpu_parity.py, test_gpu_routes.py,
test_gpu_feature_routes.py): a GPU trainer and its two oracle twins on the same inputs, the stated
comparison, the record of observed errors, the test matrices and hyper-parameter sets, and plain
float64 numpy restatements of the row solves for the cases the oracle does not define (negative
stored values under Cholesky and iALS++, where the reference's sqrt(c) is NaN)."""
import json
import os

import numpy as np
import scipy.sparse as sps

import oracle

_OBSERVED = []
_DUMP_DIR = []  # the directory of the last dump_observed call


def observe(**numbers):
    """Record the observed error of a comparison (written by ``dump_observed``, so that the stated
    tolerances can be read against what holds)."""
    name = os.environ.get("PYTEST_CURRENT_TEST", "?").split("::")[-1].split(" ")[0]
    _OBSERVED.append({"test": name, **{k: float(v) for k, v in numbers.items()}})


def dump_observed(out_dir=None):
    """Write every comparison recorded so far in the session, by every GPU module, to
    ``out_dir/parity_observed.json``.  Without ``out_dir``: $IALS_PARITY_OBSERVED_DIR, else the
    directory of the previous call (test_gpu_parity.py names the suite's output directory), else
    nothing is written."""
    out_dir = out_dir or os.environ.get("IALS_PARITY_OBSERVED_DIR") or (_DUMP_DIR[-1] if _DUMP_DIR else None)
    if out_dir is None:
        return
    _DUMP_DIR.append(out_dir)
    try:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "parity_observed.json"), "w") as f:
            json.dump(_OBSERVED, f, indent=0)
    except OSError:
        pass


def make_pair(core, X, K, alpha0=0.1, reg=0.05, nu=1.0, loss="IALSPP", seed=1):
    """(gpu trainer, f32 oracle, f64 oracle) with identical X and initial factors."""
    from irspack_b200.synth import init_factors

    U, I = X.shape
    u0, i0 = init_factors(U, K, seed), init_factors(I, K, seed + 1)
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(alpha0).set_reg(reg).set_nu(nu)
           .set_loss_type(getattr(core.LossType, loss)).build())
    g = core.IALSTrainer(cfg, X)
    g.user, g.item = u0, i0
    lt = oracle.LOSS_ORIGINAL if loss == "ORIGINAL" else oracle.LOSS_IALSPP
    o32 = oracle.OracleTrainer(X, K, alpha0, reg, nu, lt, dtype=np.float32)
    o64 = oracle.OracleTrainer(X, K, alpha0, reg, nu, lt, dtype=np.float64)
    o32.user, o32.item = u0.copy(), i0.copy()
    o64.user, o64.item = u0.astype(np.float64), i0.astype(np.float64)
    return g, o32, o64


def solver_cfg(core, solver="CG", steps=3, n_threads=1):
    st = core.SolverType.CG if solver == "CG" else core.SolverType.CHOLESKY
    return (core.IALSSolverConfigBuilder().set_solver_type(st).set_max_cg_steps(steps)
            .set_n_threads(n_threads).build())


def assert_close(gpu, o32, o64, tol, guard=4, floor=1e-6):
    """|gpu - f32 oracle| <= tol * scale, widened by twice the f32 oracle's own distance to
    the float64 twin (two float32 evaluations of an ill-conditioned, unconverged CG can
    only agree as well as each agrees with the exact arithmetic), and the GPU result must
    be as close to the float64 twin as the f32 oracle is (factor ``guard``, plus ``floor`` of
    the scale: 1e-6, or 1e-5 where the normal equations come from the 3xTF32 tensor-core Gram,
    whose 2^-22 relative error is multiplied by the condition number of the row's system)."""
    scale = np.abs(o32).max() + 1e-30
    e_ref = np.abs(o32 - o64).max()
    err = np.abs(gpu - o32).max()
    e_gpu = np.abs(gpu - o64).max()
    observe(gpu_vs_f32=err / scale, gpu_vs_f64=e_gpu / scale, f32_vs_f64=e_ref / scale, tol=tol)
    assert err <= tol * scale + 2 * e_ref, f"max err {err:.3e} vs scale {scale:.3e} (f32-vs-f64 {e_ref:.3e})"
    assert e_gpu <= guard * e_ref + floor * scale + 1e-9, (e_gpu, e_ref)


# ---- float64 numpy restatements of the row solves ----

def row_reg(nnz, n_other, alpha0, reg, nu):
    """Solver::compute_reg (IALSTrainer.hpp:117-120): every STORED entry counts, zeros included."""
    return reg * np.power(alpha0 * n_other + np.asarray(nnz, dtype=np.float64), nu)


def np_cholesky_step(target, X, other, alpha0, reg, nu, loss, prior=None):
    """Solver::step_cholesky (:273-331) as closed-form solves: per row u with stored entries (i, c),
    A = alpha0 Y^T Y + sum c y_i y_i^T + reg_u I and b = sum (bias + c) y_i, bias = alpha0 under
    the ORIGINAL loss.  A stored zero adds nothing to A, adds bias y_i to b and 1 to nnz.  Written
    with c y y^T instead of the reference's (sqrt(c) y)(sqrt(c) y)^T, so that a negative c is
    defined.  With ``prior`` (rows like ``target``) it is step_cholesky_with_prior (:333-385): b
    starts from reg_u prior_u, and a row without entries is solved (towards its prior) like the
    others.  Raises like the reference when A is not positive definite; returns a new array in
    the dtype of ``target``."""
    dt = target.dtype
    Y = np.asarray(other, dtype=dt)
    P = dt.type(alpha0) * (Y.T @ Y)
    bias = alpha0 if loss == "ORIGINAL" else 0.0
    out = np.empty_like(target)
    K = target.shape[1]
    for u in range(X.shape[0]):
        s, e = X.indptr[u], X.indptr[u + 1]
        Yr = Y[X.indices[s:e]]
        c = X.data[s:e].astype(dt)
        A = P + (Yr * c[:, None]).T @ Yr + dt.type(row_reg(e - s, Y.shape[0], alpha0, reg, nu)) * np.eye(K, dtype=dt)
        b = Yr.T @ (c + dt.type(bias))
        if prior is not None:
            b = b + dt.type(row_reg(e - s, Y.shape[0], alpha0, reg, nu)) * np.asarray(prior[u], dtype=dt)
        try:
            L = np.linalg.cholesky(A)
        except np.linalg.LinAlgError:
            raise RuntimeError("Cholesky decomposition failed.")
        out[u] = np.linalg.solve(L.T, np.linalg.solve(L, b))
    return out


def np_ialspp_step(target, X, other, alpha0, reg, nu, loss, S, iters):
    """Solver::step_ialspp (:387-535): ``iters`` sweeps of block Gauss-Seidel on the same normal
    equations as ``np_cholesky_step`` (c y y^T, so a negative c is defined), blocks of S
    consecutive dimensions.  A block that is not positive definite raises, as the oracle does.
    Returns a new array in the dtype of ``target``."""
    dt = target.dtype
    Y = np.asarray(other, dtype=dt)
    P = dt.type(alpha0) * (Y.T @ Y)
    bias = dt.type(alpha0 if loss == "ORIGINAL" else 0.0)
    x = target.copy()
    K = target.shape[1]
    for u in range(X.shape[0]):
        s, e = X.indptr[u], X.indptr[u + 1]
        Yr = Y[X.indices[s:e]]
        c = X.data[s:e].astype(dt)
        reg_u = dt.type(row_reg(e - s, Y.shape[0], alpha0, reg, nu))
        for _ in range(iters):
            pred = Yr @ x[u]
            for d0 in range(0, K, S):
                d1 = min(d0 + S, K)
                Ys = Yr[:, d0:d1]
                A = P[d0:d1, d0:d1] + (Ys * c[:, None]).T @ Ys + reg_u * np.eye(d1 - d0, dtype=dt)
                B = P[d0:d1] @ x[u] + reg_u * x[u, d0:d1] + Ys.T @ (c * (pred - 1) - bias)
                try:
                    L = np.linalg.cholesky(A)
                except np.linalg.LinAlgError:
                    raise RuntimeError("Cholesky decomposition failed.")
                delta = np.linalg.solve(L.T, np.linalg.solve(L, B))
                x[u, d0:d1] -= delta
                pred -= Ys @ delta
    return x


# ---- data ----

def fill_empty(X, rng):
    """One entry in every empty row and column (alpha0 = 0 leaves such a row singular)."""
    X = sps.lil_matrix(X)
    U, I = X.shape
    for u in np.flatnonzero(np.diff(sps.csr_matrix(X).indptr) == 0):
        X[u, rng.integers(I)] = 1.0
    Xc = sps.csc_matrix(X)
    for i in np.flatnonzero(np.diff(Xc.indptr) == 0):
        X[rng.integers(U), i] = 1.0
    X = sps.csr_matrix(X, dtype=np.float32)
    X.sort_indices()
    return X


def add_long_rows(X, rng, degrees=(3000, 9000)):
    """Rows 0 and 1 get ``degrees`` neighbours among a widened set of columns."""
    U, I = X.shape
    I2 = max(I, max(degrees) + 200)
    X = sps.lil_matrix(sps.hstack([X, sps.csr_matrix((U, I2 - I), dtype=np.float32)]))
    for u, d in enumerate(degrees):
        X.rows[u] = []
        X.data[u] = []
        cols = np.sort(rng.choice(I2, d, replace=False))
        X.rows[u] = list(cols)
        X.data[u] = list(rng.integers(1, 4, d).astype(np.float32))
    X = sps.csr_matrix(X, dtype=np.float32)
    X.sort_indices()
    return X


def make_data(variant, long_rows=False, seed=3, nnz=12000):
    """500 x 300 counts (1..5, ``nnz`` entries before filling), no empty row or column, in one of the variants:
    counts | zeros: 5 % stored zeros and three rows of stored zeros only |
    neg: 2 % of the values -0.25 | neg1: one value -0.25 | zeros+neg1."""
    from irspack_b200.synth import synth_csr

    rng = np.random.default_rng(seed)
    X = fill_empty(synth_csr(500, 300, nnz, seed=seed, values="counts"), rng)
    if long_rows:
        X = add_long_rows(X, rng)
    if "zeros" in variant:
        X.data[rng.random(X.nnz) < 0.05] = 0.0
        for u in (5, 6, 7):
            X.data[X.indptr[u]:X.indptr[u + 1]] = 0.0
    if variant == "neg":
        X.data[rng.random(X.nnz) < 0.02] = -0.25
    if variant.endswith("neg1"):
        X.data[X.indptr[20] + 1] = -0.25
    return X


def transpose(X):
    Xt = sps.csr_matrix(X.T)
    Xt.sort_indices()
    assert Xt.nnz == X.nnz  # stored zeros survive
    return Xt


# ---- hyper-parameter sets ----

HSETS = {
    # name: (nu, alpha0, reg, loss, perturbations that must move the answer)
    "H0": (0.0, 0.1, 0.05, "IALSPP", ({"nu": 0.25},)),
    "H1": (0.5, 2.0, 0.02, "ORIGINAL", ({"nu": 0.75}, {"loss": "IALSPP"})),
    "H2": (2.0, 0.05, None, "IALSPP", ({"nu": 1.75},)),  # reg: see balanced_reg
    "H3": (1.0, 0.0, 0.05, "ORIGINAL", ({"alpha0": 0.05},)),
}


def balanced_reg(X, K, alpha0, nu):
    """reg at which reg_u of a median user row equals the mean diagonal of its Gram
    alpha0 Y^T Y + sum c y y^T at the initial item factors, so neither the ridge nor the data
    term dominates the row's system."""
    from irspack_b200.synth import init_factors

    Y = init_factors(X.shape[1], K, 2).astype(np.float64)
    nnz = np.diff(X.indptr)
    u = int(np.argsort(nnz)[len(nnz) // 2])
    s, e = X.indptr[u], X.indptr[u + 1]
    Yr = Y[X.indices[s:e]]
    diag = alpha0 * (Y * Y).sum() / K + (np.abs(X.data[s:e])[:, None] * Yr * Yr).sum() / K
    return float(diag / (alpha0 * X.shape[1] + (e - s)) ** nu)


def hparams(name, X, K):
    nu, alpha0, reg, loss, perturb = HSETS[name]
    if reg is None:
        reg = balanced_reg(X, K, alpha0, nu)
    return dict(nu=nu, alpha0=alpha0, reg=reg, loss=loss), perturb


def ridge_f64(F, factors, row_weights, lam):
    """The feature weights' ridge refit W = (F^T D F + lam I)^-1 F^T D X in float64
    (oracle.feature_ridge on float64 arrays), D = diag(row_weights)."""
    return oracle.feature_ridge(F, np.asarray(factors, dtype=np.float64), np.asarray(row_weights, dtype=np.float64),
                                lam)
