"""Feature-aware iALS on the CUDA path against the oracle, at every row stride, hyper-parameter set and
feature shape its kernels meet.

When a side has features its rows go to the generic kernels, which take a prior: cg_warp_kernel<ld / 32>
for CG at every row stride (stride 128, K <= 128, included) and cholesky_tile_kernel for Cholesky at
every K <= 256 (K = 256 included).  feature.cu forms the prior F W, the row weights, the Cholesky factor
of F^T D F + lambda I, the right-hand side F^T D X and the triangular solves of the weight refit.

* Every case starts from random non-zero feature weights set through the setter (no warm-up), scaled
  so that F W has the magnitude of the factors the row solve produces: the first solve already has a
  prior that matters.  Both sides have features, dense on one and CSR on the other.
* Factors are compared with the oracle's step with ``prior=``; the refit weights with the f32 / f64
  ridge of the GPU's own new factors, which isolates feature.cu from the solve; transform_*_feature
  with F @ W in float64.  Each case also shows that it depends on what it tests: the f64 step without
  the prior, and the ridge with lambda doubled, must be more than ten tolerances away.
* Each half-step confirms its route from the number of kernels it launches.

For a negative stored value under Cholesky the reference forms sqrt(c) y and raises; the CUDA route
forms c y y^T, so those cases are compared with parity.np_cholesky_step (with the prior).
"""
import copy

import numpy as np
import pytest
import scipy.sparse as sps

import oracle
from parity import (HSETS, add_long_rows, assert_close, balanced_reg, dump_observed, hparams, make_data,
                    np_cholesky_step, observe, ridge_f64, solver_cfg, transpose)

pytestmark = pytest.mark.gpu

TOL_STEP = 2e-4
SENSITIVITY = 10  # a perturbed input must move the f64 answer by more than this many tolerances
# The refit sums every row's contribution to F^T D F and F^T D X with fp32 atomics in any order: the
# floor of the f64 guard is 1e-5 of the scale there, as for the tensor-core Gram of the routes suite.
FLOOR_W = 1e-5
TOL_PRIOR = 1e-5  # F W: a float32 dot product of one feature row, against float64
NF = (40, 33)  # feature columns of the user and the item side (33: two passes of a warp's lanes)


@pytest.fixture(scope="module")
def core():
    import irspack_b200

    if irspack_b200.device_count() == 0:
        pytest.fail("GPU test selected but no CUDA device is visible")
    from irspack_b200 import _ials_core

    return _ials_core


@pytest.fixture(scope="module", autouse=True)
def _dump_observed():
    yield
    dump_observed()


def launches():
    from irspack_b200._lib import lib

    return int(lib.ials_kernel_launch_count())


# Kernels launched by one feature-aware half-step (ials_kernel_launch_count):
#   Gram P = alpha0 Y^T Y: 3 at row stride 128 (block_jobs_kernel + wgram_kernel + wgram_reduce_sym_kernel,
#     launch_gram_tc), 2 at other strides (gram_tile_kernel + gram_finalize_kernel, gram.cu);
#   the prior F W: feature_prior_kernel (1);
#   the solve: a prior sends every row to cg_warp_kernel or cholesky_tile_kernel (1, solve_unphased);
#   the weight update: on a side's first call feature_row_weights_kernel + feature_gram_kernel +
#     feature_add_diag_kernel + feature_llt_kernel (the cached factor) + feature_rhs_kernel +
#     feature_solve_kernel (6), then feature_rhs_kernel + feature_solve_kernel (2).
def ld_of(K):
    return 128 if K <= 128 else -(-K // 32) * 32


def feature_half_step_launches(K, first=True):
    return (3 if ld_of(K) == 128 else 2) + 1 + 1 + (6 if first else 2)


# ---- data ----

def feature_matrix(n, nf, kind, seed, density=0.5):
    """n x nf features of unit scale (standard normal entries, ``density`` of them stored)."""
    rng = np.random.default_rng(seed)
    F = (rng.standard_normal((n, nf)) * (rng.random((n, nf)) < density)).astype(np.float32)
    return sps.csr_matrix(F) if kind == "csr" else F


def dense64(F):
    return np.asarray(F.toarray() if sps.issparse(F) else F, dtype=np.float64)


def row_weights(Xs, n_other, p, dtype=np.float64):
    """compute_reg of every row of Xs: the D of the ridge (stored zeros count)."""
    return oracle.compute_reg(np.diff(Xs.indptr), n_other, p["alpha0"], p["reg"], p["nu"], dtype)


def balanced_lambda(F, rw):
    """lambda = the mean diagonal of F^T D F: the ridge then matters (doubling it moves W by tens of
    percents) and F^T D F + lambda I stays well conditioned whatever the feature shape."""
    d = (dense64(F) ** 2 * rw[:, None]).sum(axis=0)
    return float(max(d.mean(), 1e-3))


def scaled_weight(F, target_rms, K, seed):
    """Random weights whose F W has the root mean square ``target_rms``."""
    W = np.random.default_rng(seed).standard_normal((F.shape[1], K))
    FW = dense64(F) @ W
    rms = np.sqrt((FW ** 2).mean())
    return (W * (target_rms / rms if rms > 0 else 1.0)).astype(np.float32)


def prior_of(F, W, dtype):
    """F W as the oracle forms it (OracleTrainer._prior), in ``dtype``."""
    F = sps.csr_matrix(F, dtype=dtype) if sps.issparse(F) else np.asarray(F, dtype=dtype)
    return np.ascontiguousarray(np.asarray(F @ np.asarray(W, dtype=dtype)), dtype=dtype)


def reference(solver, target, Xs, other, p, dtype, prior, steps=3, negative=False):
    """One half-epoch of ``solver`` on ``target`` (rows of Xs) against ``prior`` (None: the plain
    step), in ``dtype``: the oracle, or the numpy restatement where a negative value leaves the
    oracle's Cholesky undefined."""
    nt = oracle.hardware_threads()
    t = np.array(target, dtype=dtype)
    oth = np.ascontiguousarray(other, dtype=dtype)
    pr = None if prior is None else np.ascontiguousarray(prior, dtype=dtype)
    lt = oracle.LOSS_ORIGINAL if p["loss"] == "ORIGINAL" else oracle.LOSS_IALSPP
    if solver == "CG":
        oracle.step_cg(t, Xs, oth, oracle.gram(oth, p["alpha0"], nt), p["alpha0"], p["reg"], p["nu"], lt, steps, nt,
                       prior=pr)
    elif negative:
        t = np_cholesky_step(t, Xs, oth, p["alpha0"], p["reg"], p["nu"], p["loss"], prior=pr)
    else:
        oracle.step_cholesky(t, Xs, oth, oracle.gram(oth, p["alpha0"], nt), p["alpha0"], p["reg"], p["nu"], lt, nt,
                             prior=pr)
    return t


def feature_trainer(core, X, K, p, Fs, lams, warmup=0, seed=1):
    """(gpu trainer, f32 oracle, f64 oracle) with features, identical X and initial factors."""
    from irspack_b200.synth import init_factors

    U, I = X.shape
    u0, i0 = init_factors(U, K, seed), init_factors(I, K, seed + 1)
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(p["alpha0"]).set_reg(p["reg"]).set_nu(p["nu"])
           .set_loss_type(getattr(core.LossType, p["loss"])).set_lambda_user_feature(lams[0])
           .set_lambda_item_feature(lams[1]).set_feature_warmup_epochs(warmup).build())
    g = core.IALSTrainer(cfg, X, Fs[0], Fs[1])
    g.user, g.item = u0, i0
    lt = oracle.LOSS_ORIGINAL if p["loss"] == "ORIGINAL" else oracle.LOSS_IALSPP
    twins = []
    for dt in (np.float32, np.float64):
        o = oracle.OracleTrainer(X, K, p["alpha0"], p["reg"], p["nu"], lt, dtype=dt, user_features=Fs[0],
                                 item_features=Fs[1], lambda_user_feature=lams[0], lambda_item_feature=lams[1],
                                 feature_warmup_epochs=warmup)
        o.user, o.item = u0.astype(dt), i0.astype(dt)
        twins.append(o)
    return (g, *twins)


def set_weights(trainers, Ws):
    g, o32, o64 = trainers
    g.user_feature_weight, g.item_feature_weight = Ws
    for o in (o32, o64):
        o.feature_weight = [np.asarray(W, dtype=o.dtype) for W in Ws]


def weight_of(g, side):
    return g.user_feature_weight if side == 0 else g.item_feature_weight


def check_refit(g, side, F, got_factors, rw64, lam):
    """The refit weights against the f32 / f64 ridge of the GPU's own new factors, and lambda doubled
    must be far; transform_*_feature(F) against F @ W in float64."""
    W = weight_of(g, side)
    want32 = oracle.feature_ridge(F, np.asarray(got_factors, np.float32), rw64.astype(np.float32), lam)
    want64 = ridge_f64(F, got_factors, rw64, lam)
    assert_close(W, want32, want64, TOL_STEP, floor=FLOOR_W)
    moved = ridge_f64(F, got_factors, rw64, 2 * lam)
    dist = np.abs(W - moved).max() / np.abs(want64).max()
    observe(sensitivity=dist, tol=TOL_STEP)
    assert dist > SENSITIVITY * TOL_STEP, ("lambda", side, dist)
    fw = g.transform_user_feature(F) if side == 0 else g.transform_item_feature(F)
    want = dense64(F) @ W.astype(np.float64)
    err = np.abs(fw - want).max() / (np.abs(want).max() + 1e-30)
    observe(prior_vs_f64=err, tol=TOL_PRIOR)
    assert err <= TOL_PRIOR, err


def run_half_steps(core, solver, K, X, p, kinds, steps=3, negative=False, perturb=(), nf=NF, Fs=None):
    """One half-step per side from the initial factors of the other side, with random weights set
    through the setter: factors, refit weights and F W against the references, sensitivity to the prior
    (and to each parameter change in ``perturb``), and the route from the launch count."""
    from irspack_b200.synth import init_factors

    U, I = X.shape
    Xt = transpose(X)
    if Fs is None:
        Fs = [feature_matrix(U, nf[0], kinds[0], seed=11), feature_matrix(I, nf[1], kinds[1], seed=12)]
    rws = [row_weights(X, I, p), row_weights(Xt, U, p)]
    lams = [balanced_lambda(F, rw) for F, rw in zip(Fs, rws)]
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    sides = ((X, u0, i0), (Xt, i0, u0))
    # the f64 half-steps with a zero prior: the magnitude the priors are scaled to, and the answer the
    # GPU's must be far from
    plain = [reference(solver, t, Xs, o, p, np.float64, np.zeros(t.shape), steps, negative) for Xs, t, o in sides]
    Ws = [scaled_weight(F, np.sqrt((pl ** 2).mean()), K, seed=20 + s) for s, (F, pl) in enumerate(zip(Fs, plain))]
    trainers = feature_trainer(core, X, K, p, Fs, lams)
    g = trainers[0]
    set_weights(trainers, Ws)
    sc = solver_cfg(core, solver, steps)
    result = dict(g=g, Fs=Fs, Ws=Ws, got=[])
    for side, (Xs, target, other) in enumerate(sides):
        if side == 1:
            g.user = u0  # the item half-step starts from the initial user factors, as the references do
        before = launches()
        g.half_step(side, sc)
        delta = launches() - before
        assert delta == feature_half_step_launches(K), (side, delta)
        got = g.user if side == 0 else g.item
        result["got"].append(got)
        want = [reference(solver, target, Xs, other, p, dt, prior_of(Fs[side], Ws[side], dt), steps, negative)
                for dt in (np.float32, np.float64)]
        assert_close(got, *want, TOL_STEP)
        scale = np.abs(want[0]).max()
        changes = [(None, plain[side])]
        prior64 = prior_of(Fs[side], Ws[side], np.float64)
        for change in perturb:
            changes.append((change, reference(solver, target, Xs, other, {**p, **change}, np.float64, prior64, steps,
                                              negative)))
        for change, moved in changes:
            dist = np.abs(got - moved).max() / scale
            observe(sensitivity=dist, tol=TOL_STEP)
            assert dist > SENSITIVITY * TOL_STEP, (side, change or "prior", dist)
        check_refit(g, side, Fs[side], got, rws[side], lams[side])
    return result


KINDS = {"dense_csr": ("dense", "csr"), "csr_dense": ("csr", "dense")}
P_BASE = dict(nu=1.0, alpha0=0.1, reg=0.05, loss="ORIGINAL")


# ---- 1. every kernel the prior reaches ----

# CG: row strides 128 (K = 40: padded; K = 128: full), 224, 256, 320, 480, 512 -> cg_warp_kernel<NV>,
# NV = 4, 4, 7, 8, 10, 15, 16.  Cholesky: cholesky_tile_kernel<0> with a system of kd = 64 (> K = 60:
# the prior's k < K guard), 128, 200, 256.
KERNEL_CASES = [("CG", K) for K in (40, 128, 200, 256, 300, 480, 512)] + \
               [("CHOLESKY", K) for K in (60, 128, 200, 256)]


@pytest.mark.parametrize("kinds", list(KINDS))
@pytest.mark.parametrize("solver,K", KERNEL_CASES, ids=[f"{s}-{K}" for s, K in KERNEL_CASES])
def test_prior_kernels(core, solver, K, kinds):
    run_half_steps(core, solver, K, make_data("counts"), P_BASE, KINDS[kinds])


def test_cholesky_above_256_with_features_is_not_implemented(core):
    X = make_data("counts")
    U, I = X.shape
    Fs = [feature_matrix(U, 4, "dense", 1), feature_matrix(I, 3, "csr", 2)]
    g = feature_trainer(core, X, 257, P_BASE, Fs, (1.0, 1.0))[0]
    with pytest.raises(NotImplementedError, match="Cholesky solver: n_components > 256 not supported"):
        g.half_step(0, solver_cfg(core, "CHOLESKY"))


# ---- 2. hyper-parameters and data ----

HP_CASES = [("CG", 128), ("CG", 300), ("CHOLESKY", 64), ("CHOLESKY", 256)]
# H2's ridge is only as large as the data term: with a confidence of -0.25 the row's matrix is then
# indefinite, so H2 runs on the positive variants only (as in test_gpu_routes.py)
HP_PARAMS = [pytest.param(s, K, v, h, id=f"{s}-{K}-{v}-{h}") for s, K in HP_CASES for v in ("counts", "zeros", "neg")
             for h in HSETS if not (v == "neg" and h == "H2")]


@pytest.mark.parametrize("solver,K,variant,hset", HP_PARAMS)
def test_hyper_parameters_and_data(core, solver, K, variant, hset):
    """HSETS (nu = 0, 0.5, 2, 1; alpha0 = 0 in H3; both losses) on counts, counts with stored zeros
    (three rows of stored zeros only: they count in nnz, so in the row weights of the ridge) and counts
    with negative values; each listed perturbation must move the answer."""
    X = make_data(variant)
    p, perturb = hparams(hset, X, K)
    kinds = KINDS["dense_csr"] if hset in ("H0", "H2") else KINDS["csr_dense"]
    run_half_steps(core, solver, K, X, p, kinds, negative=variant == "neg", perturb=perturb)


# ---- 3. rows the prior treats differently ----

def with_empty_rows(X, rows=(40, 41, 42), cols=(7,)):
    """X without any entry in ``rows`` and ``cols``; the other stored zeros stay."""
    X = sps.coo_matrix(X)
    keep = ~np.isin(X.row, rows) & ~np.isin(X.col, cols)
    X = sps.csr_matrix((X.data[keep], (X.row[keep], X.col[keep])), shape=X.shape, dtype=np.float32)
    X.sort_indices()
    return X


@pytest.mark.parametrize("solver,K", [("CG", 128), ("CHOLESKY", 256)])
def test_empty_rows_are_solved_towards_their_prior(core, solver, K):
    """Users 40..42 and item 7 have no interactions.  At alpha0 = 0 and nu = 0 an empty row's system is
    reg I x = reg prior: its answer is the prior F W itself, to float32 rounding.  Every row also
    against the oracle."""
    X = with_empty_rows(make_data("counts"))
    p = dict(nu=0.0, alpha0=0.0, reg=0.05, loss="IALSPP")
    r = run_half_steps(core, solver, K, X, p, KINDS["dense_csr"])
    for side, rows in ((0, [40, 41, 42]), (1, [7])):
        want = dense64(r["Fs"][side])[rows] @ r["Ws"][side].astype(np.float64)
        err = np.abs(r["got"][side][rows] - want).max() / np.abs(want).max()
        observe(empty_row_vs_prior=err, tol=TOL_PRIOR)
        assert err <= TOL_PRIOR, (side, err)


def test_empty_row_without_ridge_raises(core):
    """At alpha0 = 0 and nu > 0 an empty row has reg_u = 0 and no unique embedding: step, half_step and
    transform_*_with_feature raise the reference's error; the oracle raises the same."""
    X = with_empty_rows(make_data("counts"))
    U, I = X.shape
    p = dict(nu=1.0, alpha0=0.0, reg=0.05, loss="IALSPP")
    Fs = [feature_matrix(U, 5, "dense", 11), feature_matrix(I, 4, "csr", 12)]
    g, o32, _ = feature_trainer(core, X, 128, p, Fs, (1.0, 1.0))
    msg = "not uniquely defined for an empty interaction row"
    with pytest.raises(ValueError, match=msg) as want:
        o32.step(oracle.SOLVER_CG, 3)
    sc = solver_cfg(core, "CG", 3)
    for call in (lambda: g.step(sc), lambda: g.half_step(0, sc), lambda: g.half_step(1, sc)):
        with pytest.raises(ValueError) as got:
            call()
        assert str(got.value) == str(want.value)
    Xnew = make_data("counts", seed=9)[:20]
    Xnew = with_empty_rows(Xnew, rows=(3,), cols=())
    with pytest.raises(ValueError, match=msg):
        g.transform_user_with_feature(Xnew, feature_matrix(20, 5, "dense", 5), sc)
    Xi = with_empty_rows(make_data("counts", seed=9)[:, :20], rows=(), cols=(4,))
    with pytest.raises(ValueError, match=msg):
        g.transform_item_with_feature(Xi, feature_matrix(20, 4, "csr", 6), sc)


@pytest.mark.parametrize("solver", ["CG", "CHOLESKY"])
def test_rows_of_stored_zeros_are_not_empty(core, solver):
    """Rows 5, 6, 7 hold stored zeros only: they count in nnz, so at alpha0 = 0 and nu = 1 their ridge
    is reg * nnz > 0.  Nothing raises, and every row matches the oracle."""
    X = make_data("zeros")
    assert all(X.indptr[u + 1] > X.indptr[u] and not X.data[X.indptr[u]:X.indptr[u + 1]].any() for u in (5, 6, 7))
    p = dict(nu=1.0, alpha0=0.0, reg=0.05, loss="ORIGINAL")
    run_half_steps(core, solver, 128, X, p, KINDS["csr_dense"])


@pytest.mark.parametrize("feature_side", [0, 1])
def test_long_rows_stay_on_the_prior_kernel(core, monkeypatch, feature_side):
    """Rows of 3000 and 9000 neighbours at K = 128 with IALS_HEAVY_THRESHOLD=64: the side with features
    takes cg_warp_kernel for every row (no wgram, no dense CG); the side without features (0 columns)
    still takes the heavy path.  Both match the oracle."""
    monkeypatch.setenv("IALS_HEAVY_THRESHOLD", "64")
    X = add_long_rows(make_data("counts", nnz=30000), np.random.default_rng(8))
    Xt = transpose(X)
    U, I = X.shape
    K, p = 128, P_BASE
    n = (U, I)
    Fs = [sps.csr_matrix((n[s], 0), dtype=np.float32) for s in (0, 1)]
    Fs[feature_side] = feature_matrix(n[feature_side], 24, "dense", 13)
    trainers = feature_trainer(core, X, K, p, Fs, (1.0, 1.0))
    g, o32, o64 = trainers
    stats = [g.plan_stats(s) for s in (0, 1)]
    assert min(s["heavy_rows"] for s in stats) >= 2 and max(s["max_degree"] for s in stats) >= 9000, stats
    W = scaled_weight(Fs[feature_side], 0.1, K, seed=40)
    if feature_side == 0:
        g.user_feature_weight = W
    else:
        g.item_feature_weight = W
    for o in (o32, o64):
        o.feature_weight[feature_side] = W.astype(o.dtype)
    u0 = g.user.copy()
    sc = solver_cfg(core, "CG", 3)
    for side, (Xs, other) in enumerate(((X, o64.item), (Xt, u0))):
        if side == 1:
            g.user = u0
        target = o64.user if side == 0 else o64.item
        before = launches()
        g.half_step(side, sc)
        delta = launches() - before
        if side == feature_side:
            assert delta == feature_half_step_launches(K), delta
            prior = [prior_of(Fs[side], W, dt) for dt in (np.float32, np.float64)]
            floor = 1e-6
        else:  # Gram + wgram + dense CG, + cg_rows_kernel when light rows are left
            assert delta == 3 + 2 + (stats[side]["rows"] > stats[side]["heavy_rows"]), delta
            prior = [None, None]
            floor = 1e-5  # the heavy rows' normal equations come from the 3xTF32 tensor-core Gram
        got = g.user if side == 0 else g.item
        want = [reference("CG", target, Xs, other, p, dt, pr) for dt, pr in zip((np.float32, np.float64), prior)]
        assert_close(got, *want, TOL_STEP, floor=floor)


# ---- 4. feature matrix shapes ----

def shaped_features(n, nf, form, seed):
    """Unit-scale features in one of two forms.  csr: 30 % density, every third row empty, 5 % stored
    zeros, the signs of a standard normal, and row 1 holding every column.  dense: 60 % density and an
    all-zero column (when there is more than one), whose Gram diagonal is lambda alone."""
    rng = np.random.default_rng(seed)
    if form == "dense":
        F = (rng.standard_normal((n, nf)) * (rng.random((n, nf)) < 0.6)).astype(np.float32)
        if nf > 1:
            F[:, nf // 2] = 0.0
        return F
    F = sps.lil_matrix(sps.random(n, nf, density=0.3, random_state=seed, dtype=np.float32,
                                  data_rvs=rng.standard_normal))
    F[np.arange(0, n, 3), :] = 0
    F = sps.csr_matrix(F)
    F.eliminate_zeros()
    full = sps.lil_matrix(F)
    full[1, :] = rng.standard_normal(nf).astype(np.float32)
    F = sps.csr_matrix(full, dtype=np.float32)
    F.data[rng.random(F.nnz) < 0.05] = 0.0  # stored zeros (kept: no eliminate_zeros after this)
    F.sort_indices()
    assert F.indptr[2] - F.indptr[1] == nf and F.indptr[1] == F.indptr[0]
    return F


@pytest.mark.parametrize("form", ["csr", "dense"])
@pytest.mark.parametrize("nf", [1, 33, 300, 1100])
def test_feature_shapes(core, nf, form):
    """1 column; 33 (> one pass of a warp's lanes in feature_gram_kernel); 300; 1100 (> the 1024 threads
    of feature_llt_kernel) -- on both sides, CG at K = 128."""
    X = make_data("counts")
    U, I = X.shape
    Fs = [shaped_features(U, nf, form, 50), shaped_features(I, nf, form, 51)]
    run_half_steps(core, "CG", 128, X, P_BASE, None, Fs=Fs)


# ---- 5. epochs and the loss ----

EPOCH_CASES = {"cg_k128_s3": ("CG", 128, 3), "cg_k128_s0": ("CG", 128, 0), "cholesky_k256": ("CHOLESKY", 256, 3)}


@pytest.mark.parametrize("kinds", list(KINDS))
@pytest.mark.parametrize("case", list(EPOCH_CASES))
def test_epochs_and_loss(core, case, kinds):
    """Four epochs, two of them warm-up: after each, both sides against the f32 / f64 oracle and
    compute_loss against the f64 oracle's loss at the GPU's state.  During the warm-up the factors are
    those of a plain trainer and the weights stay zero."""
    solver, K, steps = EPOCH_CASES[case]
    X = make_data("zeros")
    U, I = X.shape
    p = dict(nu=1.0, alpha0=0.1, reg=0.05, loss="IALSPP")
    Fs = [feature_matrix(U, NF[0], KINDS[kinds][0], 11), feature_matrix(I, NF[1], KINDS[kinds][1], 12)]
    lams = (0.3, 0.2)
    g, o32, o64 = feature_trainer(core, X, K, p, Fs, lams, warmup=2)
    plain = core.IALSTrainer(core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.05).set_nu(1.0)
                             .set_loss_type(core.LossType.IALSPP).build(), X)
    plain.user, plain.item = g.user, g.item
    lt = oracle.LOSS_IALSPP
    lo = oracle.OracleTrainer(X, K, 0.1, 0.05, 1.0, lt, dtype=np.float64, user_features=Fs[0], item_features=Fs[1],
                              lambda_user_feature=lams[0], lambda_item_feature=lams[1])
    sc = solver_cfg(core, solver, steps)
    osolver = oracle.SOLVER_CG if solver == "CG" else oracle.SOLVER_CHOLESKY
    for epoch in range(4):
        g.step(sc)
        for o in (o32, o64):
            o.step(osolver, steps)
        assert_close(g.user, o32.user, o64.user, TOL_STEP)
        assert_close(g.item, o32.item, o64.item, TOL_STEP)
        if epoch < 2:
            plain.step(sc)
            if ld_of(K) == 128:
                np.testing.assert_array_equal(g.user, plain.user)
                np.testing.assert_array_equal(g.item, plain.item)
            else:  # the SIMT Gram adds its per-CTA tiles with atomics
                for a, b in ((g.user, plain.user), (g.item, plain.item)):
                    np.testing.assert_allclose(a, b, rtol=0, atol=TOL_STEP * np.abs(b).max())
            assert not g.user_feature_weight.any() and not g.item_feature_weight.any()
        else:
            assert_close(g.user_feature_weight, o32.user_feature_weight, o64.user_feature_weight, TOL_STEP,
                         floor=FLOOR_W)
            assert_close(g.item_feature_weight, o32.item_feature_weight, o64.item_feature_weight, TOL_STEP,
                         floor=FLOOR_W)
        lo.user, lo.item = g.user.astype(np.float64), g.item.astype(np.float64)
        lo.feature_weight = [g.user_feature_weight.astype(np.float64), g.item_feature_weight.astype(np.float64)]
        got, ref = g.compute_loss(sc), lo.compute_loss()
        observe(loss_rel=abs(got - ref) / abs(ref), tol=1e-4)
        assert got == pytest.approx(ref, rel=1e-4)


# ---- 6. the other entry points ----

@pytest.mark.parametrize("feature_side", [0, 1])
def test_step_io_across_the_warm_up(core, feature_side):
    """step_io against set + step + get on a feature-aware trainer, across the end of a one-epoch
    warm-up.  User features only: after the warm-up the user half-epoch has a prior and the overlapped
    upload is off.  Item features only: the user side keeps the overlapped upload.  Within tolerance,
    not bitwise: feature_gram_kernel and feature_rhs_kernel add with fp32 atomics."""
    X = make_data("counts")
    U, I = X.shape
    n = (U, I)
    K = 128
    Fs = [sps.csr_matrix((n[s], 0), dtype=np.float32) for s in (0, 1)]
    Fs[feature_side] = feature_matrix(n[feature_side], 24, "csr", 14)
    p = dict(nu=1.0, alpha0=0.1, reg=0.05, loss="IALSPP")
    g = feature_trainer(core, X, K, p, Fs, (0.5, 0.5), warmup=1)[0]
    h = feature_trainer(core, X, K, p, Fs, (0.5, 0.5), warmup=1)[0]
    sc = solver_cfg(core, "CG", 3)

    def same(a, b):
        np.testing.assert_allclose(a, b, rtol=0, atol=TOL_STEP * np.abs(b).max())

    u, v = h.user.copy(), h.item.copy()
    for call in ("io", "io", "step", "io"):
        g.step(sc)
        if call == "io":
            h.step_io(sc, u, v)
        else:
            h.step(sc)
            u, v = h.user.copy(), h.item.copy()
        same(u, g.user)
        same(v, g.item)
        same(weight_of(h, feature_side), weight_of(g, feature_side))
    assert weight_of(g, feature_side).any()


TRANSFORM_CASES = [("CG", 128, 5), ("CG", 128, 0), ("CG", 300, 5), ("CG", 300, 0), ("CHOLESKY", 128, 3),
                   ("CHOLESKY", 256, 3), ("CG", 128, 1), ("CG", 300, 2)]


@pytest.mark.parametrize("solver,K,steps", TRANSFORM_CASES, ids=[f"{s}-{K}-{n}" for s, K, n in TRANSFORM_CASES])
def test_transform_with_feature(core, solver, K, steps):
    """transform_user_with_feature / transform_item_with_feature against the oracle: new rows, two of
    them without interactions, with a feature matrix that is not the training one.  With one or two CG
    steps the ridge is no larger than the data term, so the rows are far from converged and their
    answer depends on the warm start, which is the prior: the f64 fold-in from zero must be far away."""
    X = make_data("counts")
    U, I = X.shape
    early = solver == "CG" and steps in (1, 2)
    p = dict(P_BASE, reg=balanced_reg(X, K, P_BASE["alpha0"], P_BASE["nu"])) if early else P_BASE
    Fs = [feature_matrix(U, NF[0], "dense", 11), feature_matrix(I, NF[1], "csr", 12)]
    trainers = feature_trainer(core, X, K, p, Fs, (1.0, 1.0))
    g, o32, o64 = trainers
    Ws = [scaled_weight(F, 1.0, K, seed=60 + s) for s, F in enumerate(Fs)]
    set_weights(trainers, Ws)
    sc = solver_cfg(core, solver, steps)
    osolver = oracle.SOLVER_CG if solver == "CG" else oracle.SOLVER_CHOLESKY
    Xu = with_empty_rows(make_data("zeros", seed=9)[:60], rows=(3, 17), cols=())
    Fu = feature_matrix(60, NF[0], "csr", 70)
    got = g.transform_user_with_feature(Xu, Fu, sc)
    want = [o.transform_user_with_feature(Xu, Fu, osolver, steps) for o in (o32, o64)]
    assert_close(got, *want, TOL_STEP)
    if early:
        from_zero = np.zeros((60, K))
        oracle.step_cg(from_zero, Xu, o64.item, oracle.gram(o64.item, p["alpha0"]), p["alpha0"], p["reg"], p["nu"],
                       oracle.LOSS_ORIGINAL, steps, prior=prior_of(Fu, Ws[0], np.float64))
        dist = np.abs(got - from_zero).max() / np.abs(want[0]).max()
        observe(sensitivity=dist, tol=TOL_STEP)
        assert dist > SENSITIVITY * TOL_STEP, dist
    Xi = with_empty_rows(make_data("zeros", seed=10)[:, :50], rows=(), cols=(3, 17))
    Fi = feature_matrix(50, NF[1], "dense", 71)
    got = g.transform_item_with_feature(Xi, Fi, sc)
    want = [o.transform_item_with_feature(Xi, Fi, osolver, steps) for o in (o32, o64)]
    assert_close(got, *want, TOL_STEP)


def test_rejections(core):
    """IALSPP on a feature-aware trainer, and a fold-in feature matrix whose rows are not the new rows."""
    X = make_data("counts")
    U, I = X.shape
    Fs = [feature_matrix(U, 5, "dense", 11), feature_matrix(I, 4, "csr", 12)]
    g = feature_trainer(core, X, 128, P_BASE, Fs, (1.0, 1.0))[0]
    ialspp = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP).build())
    for call in (lambda: g.step(ialspp), lambda: g.half_step(0, ialspp),
                 lambda: g.transform_user_with_feature(X[:4], Fs[0][:4], ialspp)):
        with pytest.raises(ValueError, match="Feature-aware iALS does not support IALSPP."):
            call()
    with pytest.raises(ValueError, match="Feature prior shape does not match X."):
        g.transform_user_with_feature(X[:4], Fs[0][:5], solver_cfg(core))
    with pytest.raises(ValueError, match="Feature prior shape does not match X."):
        g.transform_item_with_feature(X[:, :4], Fs[1][:3], solver_cfg(core))


@pytest.mark.parametrize("side,rows", [(0, 3), (1, 7), (1, 0)], ids=["user-3", "item-7", "item-empty"])
def test_weight_shape_mismatch(core, side, rows):
    """A feature weight whose row count is not the side's feature columns (the item side of the last
    case has no features at all, and gets rows) is accepted by the setter, as the reference's def_rw
    does; the next step, half_step, step_io or compute_loss raises the oracle's error before it launches
    anything and leaves both factor matrices as they were.  A weight of the right shape trains again."""
    X = make_data("counts")
    U, I = X.shape
    nf = (5, 0 if rows == 0 else 4)
    rows = rows or 3
    Fs = [feature_matrix(U, nf[0], "dense", 11),
          feature_matrix(I, nf[1], "csr", 12) if nf[1] else sps.csr_matrix((I, 0), dtype=np.float32)]
    K = 128
    trainers = feature_trainer(core, X, K, P_BASE, Fs, (1.0, 1.0))
    g, o32, o64 = trainers
    bad = np.random.default_rng(3).standard_normal((rows, K)).astype(np.float32)
    if side == 0:
        g.user_feature_weight = bad
    else:
        g.item_feature_weight = bad
    # the oracle raises when it forms the prior, after the half-epochs before it: a copy of the f32 twin
    # gives the message, and the twins themselves stay at the initial state
    o_bad = copy.deepcopy(o32)
    o_bad.feature_weight[side] = bad.copy()
    assert weight_of(g, side).shape == (rows, K)
    with pytest.raises(ValueError) as want:
        o_bad.step(oracle.SOLVER_CG, 3)
    assert str(want.value).startswith("Shape mismatch")
    u0, i0 = g.user.copy(), g.item.copy()
    sc = solver_cfg(core, "CG", 3)
    u_in, i_in = u0 + 1.0, i0 + 1.0
    calls = {"step": lambda: g.step(sc), "half_step_user": lambda: g.half_step(0, sc),
             "half_step_item": lambda: g.half_step(1, sc), "step_io": lambda: g.step_io(sc, u_in.copy(), i_in.copy()),
             "compute_loss": lambda: g.compute_loss(sc)}
    for name, call in calls.items():
        before = launches()
        with pytest.raises(ValueError) as got:
            call()
        assert str(got.value) == str(want.value), name
        assert launches() == before, name
        np.testing.assert_array_equal(g.user, u0, err_msg=name)
        np.testing.assert_array_equal(g.item, i0, err_msg=name)
    # the right shape: the trainer trains again, as the oracle does
    good = np.random.default_rng(4).standard_normal((nf[side], K)).astype(np.float32) * 0.01
    if side == 0:
        g.user_feature_weight = good
    else:
        g.item_feature_weight = good
    for o in (o32, o64):
        o.feature_weight[side] = good.astype(o.dtype)
    g.step(sc)
    for o in (o32, o64):
        o.step(oracle.SOLVER_CG, 3)
    assert_close(g.user, o32.user, o64.user, TOL_STEP)
    assert_close(g.item, o32.item, o64.item, TOL_STEP)
    assert np.isfinite(g.compute_loss(sc))
