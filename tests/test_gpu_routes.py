"""Every solve route of the CUDA trainer against the oracle, away from the one point of the model's
inputs the parity suite holds fixed (nu = 1, max_cg_steps = 3, positive stored values, K <= 256).

* A route table names each route, how it is reached (K, solver, environment knobs) and how the
  test confirms that the trainer took it (plan_stats, or the number of kernels one half-step
  launches).
* Four hyper-parameter sets (nu = 0, 0.5, 2, 1; alpha0 = 0 included; both losses) run on every
  route, on counts, on counts with stored zeros and, where the route admits it, on counts with
  negative values.  Each case also shows that its answer depends on the parameter it is about:
  the f64 reference with that parameter perturbed must be more than ten tolerances away.
* CG step counts 1, 2, 5 and 0 (= K) with rows that exit at pass 0, K in (256, 512], the chunk
  boundaries of the tensor-core routes, step_io with several upload chunks, fold-in of long rows
  and the loss.

References: the oracle (f32 and f64) wherever it defines the answer.  For a negative stored value
under Cholesky or iALS++ the reference forms sqrt(c) y, which is NaN, and raises; the CUDA routes
form c y y^T instead, so those cases are compared with the numpy restatements in parity.py.
"""
import math

import numpy as np
import pytest
import scipy.sparse as sps

import oracle
from parity import (HSETS, assert_close, balanced_reg, dump_observed, hparams, make_data, make_pair,
                    np_cholesky_step, np_ialspp_step, observe, solver_cfg, transpose)

pytestmark = pytest.mark.gpu

TOL_STEP = 2e-4
SENSITIVITY = 10  # a perturbed parameter must move the f64 answer by more than this many tolerances


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


def ialspp_cfg(core, S, iters):
    return (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
            .set_ialspp_subspace_dimension(S).set_ialspp_iteration(iters).build())


# ---- references ----

def reference(solver, target, Xs, other, p, dtype, steps=3, S=64, iters=1, negative=False):
    """One half-epoch of ``solver`` on ``target`` (rows of Xs) from the same inputs, in ``dtype``:
    the oracle, or the numpy restatement where a negative value leaves the oracle undefined."""
    nt = oracle.hardware_threads()
    t = np.array(target, dtype=dtype)
    oth = np.ascontiguousarray(other, dtype=dtype)
    lt = oracle.LOSS_ORIGINAL if p["loss"] == "ORIGINAL" else oracle.LOSS_IALSPP
    if solver == "CG":
        oracle.step_cg(t, Xs, oth, oracle.gram(oth, p["alpha0"], nt), p["alpha0"], p["reg"], p["nu"], lt,
                       steps, nt)
    elif solver == "CHOLESKY" and negative:
        t = np_cholesky_step(t, Xs, oth, p["alpha0"], p["reg"], p["nu"], p["loss"])
    elif solver == "CHOLESKY":
        oracle.step_cholesky(t, Xs, oth, oracle.gram(oth, p["alpha0"], nt), p["alpha0"], p["reg"], p["nu"],
                             lt, nt)
    elif negative:
        t = np_ialspp_step(t, Xs, oth, p["alpha0"], p["reg"], p["nu"], p["loss"], S, iters)
    else:
        oracle.step_ialspp(t, Xs, oth, oracle.gram(oth, p["alpha0"], nt), p["alpha0"], p["reg"], p["nu"],
                           lt, S, iters, nt)
    return t


# ---- the route table ----

class Route:
    def __init__(self, name, K, solver, S=None, iters=None, env=None, negative="may", launches=None,
                 check=None, tensor=False, nnz=12000):
        self.name, self.K, self.solver, self.S, self.iters = name, K, solver, S, iters
        self.nnz = nnz  # of the test matrix: enough rows above IALS_HEAVY_THRESHOLD on the heavy route
        self.env = env or {}
        self.negative = negative  # "may" | "never" (the route needs positive values) | "must"
        self.launches = launches  # expected kernels of one half-step, or None
        self.check = check        # "light" | "heavy" | None
        self.tensor = tensor      # normal equations on the tensor cores: floor 1e-5 in assert_close

    def cfg(self, core, steps=3):
        if self.solver == "IALSPP":
            return ialspp_cfg(core, self.S, self.iters)
        return solver_cfg(core, self.solver, steps)

    def variants(self):
        return {"may": ["counts", "zeros", "neg"], "never": ["counts", "zeros"],
                "must": ["neg1", "zeros+neg1"]}[self.negative]


# Kernels launched by one half-step (ials_kernel_launch_count):
#   Gram P = alpha0 Y^T Y: 3 at row stride 128 (block_jobs_kernel + wgram_kernel +
#     wgram_reduce_sym_kernel, wgram.cu launch_gram_tc), 2 at other strides (gram_tile_kernel +
#     gram_finalize_kernel, gram.cu);
#   CG, stride 128: cg_rows_kernel for the light rows (1), wgram_kernel + dense_cg_kernel for the
#     heavy ones (2); other strides: cg_warp_kernel (1);
#   Cholesky, register-tiled: cholesky_tile_kernel (1); K = 256 on the tensor cores: per chunk of jobs
#     wgram256_kernel + cholesky_ll_kernel (2), one chunk here;
#   iALS++ on the tensor cores: per chunk wgram_kernel + ialspp_dense_kernel (2), one chunk here;
#   iALS++ per-block SIMT route: per sweep ialspp_predict_kernel + one cholesky_tile_kernel<SUB>
#     per block of S dimensions: iters * (1 + ceil(K / S)).
def _simt_ialspp(gram, K, S, iters):
    return gram + iters * (1 + math.ceil(K / S))


ROUTES = [
    Route("light_k128", 128, "CG", launches=3 + 1, check="light"),
    Route("light_k40", 40, "CG", launches=3 + 1, check="light"),
    Route("heavy_k128", 128, "CG", env={"IALS_HEAVY_THRESHOLD": "64"}, negative="never", check="heavy",
          tensor=True, nnz=30000),
    Route("warp_k160", 160, "CG", launches=2 + 1),
    Route("warp_k256", 256, "CG", launches=2 + 1),
    Route("warp_k300", 300, "CG", launches=2 + 1),
    Route("warp_k512", 512, "CG", launches=2 + 1),
    Route("tile_k64", 64, "CHOLESKY", launches=3 + 1),
    Route("tile_k136", 136, "CHOLESKY", launches=2 + 1),
    Route("tile_k256_neg", 256, "CHOLESKY", negative="must", launches=2 + 1),
    Route("tc_chol_k256", 256, "CHOLESKY", negative="never", launches=2 + 2, tensor=True),
    Route("tc_chol_k240", 240, "CHOLESKY", negative="never", launches=2 + 2, tensor=True),
    Route("ialspp_dense_s64", 128, "IALSPP", S=64, iters=2, negative="never", launches=3 + 2, tensor=True),
    Route("ialspp_dense_s48", 128, "IALSPP", S=48, iters=2, negative="never", launches=3 + 2, tensor=True),
    Route("ialspp_simt_k128_neg", 128, "IALSPP", S=64, iters=2, negative="must",
          launches=_simt_ialspp(3, 128, 64, 2)),
    Route("ialspp_simt_k160", 160, "IALSPP", S=64, iters=2, launches=_simt_ialspp(2, 160, 64, 2)),
    Route("ialspp_simt_k300", 300, "IALSPP", S=100, iters=2, launches=_simt_ialspp(2, 300, 100, 2)),
]
ROUTE = {r.name: r for r in ROUTES}


def confirm_route(route, g, delta):
    stats = [g.plan_stats(side) for side in (0, 1)]
    if route.check == "light":  # every row on cg_rows_kernel: none heavy, or a negative value
        assert all(s["heavy_rows"] == 0 or s["has_negative"] for s in stats), stats
    if route.check == "heavy":
        assert min(s["heavy_rows"] for s in stats) >= 50, stats
        assert not any(s["has_negative"] for s in stats)
        # Gram + wgram + dense CG, + cg_rows_kernel when light rows are left
        assert delta == 3 + 2 + (stats[0]["rows"] > stats[0]["heavy_rows"]), delta
    if route.launches is not None:
        assert delta == route.launches, (route.name, delta, route.launches)


def run_case(core, monkeypatch, route, variant, hset):
    for k, v in route.env.items():
        monkeypatch.setenv(k, v)  # plan_csr reads the knobs when the trainer is created
    long_rows = variant == "neg" and route.name == "light_k128"
    X = make_data(variant, long_rows=long_rows, nnz=route.nnz)
    negative = "neg" in variant
    p, perturb = hparams(hset, X, route.K)
    g, o32, o64 = make_pair(core, X, route.K, **p)
    assert g.plan_stats(0)["has_negative"] == int(negative)
    Xt = transpose(X)
    sc = route.cfg(core)
    kw = dict(S=route.S, iters=route.iters, negative=negative)
    floor = 1e-5 if route.tensor else 1e-6
    u0 = o32.user.copy()
    state32 = {"user": o32.user, "item": o32.item}
    state64 = {"user": o64.user, "item": o64.item}
    for side, (name, other, Xs) in enumerate((("user", "item", X), ("item", "user", Xt))):
        if side == 1:
            # the item half-epoch starts from the initial user factors: both sides then solve systems of
            # the same scale, on which the perturbed parameter still matters (the first half-epoch's
            # factors are ~100x larger and would leave the item side's ridge negligible)
            g.user = u0
            state32["user"], state64["user"] = u0, u0.astype(np.float64)
        before = launches()
        g.half_step(side, sc)
        delta = launches() - before
        if side == 0:
            confirm_route(route, g, delta)
        got = g.user if side == 0 else g.item
        want32 = reference(route.solver, state32[name], Xs, state32[other], p, np.float32, **kw)
        want64 = reference(route.solver, state64[name], Xs, state64[other], p, np.float64, **kw)
        assert_close(got, want32, want64, TOL_STEP, floor=floor)
        scale = np.abs(want32).max()
        for change in perturb:
            moved = reference(route.solver, state64[name], Xs, state64[other], {**p, **change}, np.float64, **kw)
            dist = np.abs(got - moved).max() / scale
            observe(sensitivity=dist, tol=TOL_STEP)
            assert dist > SENSITIVITY * TOL_STEP, (side, change, dist)
        state32[name], state64[name] = want32, want64


# H2's ridge is only as large as the data term: with a confidence of -0.25 the row's matrix is then
# indefinite and the solve raises (CG: singular system, Cholesky: decomposition failed), so H2 runs
# on the positive variants only
CASES = [pytest.param(r.name, v, h, id=f"{r.name}-{v}-{h}") for r in ROUTES for v in r.variants() for h in HSETS
         if not ("neg" in v and h == "H2")]


@pytest.mark.parametrize("route,variant,hset", CASES)
def test_route_hyper_parameters(core, monkeypatch, route, variant, hset):
    run_case(core, monkeypatch, ROUTE[route], variant, hset)


EMPTY_ROW_ROUTES = [r.name for r in ROUTES if r.solver != "CG"]


@pytest.mark.parametrize("route", EMPTY_ROW_ROUTES)
def test_empty_row_at_alpha0_zero_raises_like_the_reference(core, monkeypatch, route):
    """alpha0 = 0 leaves an empty row with A = 0 under Cholesky and iALS++ (reg_u = reg * 0^nu): the
    GPU raises exactly when the reference does, with its message."""
    r = ROUTE[route]
    for k, v in r.env.items():
        monkeypatch.setenv(k, v)
    variant = "neg1" if r.negative == "must" else "counts"
    X = sps.lil_matrix(make_data(variant))
    X[40, :] = 0
    X = sps.csr_matrix(X)
    X.eliminate_zeros()
    p = dict(nu=1.0, alpha0=0.0, reg=0.05, loss="ORIGINAL")
    g, o32, _ = make_pair(core, X, r.K, **p)
    with pytest.raises(RuntimeError) as want:
        reference(r.solver, o32.user, X, o32.item, p, np.float64, S=r.S, iters=r.iters,
                  negative=r.negative == "must")
    with pytest.raises(RuntimeError) as got:
        g.half_step(0, r.cfg(core))
    assert str(got.value) == str(want.value) == "Cholesky decomposition failed."


# ---- CG step counts and the exits of the CG kernels ----

@pytest.mark.parametrize("steps", [1, 2, 5, 0])
@pytest.mark.parametrize("route", ["light_k128", "heavy_k128", "warp_k160", "warp_k300"])
def test_cg_step_counts_and_early_exits(core, monkeypatch, route, steps):
    """max_cg_steps 1, 2, 5 and 0 (= K).  Rows made only of stored zeros have b = 0 under the IALSPP
    loss: with a zero warm start r = 0 and the row leaves at pass 0 (its partner warp in cg_rows_kernel
    keeps iterating); with a non-zero one it iterates.  The zero-start rows stay exactly zero."""
    r = ROUTE[route]
    for k, v in r.env.items():
        monkeypatch.setenv(k, v)
    X = make_data("counts", seed=4, nnz=r.nnz)
    deg = np.diff(X.indptr)
    by_degree = np.argsort(-deg, kind="stable")
    zero_rows = np.concatenate([by_degree[:4], by_degree[200:204], by_degree[-4:]])  # heavy, mid, short
    for u in zero_rows:
        X.data[X.indptr[u]:X.indptr[u + 1]] = 0.0
    # a ridge no larger than the data term: CG is far from converged after 5 steps, every step counts
    p = dict(nu=1.0, alpha0=0.1, reg=balanced_reg(X, r.K, 0.1, 1.0), loss="IALSPP")
    g, o32, o64 = make_pair(core, X, r.K, **p)
    if r.check == "heavy":
        assert g.plan_stats(0)["heavy_rows"] >= 50
    start0 = zero_rows[::2]  # every other zero row starts from zero
    u = g.user.copy()
    u[start0] = 0.0
    g.user = u
    o32.user[start0] = 0.0
    o64.user[start0] = 0.0
    sc = solver_cfg(core, "CG", steps)
    Xt = transpose(X)
    floor = 1e-5 if r.tensor else 1e-6
    g.half_step(0, sc)
    want32 = reference("CG", o32.user, X, o32.item, p, np.float32, steps=steps)
    want64 = reference("CG", o64.user, X, o64.item, p, np.float64, steps=steps)
    assert_close(g.user, want32, want64, TOL_STEP, floor=floor)
    assert not g.user[start0].any()
    assert np.abs(g.user[zero_rows[1::2]]).max() > 0
    if steps in (1, 2, 5):  # the step count matters: three steps are a different answer
        other = reference("CG", o64.user, X, o64.item, p, np.float64, steps=3)
        dist = np.abs(g.user - other).max() / np.abs(want32).max()
        observe(sensitivity=dist, tol=TOL_STEP)
        assert dist > SENSITIVITY * TOL_STEP, dist
    # the item half-epoch from the initial user factors, as in run_case: after the user half-epoch the
    # item systems are ill-conditioned and two float32 CG runs differ by percents, which says nothing
    g.user = u
    g.half_step(1, sc)
    w32 = reference("CG", o32.item, Xt, u, p, np.float32, steps=steps)
    w64 = reference("CG", o64.item, Xt, u, p, np.float64, steps=steps)
    assert_close(g.item, w32, w64, TOL_STEP, floor=floor)


# ---- K in (256, 512] ----

@pytest.mark.parametrize("K", [257, 288, 300, 333, 384, 416, 480, 512])
def test_wide_factors_cg_gram_scores_loss_fold_in(core, K):
    """Every row stride new_trainer produces above 256 has a CG kernel (cg_warp_kernel<ld / 32>):
    both half-epochs, the Gram, the scores, the loss and a CG fold-in against the oracle."""
    X = make_data("counts")
    p = dict(nu=1.0, alpha0=0.1, reg=0.02, loss="ORIGINAL")
    g, o32, o64 = make_pair(core, X, K, **p)
    sc = solver_cfg(core, "CG", 3)
    assert_close(g.gram(1), oracle.gram(o32.user, 0.1), oracle.gram(o64.user, 0.1), 1e-5)
    # fold-in against the initial item factors (after an epoch the factors are ~100x larger and five CG
    # steps leave the fold-in systems unconverged, so two float32 evaluations drift apart)
    Xnew = make_data("zeros", seed=9)[:60]
    got = g.transform_user(Xnew, solver_cfg(core, "CG", 5))
    assert_close(got, o32.transform_user(Xnew, oracle.SOLVER_CG, 5), o64.transform_user(Xnew, oracle.SOLVER_CG, 5),
                 TOL_STEP)
    g.half_step(0, sc)
    g.half_step(1, sc)
    for o in (o32, o64):
        o.step(oracle.SOLVER_CG, 3)
    assert_close(g.user, o32.user, o64.user, TOL_STEP)
    assert_close(g.item, o32.item, o64.item, TOL_STEP)
    user, item = g.user, g.item
    want = user[17:193].astype(np.float64) @ item.astype(np.float64).T
    np.testing.assert_allclose(g.user_scores(17, 193, sc), want, rtol=2e-5, atol=2e-5)
    o64.user, o64.item = user.astype(np.float64), item.astype(np.float64)
    o32.user, o32.item = user.copy(), item.copy()
    got, ref = g.compute_loss(sc), o64.compute_loss(oracle.hardware_threads())
    observe(loss_rel=abs(got - ref) / abs(ref), tol=1e-4)
    assert got == pytest.approx(ref, rel=1e-4)


@pytest.mark.parametrize("S", [64, 100])
def test_wide_factors_ialspp(core, S):
    X = make_data("counts")
    p = dict(nu=1.0, alpha0=0.1, reg=0.02, loss="ORIGINAL")
    g, o32, o64 = make_pair(core, X, 300, **p)
    sc = ialspp_cfg(core, S, 1)
    for o in (o32, o64):
        o.ialspp_subspace_dimension, o.ialspp_iteration = S, 1
    g.step(sc)
    for o in (o32, o64):
        o.step(oracle.SOLVER_IALSPP)
    assert_close(g.user, o32.user, o64.user, TOL_STEP)
    assert_close(g.item, o32.item, o64.item, TOL_STEP)


def test_wide_factors_limits(core):
    X = make_data("counts")
    g, _, _ = make_pair(core, X, 257)
    with pytest.raises(NotImplementedError, match="Cholesky solver: n_components > 256 not supported"):
        g.step(solver_cfg(core, "CHOLESKY"))
    with pytest.raises(ValueError, match=r"K must be in \[1, 512\]"):
        make_pair(core, X, 513)


# ---- chunk boundaries of the tensor-core routes ----

def jobs_of(degrees, job_len):
    """build_heavy_plan's cutting rule (csr.cu): a row of d > 0 neighbours is cut into
    ceil(d / per) jobs, per = round_up(ceil(d / pieces), 32), pieces = ceil(d / job_len)."""
    d = np.asarray(degrees, dtype=np.int64)
    d = d[d > 0]
    pieces = -(-d // job_len)
    per = -(-(-(-d // pieces)) // 32) * 32
    return int((-(-d // per)).sum())


def banded_matrix(n_users, n_items, lo, hi, seed):
    """Users of lo..hi neighbours (every degree present), counts 1..3."""
    rng = np.random.default_rng(seed)
    every = np.arange(lo, hi + 1)[:n_users]
    deg = np.concatenate([every, rng.integers(lo, hi + 1, n_users - every.size)])
    rng.shuffle(deg)
    keys = rng.random((n_users, n_items)).argsort(axis=1)
    rows = np.repeat(np.arange(n_users), deg)
    cols = np.concatenate([np.sort(keys[u, :d]) for u, d in enumerate(deg)])
    vals = rng.integers(1, 4, rows.size).astype(np.float32)
    return sps.csr_matrix((vals, (rows, cols)), shape=(n_users, n_items), dtype=np.float32)


def test_chunks_ialspp_tensor_route(core, monkeypatch):
    """iALS++ on the tensor cores works in chunks of <= 4096 Gram jobs (solve.cu): with jobs of 64
    entries, 2500 users of 65..190 neighbours need more than 4096; every row against the oracle."""
    monkeypatch.setenv("IALS_HEAVY_JOB_LEN", "64")
    X = banded_matrix(2500, 700, 65, 190, seed=31)
    Xt = transpose(X)
    assert jobs_of(np.diff(X.indptr), 64) > 4096
    p = dict(nu=1.0, alpha0=0.1, reg=0.02, loss="ORIGINAL")
    g, o32, o64 = make_pair(core, X, 128, **p)
    sc = ialspp_cfg(core, 64, 1)
    before = launches()
    g.half_step(0, sc)
    assert launches() - before >= 3 + 2 * 2  # Gram + at least two chunks of wgram + ialspp_dense
    w32 = reference("IALSPP", o32.user, X, o32.item, p, np.float32, S=64, iters=1)
    w64 = reference("IALSPP", o64.user, X, o64.item, p, np.float64, S=64, iters=1)
    assert_close(g.user, w32, w64, TOL_STEP, floor=1e-5)
    g.half_step(1, sc)
    assert_close(g.item, reference("IALSPP", o32.item, Xt, w32, p, np.float32, S=64, iters=1),
                 reference("IALSPP", o64.item, Xt, w64, p, np.float64, S=64, iters=1), TOL_STEP, floor=1e-5)


def test_chunks_cholesky_tensor_route(core, monkeypatch):
    """K = 256 Cholesky on the tensor cores works in chunks of <= 16384 Gram jobs (solve.cu): with jobs
    of 64 entries, 7000 users of 65..190 neighbours need more; every row against the oracle."""
    monkeypatch.setenv("IALS_HEAVY_JOB_LEN", "64")
    X = banded_matrix(7000, 1500, 65, 190, seed=32)
    Xt = transpose(X)
    assert jobs_of(np.diff(X.indptr), 64) > 16384
    p = dict(nu=1.0, alpha0=0.1, reg=0.02, loss="IALSPP")
    g, o32, o64 = make_pair(core, X, 256, **p)
    sc = solver_cfg(core, "CHOLESKY")
    before = launches()
    g.half_step(0, sc)
    assert launches() - before >= 2 + 2 * 2  # Gram + at least two chunks of wgram256 + cholesky_ll
    w32 = reference("CHOLESKY", o32.user, X, o32.item, p, np.float32)
    w64 = reference("CHOLESKY", o64.user, X, o64.item, p, np.float64)
    assert_close(g.user, w32, w64, TOL_STEP, floor=1e-5)
    g.half_step(1, sc)
    assert_close(g.item, reference("CHOLESKY", o32.item, Xt, w32, p, np.float32),
                 reference("CHOLESKY", o64.item, Xt, w64, p, np.float64), TOL_STEP, floor=1e-5)


# ---- step_io with several upload chunks ----

STEP_IO_CASES = {
    # name: (K, solver, environment, one negative value)
    "cg_k128_heavy": (128, "CG", {"IALS_HEAVY_THRESHOLD": "64"}, False),
    "cg_k128_heavy_negative": (128, "CG", {"IALS_HEAVY_THRESHOLD": "64"}, True),
    "cg_k64": (64, "CG", {}, False),
    "cholesky_k256": (256, "CHOLESKY", {}, False),
    "ialspp_k128": (128, "IALSPP", {}, False),
}


@pytest.mark.parametrize("case", list(STEP_IO_CASES))
def test_step_io_several_upload_chunks(core, monkeypatch, case):
    """9692 users: two full upload chunks of 4096 rows and a partial one.  CG at stride 128 solves while
    the chunks arrive (light rows in arrival order, heavy rows after them; none heavy when a value is
    negative); the other solvers upload first.  Two step_io, a step, a step_io: each equal to set +
    step + get on a twin trainer, bit for bit at row stride 128."""
    K, solver, env, negative = STEP_IO_CASES[case]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(5)
    U = 9692
    from irspack_b200.synth import synth_csr

    X = sps.lil_matrix(synth_csr(U, 400, 150000, seed=6, values="counts"))
    for u in range(0, U, 300):  # a long row in every chunk
        X.rows[u] = list(np.sort(rng.choice(400, 100, replace=False)))
        X.data[u] = [2.0] * 100
    X = sps.csr_matrix(X, dtype=np.float32)
    if negative:
        X.data[7] = -0.25
    sc = ialspp_cfg(core, 64, 1) if solver == "IALSPP" else solver_cfg(core, solver)
    g, _, _ = make_pair(core, X, K)
    h, _, _ = make_pair(core, X, K)
    stats = h.plan_stats(0)
    assert stats["has_negative"] == int(negative)
    if env:
        assert stats["heavy_rows"] >= U // 300
    # At row strides other than 128 the Gram P = alpha0 Y^T Y is the FP32 SIMT kernel, which adds its
    # per-CTA tiles with atomics (gram.cu): two trainers agree to rounding there, not bit for bit (one
    # ulp after the first epoch, 2.5e-5 of the scale after four on a B200), so the one-step tolerance
    if K == 128 or K == 64:
        same = np.testing.assert_array_equal
    else:
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
    same(h.user, g.user)


# ---- fold-in ----

def fold_in_rows(n_rows, n_cols, lo, hi, variant, seed):
    rng = np.random.default_rng(seed)
    X = banded_matrix(n_rows, n_cols, lo, hi, seed)
    if variant == "zeros":
        X.data[rng.random(X.nnz) < 0.05] = 0.0
        X.data[X.indptr[3]:X.indptr[4]] = 0.0
    if variant == "neg":
        X.data[rng.random(X.nnz) < 0.02] = -0.25
    return X


@pytest.mark.parametrize("variant", ["counts", "zeros", "neg"])
def test_fold_in_long_rows_cg(core, variant):
    """Fold-in rows of 2500..4500 neighbours take wgram_kernel + dense_cg_kernel from a zero start
    (all rows cg_rows_kernel when a value is negative)."""
    X = make_data("counts")
    X = sps.hstack([X, sps.csr_matrix((X.shape[0], 4700), dtype=np.float32)], format="csr")
    p = dict(nu=0.5, alpha0=0.1, reg=0.05, loss="ORIGINAL")
    g, o32, o64 = make_pair(core, X, 128, **p)
    g.step(solver_cfg(core))
    for o in (o32, o64):
        o.user, o.item = g.user.astype(o.dtype), g.item.astype(o.dtype)
    Xnew = fold_in_rows(24, X.shape[1], 2500, 4500, variant, seed=40)
    got = g.transform_user(Xnew, solver_cfg(core, "CG", 5))
    assert_close(got, o32.transform_user(Xnew, oracle.SOLVER_CG, 5), o64.transform_user(Xnew, oracle.SOLVER_CG, 5),
                 TOL_STEP, floor=1e-5)


@pytest.mark.parametrize("variant", ["counts", "zeros", "neg"])
@pytest.mark.parametrize("solver", ["CHOLESKY", "IALSPP"])
def test_fold_in_cholesky_and_ialspp(core, solver, variant):
    """transform_user / transform_item with Cholesky at K = 256 (register-tiled kernel: a fold-in matrix
    is not the trainer's own) and iALS++ at K = 128, S = 64, two sweeps (per-block SIMT route)."""
    K, S, iters = (256, None, None) if solver == "CHOLESKY" else (128, 64, 2)
    X = make_data("counts")
    p = dict(nu=2.0, alpha0=0.1, reg=1e-4, loss="ORIGINAL")
    g, o32, o64 = make_pair(core, X, K, **p)
    sc = solver_cfg(core, "CHOLESKY") if solver == "CHOLESKY" else ialspp_cfg(core, S, iters)
    negative = variant == "neg"
    for side in (0, 1):
        Xs = fold_in_rows(40, X.shape[1 - side], 5, 60, variant, seed=41 + side)  # the rows to fold in
        got = g.transform_user(Xs, sc) if side == 0 else g.transform_item(transpose(Xs), sc)
        other32 = o32.item if side == 0 else o32.user
        other64 = o64.item if side == 0 else o64.user
        zero = np.zeros((Xs.shape[0], K))
        want32 = reference(solver, zero, Xs, other32, p, np.float32, S=S, iters=iters, negative=negative)
        want64 = reference(solver, zero, Xs, other64, p, np.float64, S=S, iters=iters, negative=negative)
        assert_close(got, want32, want64, TOL_STEP)


# ---- loss ----

@pytest.mark.parametrize("variant", ["zeros", "neg"])
@pytest.mark.parametrize("K", [64, 256, 300])
@pytest.mark.parametrize("hset", list(HSETS))
def test_loss(core, hset, K, variant):
    """compute_loss against the f64 oracle within 1e-4 relative: the GPU sums each row's terms in
    float32 (as the reference does) and the rows in float64, so its distance to the f64 oracle is
    the float32 rounding of a row's dot products, far below 1e-4 (the observed margins are recorded)."""
    X = make_data(variant)
    p, _ = hparams(hset, X, K)
    g, _, o64 = make_pair(core, X, K, **p)
    sc = solver_cfg(core)
    got, ref = g.compute_loss(sc), o64.compute_loss(oracle.hardware_threads())
    observe(loss_rel=abs(got - ref) / abs(ref), tol=1e-4)
    assert got == pytest.approx(ref, rel=1e-4)
