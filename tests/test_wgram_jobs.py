"""The tensor-core Gram (irspack_b200/csrc/wgram.cu: wgram_kernel for K <= 128, wgram256_kernel for
K <= 256) job by job, against float64 numpy.

The solvers add up the blocks of a row's jobs themselves (dense_cg, ialspp_dense, cholesky_ll), so
every job's block is checked on its own here (``ops.weighted_gram_jobs``), on explicit job plans:
empty, overlapping and out-of-order jobs, plans cut like build_heavy_plan, more jobs than SMs (a CTA
runs job j, j + grid, ...: its second accumulator buffer, the hand-back between jobs, the flush of
b partials across jobs).

Exact cases: Y integer in [-2, 2], w in {0, 1/4, 1, 4} (sqrt(w) exact), bias 1/2, jobs of at most
1024 entries (y in {-1, 0, 1} and w in {0, 1} in longer ones).  Then u = sqrt(w) y is a power of two
or zero, the TF32 hi/lo split has lo = 0, and every partial sum is a multiple of 1/4 below 2^14: the
blocks equal the float64 result bit for bit.  Float cases: the bound of test_wgram.py with L the
job's own length.  Trainer-level: the K1 Gram exactly on integer factors, the job plan against its
numpy restatement, and rows made of up to 250 jobs through the three routes that use these
kernels."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sps

import oracle
from parity import assert_close, dump_observed, observe

pytestmark = pytest.mark.gpu

TOL_STEP = 2e-4
LENGTHS = [0, 1, 7, 8, 9, 31, 32, 33, 0, 63, 64, 65, 127, 128, 129, 4095, 4096, 4097, 0]
KS = [5, 20, 48, 100, 128, 136, 240, 256]


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
    dump_observed()  # $IALS_PARITY_OBSERVED_DIR, else the directory of an earlier module's dump


def gram_jobs(Y, jb, je, idx=None, w=None, bias=0.0):
    from irspack_b200.ops import weighted_gram_jobs

    return weighted_gram_jobs(Y, np.asarray(jb), np.asarray(je), idx, w, bias)


def ref_job(Y64, idx, w, b, e, bias):
    rows = Y64[b:e] if idx is None else Y64[idx[b:e]]
    ww = np.ones(e - b) if w is None else w[b:e].astype(np.float64)
    return (rows * ww[:, None]).T @ rows, ((bias + ww)[:, None] * rows).sum(axis=0)


def assert_jobs_exact(G, b, Y, idx, w, jb, je, bias):
    """Every job's G and b equal the float64 result bit for bit."""
    Y64 = Y.astype(np.float64)
    err = 0.0
    for j, (lo, hi) in enumerate(zip(jb, je)):
        G64, b64 = ref_job(Y64, idx, w, lo, hi, bias)
        e = max(np.abs(G[j] - G64).max(), np.abs(b[j] - b64).max())
        assert e == 0, f"job {j} [{lo}, {hi}): max error {e:.3e}"
        err = max(err, e)
    observe(max_abs_err=err, jobs=len(jb))


def tol(L, wide):
    t = 6e-8 * L / 8
    return 2e-6 + (2 * t if wide else t)


def assert_jobs_within_bound(G, b, Y, idx, w, jb, je, bias):
    """The stated bound of test_wgram.py per job, L = the job's length; returns the worst ratio."""
    Y64 = Y.astype(np.float64)
    wide = Y.shape[1] > 128
    worst = 0.0
    for j, (lo, hi) in enumerate(zip(jb, je)):
        G64, b64 = ref_job(Y64, idx, w, lo, hi, bias)
        if hi == lo:
            assert not G[j].any() and not b[j].any(), j
            continue
        scale = max(np.abs(G64).max(), 1e-300)
        bound = tol(hi - lo, wide) * scale
        e = np.abs(G[j] - G64).max()
        assert e <= bound, f"job {j} (L = {hi - lo}): {e / scale:.3e} > {bound / scale:.3e}"
        rows = Y64[idx[lo:hi]]
        bscale = max((np.abs(rows) * (bias + w[lo:hi].astype(np.float64))[:, None]).sum(axis=0).max(), 1e-300)
        assert np.abs(b[j] - b64).max() <= 1e-5 * bscale, j
        np.testing.assert_array_equal(G[j], G[j].T)
        worst = max(worst, e / bound)
    observe(worst_err_over_bound=worst, jobs=len(jb))
    return worst


# ---- exact inputs ----

def int_factors(rng, n, K):
    """Rows [0, n/2): integers in [-2, 2]; rows [n/2, n): {-1, 0, 1} (for jobs longer than 1024);
    three all-zero rows, none of them the last."""
    Y = rng.integers(-2, 3, (n, K)).astype(np.float32)
    Y[n // 2:] = rng.integers(-1, 2, (n - n // 2, K))
    Y[rng.choice(n - 1, 3, replace=False)] = 0
    Y[n - 1, 0] = 1  # the last row is used (below) and is not zero
    return Y


def int_entries(rng, n, lengths):
    """Contiguous jobs of the given lengths laid out in a shuffled order; entries of jobs longer than
    1024 gather the {-1, 0, 1} rows with weights in {0, 1}."""
    m = int(sum(lengths))
    pos = np.zeros(len(lengths), np.int64)
    perm = rng.permutation(len(lengths))
    pos[perm] = np.concatenate([[0], np.cumsum(np.asarray(lengths)[perm])[:-1]])
    idx = rng.integers(0, n, m).astype(np.int32)
    w = rng.choice(np.float32([0, 0.25, 1, 4]), m)
    for p, L in zip(pos, lengths):
        if L > 1024:
            idx[p:p + L] = rng.integers(n // 2, n, L)
            w[p:p + L] = rng.choice(np.float32([0, 1]), L)
    return idx, w, pos, pos + np.asarray(lengths, np.int64)


@pytest.mark.parametrize("K", KS)
def test_exact_job_lengths(core, K):
    """Jobs of 0 .. 4097 entries around the 8-neighbour MMA step and the 32-neighbour stage, empty
    jobs first, in the middle and last, a job of one repeated index, a job that overlaps two others,
    a repeated job, and empty jobs at both ends of the entries."""
    rng = np.random.default_rng(K)
    n = 600
    Y = int_factors(rng, n, K)
    idx, w, jb, je = int_entries(rng, n, LENGTHS)
    m = idx.shape[0]
    k65 = LENGTHS.index(65)
    idx[jb[k65]:je[k65]] = 17  # one row 65 times
    k129 = LENGTHS.index(129)
    idx[je[k129] - 1] = n - 1
    k64 = LENGTHS.index(64)
    extra_b = [jb[k64] + 3, jb[k129], 0, m, max(jb[k65] - 40, 0)]
    extra_e = [min(jb[k64] + 200, m), je[k129], 0, m, jb[k65] + 40]
    jb = np.concatenate([jb, extra_b])
    je = np.concatenate([je, extra_e])
    G, b = gram_jobs(Y, jb, je, idx, w, bias=0.5)
    assert_jobs_exact(G, b, Y, idx, w, jb, je, 0.5)


@pytest.mark.parametrize("K", [20, 256])
def test_exact_all_jobs_empty(core, K):
    rng = np.random.default_rng(1)
    Y = int_factors(rng, 50, K)
    idx = rng.integers(0, 50, 100).astype(np.int32)
    jb = je = np.array([0, 7, 100, 7, 0])
    G, b = gram_jobs(Y, jb, je, idx, None, bias=0.5)
    assert not G.any() and not b.any()


@pytest.mark.parametrize("n_jobs,K", [(149, 128), (296, 48), (1000, 100), (4096, 128), (149, 256), (1024, 240)])
def test_exact_more_jobs_than_sms(core, n_jobs, K):
    """n_jobs > 148: a CTA runs several jobs (job j on CTA j mod 148), and with lengths mixed (about
    a fifth of the jobs empty) the CTAs run different numbers of them; the jobs come in shuffled
    order over the entries."""
    rng = np.random.default_rng(n_jobs + K)
    n = 2000
    Y = int_factors(rng, n, K)
    lengths = rng.choice([0, 0, 1, 8, 31, 32, 33, 64, 65, 129, 300], n_jobs)
    idx, w, jb, je = int_entries(rng, n, lengths)
    G, b = gram_jobs(Y, jb, je, idx, w, bias=0.5)
    assert_jobs_exact(G, b, Y, idx, w, jb, je, 0.5)


def plan_jobs(indptr, threshold, job_len):
    """build_heavy_plan (csr.cu) restated: the rows with more than `threshold` entries by descending
    degree, each cut into jobs of per = round_up(ceil(d / ceil(d / job_len)), 32) entries (whole
    32-entry pipeline stages).  Returns (job_begin, job_end, first job of each heavy row)."""
    deg = np.diff(indptr)
    jb, je, first = [], [], [0]
    for u in np.argsort(-deg, kind="stable"):
        b, e = int(indptr[u]), int(indptr[u + 1])
        d = e - b
        if d <= threshold:
            break
        pieces = -(-d // job_len)
        per = -(-(-(-d // pieces)) // 32) * 32
        for p in range(b, e, per):
            jb.append(p)
            je.append(min(p + per, e))
        first.append(len(jb))
    return np.array(jb, np.int64), np.array(je, np.int64), first


def degree_csr(rng, degrees, n_cols, values=(1.0,)):
    rows = np.repeat(np.arange(len(degrees)), degrees)
    cols = np.concatenate([np.sort(rng.choice(n_cols, d, replace=False)) for d in degrees])
    vals = rng.choice(np.float32(values), rows.shape[0])
    X = sps.csr_matrix((vals, (rows, cols)), shape=(len(degrees), n_cols), dtype=np.float32)
    X.sort_indices()
    return X


@pytest.mark.parametrize("job_len", [32, 33, 96, 100, 1000, 4096])
@pytest.mark.parametrize("K", [128, 256])
def test_exact_heavy_plan_jobs(core, job_len, K):
    """Jobs cut exactly like the trainer's (threshold 0: every row with entries), job lengths that
    are and are not multiples of 32; every job exact, so every row's sum of jobs is too."""
    rng = np.random.default_rng(job_len)
    degrees = [0, 1, 31, 32, 33, 64, 65, 97, 1000, 1023, 2049, 4097, 5000, 3, 0]
    X = degree_csr(rng, degrees, 6000, values=(0.0, 1.0))
    Y = rng.integers(-1, 2, (6000, K)).astype(np.float32)
    jb, je, _ = plan_jobs(X.indptr, 0, job_len)
    G, b = gram_jobs(Y, jb, je, X.indices, X.data, bias=0.5)
    assert_jobs_exact(G, b, Y, X.indices, X.data, jb, je, 0.5)


# ---- float inputs ----

def tf32_boundary_values(rng, shape):
    """Floats whose 13 bits below the TF32 mantissa sit at or next to a rounding boundary (0x0000,
    0x0001, 0x0fff, 0x1000, 0x1001, 0x1fff): the lo part is 0, 1 ulp, or close to half a TF32 ulp."""
    base = rng.uniform(0.5, 2.0, shape).astype(np.float32) * rng.choice(np.float32([-1, 1]), shape)
    low = rng.choice(np.uint32([0x0000, 0x0001, 0x0FFF, 0x1000, 0x1001, 0x1FFF]), shape)
    return ((base.view(np.uint32) & np.uint32(0xFFFFE000)) | low).view(np.float32)


FLOAT_CASES = ["normal", "scaled_rows", "heavy_weights", "tf32_boundary"]


@pytest.mark.parametrize("case", FLOAT_CASES)
@pytest.mark.parametrize("K", [20, 128, 136, 256])
def test_float_jobs_within_bound(core, case, K):
    """Random floats per job within the stated bound.  scaled_rows: each job gathers rows scaled by
    2^20, 1 or 2^-20; heavy_weights: confidences up to 1e4; tf32_boundary: the lo part is as large as
    it gets (dropping a cross term is ~2^-11 off)."""
    rng = np.random.default_rng(K + 7 * FLOAT_CASES.index(case))
    n = 900
    lengths = [1, 8, 33, 0, 64, 200, 1024, 1500, 129, 0, 4097, 31]
    m = int(sum(lengths))
    jb = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    je = jb + np.asarray(lengths, np.int64)
    Y = (rng.standard_normal((n, K)) * rng.uniform(0.01, 3.0, size=(1, K))).astype(np.float32)
    idx = rng.integers(0, n, m).astype(np.int32)
    w = rng.choice(np.float32([0.0, 0.5, 1.0, 2.0, 4.7]), m)
    if case == "scaled_rows":
        Y[:300] *= np.float32(2.0 ** 20)
        Y[600:] *= np.float32(2.0 ** -20)
        for j, (lo, hi) in enumerate(zip(jb, je)):
            idx[lo:hi] = rng.integers(300 * (j % 3), 300 * (j % 3 + 1), hi - lo)
    elif case == "heavy_weights":
        w = rng.uniform(0.0, 1e4, m).astype(np.float32)
    elif case == "tf32_boundary":
        Y = tf32_boundary_values(rng, (n, K))
        w = rng.choice(np.float32([1.0, 4.0]), m)
    G, b = gram_jobs(Y, jb, je, idx, w, bias=0.1)
    assert_jobs_within_bound(G, b, Y, idx, w, jb, je, 0.1)


@pytest.mark.parametrize("K,m,jobs", [(128, 5000, 7), (48, 333, 4), (128, 40000, 300), (256, 5000, 3), (240, 1000, 2)])
def test_even_split_operators_are_the_sum_of_their_jobs(core, K, m, jobs):
    """ials_weighted_gram(256) = the sum of the per-job blocks of their even split: bit for bit for
    the 128-column operator (its device reduction adds W_j + W_j^T in job order in float32), to
    rounding for the 256-column one and for b (float64 sums of the same partials)."""
    from irspack_b200.ops import weighted_gram, weighted_gram256

    rng = np.random.default_rng(m + K)
    n = 700
    Y = (rng.standard_normal((n, K)) * 0.3).astype(np.float32)
    idx = rng.integers(0, n, m).astype(np.int32)
    w = rng.choice(np.float32([0.0, 0.5, 1.0, 4.7]), m)
    per = -(-m // jobs)
    jb = np.minimum(np.arange(jobs) * per, m)
    je = np.minimum(jb + per, m)
    Gj, bj = gram_jobs(Y, jb, je, idx, w, bias=0.1)
    if K <= 128:
        G, b = weighted_gram(Y, idx, w, n_jobs=jobs, bias=0.1)
        acc = np.zeros((K, K), np.float32)
        for g in Gj:
            acc = acc + g
        np.testing.assert_array_equal(G, acc)
    else:
        G, b = weighted_gram256(Y, idx, w, n_jobs=jobs, bias=0.1)
        S = Gj.astype(np.float64).sum(axis=0)
        assert np.abs(G - S).max() <= 2 ** -22 * np.abs(S).max()
    bscale = (np.abs(Y[idx]).astype(np.float64) * (0.1 + w)[:, None]).sum(axis=0).max()
    assert np.abs(b - bj.astype(np.float64).sum(axis=0)).max() <= 1e-5 * bscale


def test_job_bounds_rejected(core):
    Y = np.ones((4, 8), np.float32)
    idx = np.array([0, 1, 2], np.int32)
    for jb, je in (([0], [4]), ([-1], [2]), ([2], [1])):
        with pytest.raises(ValueError, match="job bounds"):
            gram_jobs(Y, jb, je, idx)
    with pytest.raises(ValueError, match="n_jobs"):
        gram_jobs(np.ones((4, 200), np.float32), np.zeros(1025), np.zeros(1025), idx)


# ---- the trainer ----

def make_trainer(core, X, K, alpha0=0.125, reg=0.05, loss="IALSPP"):
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(alpha0).set_reg(reg).set_nu(1.0)
           .set_init_stdev(0.0).set_loss_type(getattr(core.LossType, loss)).build())
    return core.IALSTrainer(cfg, X)


@pytest.mark.parametrize("n,K", [(1, 128), (31, 128), (32, 128), (33, 100), (255, 128), (256, 128), (257, 20),
                                 (148 * 256 - 1, 128), (148 * 256 + 1, 128), (1_000_003, 64),
                                 (1000, 160), (5000, 240), (777, 512)])
def test_k1_gram_exact_on_integer_factors(core, n, K):
    """P = alpha0 Y^T Y with alpha0 = 1/8 and integer factors: bit for bit.  Row stride 128 takes the
    tensor cores (block_jobs_kernel: one job of >= 8 stages per 256 rows, at most 148, cut at whole
    32-row stages); strides 160, 256 and 512 take the SIMT Gram (gram.cu)."""
    rng = np.random.default_rng(n)
    X = sps.csr_matrix((np.ones(1, np.float32), ([0], [0])), shape=(n, 3))
    g = make_trainer(core, X, K)
    Y = rng.integers(-2, 3, (n, K)).astype(np.float32)
    g.user = Y
    Y64 = Y.astype(np.float64)
    P64 = 0.125 * (Y64.T @ Y64)
    P = g.gram(1)
    err = np.abs(P - P64).max()
    observe(max_abs_err=err, rows=n, K=K)
    assert err == 0, err


# degrees of the user rows of the plan test: around the thresholds and the job lengths
PLAN_DEGREES = [0, 1, 2, 31, 32, 33, 64, 65, 96, 97, 2048, 2049, 4096, 4097, 5000, 40, 0, 1]


@pytest.mark.parametrize("threshold", ["0", "1", "64", "2048"])
@pytest.mark.parametrize("job_len", ["1", "32", "33", "96", "4096", "1000000"])
def test_plan_stats_match_the_plan_restated(core, monkeypatch, threshold, job_len):
    monkeypatch.setenv("IALS_HEAVY_THRESHOLD", threshold)
    monkeypatch.setenv("IALS_HEAVY_JOB_LEN", job_len)
    rng = np.random.default_rng(5)
    X = degree_csr(rng, PLAN_DEGREES, 6000)
    g = make_trainer(core, X, 64)
    for side, M in ((0, X), (1, sps.csr_matrix(X.T))):
        jb, _, first = plan_jobs(M.indptr, max(int(threshold), 1), int(job_len))
        st = g.plan_stats(side)
        assert (st["heavy_rows"], st["jobs"]) == (len(first) - 1, len(jb)), (side, st)


@pytest.mark.parametrize("value", ["0", "-5", "abc"])
def test_heavy_job_len_must_be_a_positive_integer(core, monkeypatch, value):
    monkeypatch.setenv("IALS_HEAVY_JOB_LEN", value)
    X = sps.csr_matrix(np.eye(4, dtype=np.float32))
    with pytest.raises(ValueError, match="IALS_HEAVY_JOB_LEN"):
        make_trainer(core, X, 8)


def test_trainer_rejects_nnz_past_the_gram_cap(core):
    """An indptr that claims 2^31 - 63 entries is rejected before its indices are read."""
    from irspack_b200._lib import IALS_ERR_INVALID_ARGUMENT, ModelConfigStruct, lib

    cfg = ModelConfigStruct(K=8, alpha0=0.1, reg=0.1, nu=1.0, init_stdev=0.0, random_seed=0, loss_type=0)
    indptr = (ctypes.c_int64 * 2)(0, 2 ** 31 - 63)
    indices, data = (ctypes.c_int32 * 1)(0), (ctypes.c_float * 1)(1.0)
    h = ctypes.c_void_p()
    P = ctypes.c_void_p
    st = lib.ials_trainer_create(ctypes.byref(cfg), 1, 5, ctypes.cast(indptr, P), ctypes.cast(indices, P),
                                 ctypes.cast(data, P), 0, ctypes.byref(h))
    assert st == IALS_ERR_INVALID_ARGUMENT and "2^31 - 64" in lib.ials_last_error().decode()


# ---- rows made of many jobs ----

@pytest.fixture(scope="module")
def X_many_jobs():
    """40 users x 9000 items: 27 users with 3000 .. 8000 neighbours (94 .. 250 jobs of 32 each, 4500
    jobs together: more than one 4096-job chunk of the iALS++ route), 12 short rows, one empty."""
    rng = np.random.default_rng(21)
    degrees = list(np.linspace(3000, 8000, 27).astype(int)) + list(rng.integers(1, 100, 12)) + [0]
    X = degree_csr(rng, degrees, 9000)
    X.data = rng.integers(1, 4, X.nnz).astype(np.float32)
    return X


def make_oracle_pair(core, X, K, **kw):
    from irspack_b200.synth import init_factors

    g = make_trainer(core, X, K, alpha0=0.1, reg=0.02, loss="ORIGINAL")
    u0, i0 = init_factors(X.shape[0], K, 1), init_factors(X.shape[1], K, 2)
    g.user, g.item = u0, i0
    os_ = [oracle.OracleTrainer(X, K, 0.1, 0.02, 1.0, oracle.LOSS_ORIGINAL, dtype=dt) for dt in (np.float32, np.float64)]
    for o in os_:
        o.user, o.item = u0.astype(o.dtype), i0.astype(o.dtype)
    return g, os_


@pytest.mark.parametrize("route", ["heavy_cg", "ialspp_tensor", "cholesky256_tensor"])
def test_rows_of_many_jobs(core, monkeypatch, X_many_jobs, route):
    """IALS_HEAVY_JOB_LEN = 32: user rows of up to 250 Gram jobs, summed by the solver of each route
    (dense_cg, ialspp_dense, cholesky_ll); the user half-epoch against the oracle."""
    monkeypatch.setenv("IALS_HEAVY_JOB_LEN", "32")
    X = X_many_jobs
    jb, _, first = plan_jobs(X.indptr, 0, 32)
    assert len(jb) > 4096 and 4096 not in first  # two iALS++ chunks; a row moves past the boundary
    nt = oracle.hardware_threads()
    if route == "heavy_cg":
        monkeypatch.setenv("IALS_HEAVY_THRESHOLD", "64")
        g, os_ = make_oracle_pair(core, X, 128)
        assert g.plan_stats(0)["jobs"] == len(plan_jobs(X.indptr, 64, 32)[0])
        sc = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CG).set_max_cg_steps(3).build())
        solver = oracle.SOLVER_CG
    elif route == "ialspp_tensor":
        g, os_ = make_oracle_pair(core, X, 128)
        sc = (core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP)
              .set_ialspp_subspace_dimension(64).set_ialspp_iteration(1).build())
        for o in os_:
            o.ialspp_subspace_dimension, o.ialspp_iteration = 64, 1
        solver = oracle.SOLVER_IALSPP
    else:
        g, os_ = make_oracle_pair(core, X, 256)
        sc = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CHOLESKY).build()
        solver = oracle.SOLVER_CHOLESKY
    g.half_step(0, sc)
    for o in os_:
        o._solve(o.user, o.X, o.item, solver, 3, nt)
    assert_close(g.user, os_[0].user, os_[1].user, TOL_STEP, floor=1e-5)
