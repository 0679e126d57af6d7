"""Explanations (``IALSTrainer.explain`` / ``explain_history``, ``ials_trainer_explain``) against a float64
numpy restatement of the contract on factors set through the setters.

For a query row u with history (j, c_j):  A_u = alpha0 Y^T Y + sum c_j y_j y_j^T + reg_u I,
x_u = A_u^-1 (sum (bias + c_j) y_j + reg_u prior_u),  w_t = A_u^-1 y_t;  per (u, t): score = y_t . x_u,
prior = reg_u w_t . prior_u and the contributions (bias + c_j) w_t . y_j, best first.

Tolerances are relative to the pair's float64 scale (|score| + |prior| + sum |contribution|); entries whose
contributions lie within that tolerance may come in either order."""
import numpy as np
import pytest
import scipy.sparse as sps

pytestmark = pytest.mark.gpu

TOL = 3e-3
HYPER = [dict(alpha0=0.1, reg=0.02, nu=1.0), dict(alpha0=0.1, reg=0.05, nu=0.5),
         dict(alpha0=0.1, reg=1e-4, nu=2.0), dict(alpha0=0.0, reg=0.05, nu=1.0)]


@pytest.fixture(scope="module")
def core():
    import irspack_b200

    if irspack_b200.device_count() == 0:
        pytest.fail("GPU test selected but no CUDA device is visible")
    from irspack_b200 import _ials_core

    return _ials_core


def launches(core):
    return int(core.lib.ials_kernel_launch_count())


def _matrix(rng, U, I, density, negative=True):
    """Counts 1..3, some stored zeros and (optionally) some small negative values."""
    M = sps.random(U, I, density=density, format="csr", random_state=rng, dtype=np.float32)
    v = rng.integers(1, 4, size=M.nnz).astype(np.float32)
    v[rng.random(M.nnz) < 0.1] = 0.0
    if negative:
        v[rng.random(M.nnz) < 0.05] = -0.1
    M.data = v
    return M


def _trainer(core, X, K, p, loss="ORIGINAL", seed=0):
    rng = np.random.default_rng(seed)
    U, I = X.shape
    b = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(p["alpha0"]).set_reg(p["reg"]).set_nu(p["nu"])
         .set_loss_type(getattr(core.LossType, loss)))
    tr = core.IALSTrainer(b.build(), X)
    scale = 0.3 / np.sqrt(K)
    tr.user = (rng.standard_normal((U, K)) * scale).astype(np.float32)
    tr.item = (rng.standard_normal((I, K)) * scale).astype(np.float32)
    return tr


def _without_rows(X, rows):
    """X with the given rows emptied (no stored entry left)."""
    L = sps.lil_matrix(X)
    for r in rows:
        L.rows[r], L.data[r] = [], []
    return sps.csr_matrix(L)


def _reference(Y, cols, vals, p, bias, targets, prior=None):
    """float64: (score [T], prior [T], contributions [T, len])."""
    Y = Y.astype(np.float64)
    K = Y.shape[1]
    cols = np.asarray(cols, dtype=np.int64)
    vals = np.asarray(vals, dtype=np.float64)
    T = len(targets)
    if cols.size == 0 and prior is None:
        return np.zeros(T), np.zeros(T), np.zeros((T, 0))
    reg_u = p["reg"] * (p["alpha0"] * Y.shape[0] + cols.size) ** p["nu"]
    Yh = Y[cols]
    A = p["alpha0"] * Y.T @ Y + (Yh * vals[:, None]).T @ Yh + reg_u * np.eye(K)
    b = ((bias + vals)[:, None] * Yh).sum(0)
    if prior is not None:
        b = b + reg_u * prior
    x = np.linalg.solve(A, b)
    Yt = Y[np.asarray(targets, dtype=np.int64)]
    W = np.linalg.solve(A, Yt.T)  # [K, T]
    pr = reg_u * (W.T @ prior) if prior is not None else np.zeros(T)
    return Yt @ x, pr, (Yh @ W).T * (bias + vals)[None, :]


def _check(e, r, pair, ref, cols, n_top):
    """Pair `pair` of Explanation `e` against the float64 reference (score, prior, contributions [len])."""
    score, prior, contrib = ref
    scale = abs(score) + abs(prior) + np.abs(contrib).sum() + 1e-6
    tol = TOL * scale
    assert abs(e.score[pair] - score) <= tol, (r, pair, e.score[pair], score)
    assert abs(e.prior[pair] - prior) <= tol, (r, pair, e.prior[pair], prior)
    n = min(n_top, contrib.size)
    assert e.counts[pair] == n
    assert np.all(e.indices[pair, n:] == -1) and np.all(e.contributions[pair, n:] == -np.inf)
    want = np.sort(contrib)[::-1][:n]
    got_c = e.contributions[pair, :n].astype(np.float64)
    assert np.all(np.abs(got_c - want) <= tol), (r, pair)
    assert np.all(np.diff(got_c) <= 0)
    cols = np.asarray(cols)
    for k in range(n):  # each returned id names an entry of the history with that contribution
        hits = contrib[cols == e.indices[pair, k]]
        assert hits.size and np.min(np.abs(hits - got_c[k])) <= tol, (r, pair, k)
    if n_top >= contrib.size:  # the contributions and the prior add up to the score
        assert abs(got_c.sum() + e.prior[pair] - e.score[pair]) <= tol


def _check_all(e, rows_hist, Y, p, bias, targets, n_top, priors=None):
    for r, (cols, vals) in enumerate(rows_hist):
        tl = targets[r]
        ref = _reference(Y, cols, vals, p, bias, tl, None if priors is None else priors[r])
        assert e.indptr[r + 1] - e.indptr[r] == len(tl)
        for q in range(len(tl)):
            _check(e, r, int(e.indptr[r]) + q, (ref[0][q], ref[1][q], ref[2][q]), cols, n_top)


def _hist(X, rows):
    X = sps.csr_matrix(X)
    return [(X.indices[X.indptr[r]:X.indptr[r + 1]], X.data[X.indptr[r]:X.indptr[r + 1]]) for r in rows]


@pytest.mark.parametrize("loss", ["ORIGINAL", "IALSPP"])
@pytest.mark.parametrize("K", [8, 16, 60, 128, 136, 200, 256])
def test_shapes_losses_and_hyper_parameters(core, K, loss):
    rng = np.random.default_rng(K)
    U, I = 40, 300
    X = _matrix(rng, U, I, 0.08)
    X = _without_rows(X, [3])
    for h, p in enumerate(HYPER):
        tr = _trainer(core, X, K, p, loss, seed=h)
        bias = p["alpha0"] if loss == "ORIGINAL" else 0.0
        q = np.array([5, 3, 0, 5, 17, 39])
        targets = [rng.integers(0, I, size=int(n)) for n in (4, 2, 1, 33, 0, 7)]
        for n_top in (1, 5, 1024):
            e = tr.explain(0, q, targets, n_top=n_top)
            _check_all(e, _hist(X, q), tr.item, p, bias, targets, n_top)
        empty = e.indptr[1]  # the empty row without a prior: nothing solved
        assert np.all(e.score[empty:empty + 2] == 0) and np.all(e.counts[empty:empty + 2] == 0)


@pytest.mark.parametrize("K", [128, 256])
def test_history_lengths(core, K):
    rng = np.random.default_rng(1)
    I = 5000
    lengths = [0, 1, 31, 32, 33, 256, 257, 4500, I]
    rows = [np.sort(rng.choice(I, n, replace=False)) for n in lengths]
    X = sps.csr_matrix((np.concatenate([rng.integers(1, 4, size=n) for n in lengths]).astype(np.float32),
                        np.concatenate(rows), np.concatenate([[0], np.cumsum(lengths)])), shape=(len(lengths), I))
    p = HYPER[0]
    tr = _trainer(core, X, K, p)
    targets = [rng.integers(0, I, size=3) for _ in lengths]
    for n_top in (5, 1024):
        e = tr.explain(0, range(len(lengths)), targets, n_top=n_top)
        _check_all(e, _hist(X, range(len(lengths))), tr.item, p, p["alpha0"], targets, n_top)


@pytest.mark.parametrize("side", [0, 1])
def test_query_forms(core, side):
    rng = np.random.default_rng(2 + side)
    U, I, K = 80, 120, 32
    X = _matrix(rng, U, I, 0.1)
    p = HYPER[0]
    tr = _trainer(core, X, K, p)
    Xs = X if side == 0 else sps.csr_matrix(X.T)
    Y = tr.item if side == 0 else tr.user
    n_side, n_other = Xs.shape
    q = rng.integers(0, n_side, size=20)
    q[5] = q[2]
    targets = [rng.integers(0, n_other, size=int(n)) for n in rng.integers(0, 6, size=q.size)]
    e = tr.explain(side, q, targets, n_top=7)
    _check_all(e, _hist(Xs, q), Y, p, p["alpha0"], targets, 7)
    # a range, with targets as (indptr, indices) arrays
    ip = np.arange(0, 2 * 10 + 1, 2, dtype=np.int64)
    ix = rng.integers(0, n_other, size=20)
    e2 = tr.explain(side, range(30, 40), (ip, ix), n_top=4)
    _check_all(e2, _hist(Xs, range(30, 40)), Y, p, p["alpha0"], [ix[a:a + 2] for a in ip[:-1]], 4)
    # cold rows: an unsorted row, a repeated column, a stored zero alone on its row, an empty row
    cold_rows = [([7, 3, 50, 1], [1.0, 2.0, 3.0, 1.0]), ([9, 9, 4], [1.0, 2.0, 1.0]), ([11], [0.0]), ([], [])]
    ip = np.concatenate([[0], np.cumsum([len(c) for c, _ in cold_rows])]).astype(np.int64)
    C = sps.csr_matrix((np.concatenate([v for _, v in cold_rows]).astype(np.float32),
                        np.concatenate([c for c, _ in cold_rows]).astype(np.int32), ip), shape=(4, n_other))
    assert C.indices[0] == 7  # kept as given
    ct = [[0, 1, 2], [5], [6, 6], [8]]
    e3 = tr.explain_history(side, C, ct, n_top=10)
    _check_all(e3, cold_rows, Y, p, p["alpha0"], ct, 10)
    assert e3.counts[e3.indptr[2]] == 1 and e3.counts[e3.indptr[3]] == 0
    # the cold score is the fold-in's: y_t . transform(row)
    chol = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CHOLESKY).build()
    row = sps.csr_matrix(C[0])
    emb = tr.transform_user(row, chol) if side == 0 else tr.transform_item(sps.csr_matrix(row.T), chol)
    want = Y[ct[0]].astype(np.float64) @ emb[0].astype(np.float64)
    assert np.allclose(e3.score[:3], want, rtol=0, atol=TOL * (np.abs(want).max() + 1e-6))


@pytest.mark.parametrize("K", [128, 256])
def test_score_is_the_solved_row_after_a_cholesky_half_step(core, K):
    rng = np.random.default_rng(K)
    U, I = 300, 700
    X = _matrix(rng, U, I, 0.05, negative=False)
    tr = _trainer(core, X, K, HYPER[0])
    tr.half_step(0, core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CHOLESKY).build())
    q = rng.integers(0, U, size=50)
    targets = [rng.integers(0, I, size=5) for _ in q]
    e = tr.explain(0, q, targets, n_top=3)
    user, item = tr.user.astype(np.float64), tr.item.astype(np.float64)
    for r, u in enumerate(q):
        want = item[targets[r]] @ user[u]
        got = e.score[e.indptr[r]:e.indptr[r + 1]]
        scale = np.abs(item[targets[r]]).sum(1) * np.abs(user[u]).max() + 1e-6
        assert np.all(np.abs(got - want) <= 1e-4 * scale), (K, r)


@pytest.mark.parametrize("warmup", [0, 1])
def test_feature_prior(core, warmup):
    rng = np.random.default_rng(5)
    U, I, K, nf = 60, 200, 16, 6
    X = _matrix(rng, U, I, 0.06, negative=False)
    X = _without_rows(X, [7])
    F = rng.standard_normal((U, nf)).astype(np.float32)
    p = HYPER[0]
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(p["alpha0"]).set_reg(p["reg"]).set_nu(p["nu"])
           .set_loss_type(core.LossType.ORIGINAL).set_lambda_user_feature(0.3).set_feature_warmup_epochs(warmup)
           .build())
    tr = core.IALSTrainer(cfg, X, F, np.zeros((I, 0), dtype=np.float32))
    tr.user = (rng.standard_normal((U, K)) * 0.1).astype(np.float32)
    tr.item = (rng.standard_normal((I, K)) * 0.1).astype(np.float32)
    W = (rng.standard_normal((nf, K)) * 0.1).astype(np.float32)
    tr.user_feature_weight = W
    q = np.array([7, 1, 2, 30])
    targets = [rng.integers(0, I, size=4) for _ in q]
    e = tr.explain(0, q, targets, n_top=1024)
    prior = F.astype(np.float64) @ W.astype(np.float64)
    priors = [prior[u] for u in q] if warmup == 0 else None
    _check_all(e, _hist(X, q), tr.item, p, p["alpha0"], targets, 1024, priors)
    if warmup:
        assert np.all(e.prior == 0)
    else:
        assert np.all(e.prior != 0)


def test_errors(core):
    rng = np.random.default_rng(9)
    U, I, K = 30, 50, 16
    X = _matrix(rng, U, I, 0.1)
    tr = _trainer(core, X, K, HYPER[0])
    with pytest.raises(ValueError):
        tr.explain(2, [0], [[0]])
    for bad in ([-1], [U]):
        with pytest.raises(ValueError):
            tr.explain(0, bad, [[0]])
    for bad in ([[-1]], [[I]]):
        with pytest.raises(ValueError):
            tr.explain(0, [0], bad)
    for n_top in (0, 1025):
        with pytest.raises(ValueError):
            tr.explain(0, [0], [[0]], n_top=n_top)
    with pytest.raises(ValueError):
        tr.explain_history(0, sps.csr_matrix((1, I + 1), dtype=np.float32), [[0]])
    # through the C ABI: what the wrappers cannot express
    from irspack_b200._ials_core import _ptr

    q = np.array([0], dtype=np.int64)
    ip = np.array([0, 1], dtype=np.int64)
    ix = np.array([0], dtype=np.int32)
    hd = np.array([1.0], dtype=np.float32)
    out_f = np.empty(1, np.float32)
    out_i = np.empty((1, 4), np.int32)
    out_c = np.empty((1, 4), np.float32)
    cnt = np.empty(1, np.int32)

    def call(qp, begin, end, hip, hix, hdp, tix=ix, n_top=4, side=0):
        return core.lib.ials_trainer_explain(tr._handle, side, qp, begin, end, hip, hix, hdp, _ptr(ip), _ptr(tix),
                                             n_top, _ptr(out_f), None, _ptr(out_i), _ptr(out_c), _ptr(cnt))

    bad_col = np.array([I], dtype=np.int32)
    for status in (call(_ptr(q), 0, 1, _ptr(ip), _ptr(ix), _ptr(hd)),  # both query forms
                   call(_ptr(q), 1, 2, None, None, None),  # begin != 0 with indices
                   call(None, 0, 1, _ptr(ip), _ptr(bad_col), _ptr(hd)),  # history column out of range
                   call(None, 0, 1, _ptr(ip), _ptr(ix), _ptr(hd), tix=bad_col),  # target out of range
                   call(_ptr(q), 0, 1, None, None, None, n_top=0),
                   call(_ptr(q), 0, 1, None, None, None, n_top=1025),
                   call(_ptr(q), 0, 1, None, None, None, side=-1),
                   call(None, U - 1, U + 1, None, None, None)):  # range past the side
        assert status == core._lib.IALS_ERR_INVALID_ARGUMENT
    # an indefinite system is a handled error, not a device fault
    ind = _trainer(core, X, K, dict(alpha0=0.0, reg=0.0, nu=1.0))
    with pytest.raises(RuntimeError, match="Cholesky decomposition failed."):
        ind.explain_history(0, sps.csr_matrix(([-1.0], [3], [0, 1]), shape=(1, I), dtype=np.float32), [[0]])
    e = ind.explain_history(0, sps.csr_matrix((1, I), dtype=np.float32), [[0]])
    assert e.score[0] == 0 and e.counts[0] == 0  # nothing solved, and the flag was cleared
    for K in (257, 300):
        wide = _trainer(core, X, K, HYPER[0])
        with pytest.raises(NotImplementedError):
            wide.explain(0, [0], [[0]])


def test_no_side_effects_slabs_and_launches(core):
    rng = np.random.default_rng(11)
    U, I, K = 50, 5000, 8
    X = _matrix(rng, U, I, 0.02, negative=False)
    X[0] = 1.0  # two rows whose history is the whole side
    X[1] = 2.0
    X = sps.csr_matrix(X)
    p = HYPER[0]
    tr = _trainer(core, X, K, p, seed=3)
    twin = _trainer(core, X, K, p, seed=3)
    u0, i0 = tr.user.copy(), tr.item.copy()
    # 2 rows x 4 000 targets x 5 000 entries: more contributions than one slab holds
    targets = [rng.integers(0, I, size=4000) for _ in range(2)]
    n0 = launches(core)
    e = tr.explain(0, [0, 1], targets, n_top=3)
    n_call = launches(core) - n0
    for r in range(2):
        ref = _reference(tr.item, *_hist(X, [r])[0], p, p["alpha0"], targets[r][:50])
        for q in range(50):
            _check(e, r, int(e.indptr[r]) + q, (ref[0][q], ref[1][q], ref[2][q]), _hist(X, [r])[0][0], 3)
        ref = _reference(tr.item, *_hist(X, [r])[0], p, p["alpha0"], targets[r][-50:])
        for q in range(50):
            _check(e, r, int(e.indptr[r + 1]) - 50 + q, (ref[0][q], ref[1][q], ref[2][q]), _hist(X, [r])[0][0], 3)
    n0 = launches(core)
    tr.gram(0)
    n_gram = launches(core) - n0
    assert n_call - n_gram == 2 * 2  # two slabs: the explain kernel and the top-k each
    # one slab: two launches besides the Gram, whatever the catalogue
    for n_items in (300, 5000):
        small = _trainer(core, sps.csr_matrix(X[:, :n_items]), K, p)
        n0 = launches(core)
        small.gram(0)
        n_gram = launches(core) - n0
        n0 = launches(core)
        small.explain(0, range(10), [[0, 1]] * 10)
        assert launches(core) - n0 - n_gram == 2, n_items
    assert np.array_equal(tr.user, u0) and np.array_equal(tr.item, i0)
    cfg = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CHOLESKY).build()
    tr.step(cfg)
    twin.step(cfg)
    assert np.array_equal(tr.user, twin.user) and np.array_equal(tr.item, twin.item)
