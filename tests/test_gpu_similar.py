"""Similar items and similar users (``IALSTrainer.similar``, ``ials_trainer_similar``) against float64
numpy on the same factors.

* Lists: identical to the float64 order (-score, index) except where two entries' float64 scores
  differ by less than 1e-5 of the row's largest |score| (the tie convention of the recommend tests);
  entries with exactly equal float64 scores must come in ascending index order.  Scores within 2e-5
  (relative to the row's largest |score|) of float64.
* Every row stride (K = 16 .. 512: strides 32 .. 512, both fused layouts), both metrics on both sides,
  cutoffs on the fused route (1, 10, 128) and on the SIMT route (150, 1024), confirmed by the number of
  kernels one call launches.
* Queries by index (repeats, any order), by range and over the whole side, one whole-side pass over
  more than one slab of 262 144 rows; self-exclusion on and off, zero rows, duplicate rows, forbidden
  lists, shared and per-query allow-lists, short lists; rejected arguments; no side effects.
Factors are set through the setters."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sps

pytestmark = pytest.mark.gpu

TIE = 1e-5
TOL_SCORE = 2e-5
SLAB = 262144  # kListSlabRows


@pytest.fixture(scope="module")
def core():
    import irspack_b200

    if irspack_b200.device_count() == 0:
        pytest.fail("GPU test selected but no CUDA device is visible")
    from irspack_b200 import _ials_core

    return _ials_core


def _factors(n, K, seed, zero_rows=(), duplicates=()):
    """A common direction plus noise (so that neighbours are not all near-ties), some rows zero and
    some rows exact copies of others."""
    rng = np.random.default_rng(seed)
    Y = (rng.standard_normal((n, 1)) * 0.2 + rng.standard_normal((n, K)) * 0.3).astype(np.float32)
    Y *= rng.uniform(0.2, 3.0, size=(n, 1)).astype(np.float32)  # norms differ: cosine != dot order
    for r in zero_rows:
        Y[r] = 0.0
    for dst, src in duplicates:
        Y[dst] = Y[src]
    return Y


def _trainer(core, U, I, K, seed=0, **kw):
    rng = np.random.default_rng(seed + 100)
    X = sps.csr_matrix((rng.random((U, I)) < 0.02).astype(np.float32))
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.05).build()
    tr = core.IALSTrainer(cfg, X)
    user, item = _factors(U, K, seed + 1, **kw.get("user", {})), _factors(I, K, seed + 2, **kw.get("item", {}))
    tr.user = user
    tr.item = item
    return tr, user, item


def _ref_scores(Y, q, metric):
    """float64 scores of the query rows q against every row of Y."""
    Y64 = Y.astype(np.float64)
    if metric == "cosine":
        nrm = np.linalg.norm(Y64, axis=1)
        Y64 = np.where(nrm[:, None] > 0, Y64 / np.where(nrm > 0, nrm, 1.0)[:, None], 0.0)
    return Y64[q] @ Y64.T


def _candidates(n, q, exclude_self, forbidden=None, allowed=None):
    """Boolean [len(q), n]: the rows each query may receive."""
    ok = np.ones((len(q), n), dtype=bool)
    if exclude_self:
        ok[np.arange(len(q)), q] = False
    if forbidden is not None:
        f = sps.csr_matrix(forbidden)
        f.eliminate_zeros()
        ok &= ~(f.toarray() != 0)
    if allowed is not None:
        n_lists, ip, ix = allowed
        a = np.zeros((len(q), n), dtype=bool)
        for r in range(len(q)):
            lst = 0 if n_lists == 1 else r
            a[r, ix[ip[lst]:ip[lst + 1]]] = True
        ok &= a
    return ok


def _check(S, ok, k, idx, cnt, sc):
    """The lists (idx, cnt, sc) of cutoff k against float64 scores S restricted to ok."""
    rows = S.shape[0]
    assert idx.shape == (rows, k) and cnt.shape == (rows,) and sc.shape == (rows, k)
    for r in range(rows):
        cand = np.flatnonzero(ok[r])
        s = S[r, cand]
        order = np.lexsort((cand, -s))  # (-score, index)
        ref, rs = cand[order], s[order]
        n_exp = min(k, cand.size)
        assert cnt[r] == n_exp, (r, cnt[r], n_exp)
        got = idx[r, :n_exp]
        assert np.all(idx[r, n_exp:] == -1), r
        assert np.all(ok[r, got]), r
        assert np.unique(got).size == n_exp, r
        scale = np.abs(s).max(initial=0.0) or 1.0
        tie = TIE * scale
        gs = S[r, got]
        assert np.abs(sc[r, :n_exp] - gs).max(initial=0.0) <= TOL_SCORE * scale, r
        assert np.abs(gs - rs[:n_exp]).max(initial=0.0) <= tie, r  # the same scores, position by position
        # ordered by (-score, index): exact float64 ties by index, near-ties in either order
        for p in range(n_exp - 1):
            assert gs[p] >= gs[p + 1] - tie, (r, p)
            if gs[p] == gs[p + 1]:
                assert got[p] < got[p + 1], (r, p)
        # an entry clear of its neighbours by more than the tie tolerance sits at its own position
        gap = np.full(rs.size + 1, np.inf)
        gap[1:-1] = rs[:-1] - rs[1:]
        clear = (gap[:-1] > tie) & (gap[1:] > tie)
        p = np.flatnonzero(clear[:n_exp])
        assert np.array_equal(got[p], ref[p]), r


def _launches(core):
    return int(core.lib.ials_kernel_launch_count())


@pytest.mark.parametrize("K", [16, 64, 100, 128, 200, 256, 512])
def test_row_strides_metrics_and_sides(core, K):
    U, I = 301, 413  # neither a multiple of 128
    tr, user, item = _trainer(core, U, I, K, seed=K)
    for side, Y in ((0, user), (1, item)):
        n = Y.shape[0]
        q = np.arange(n)
        for metric in ("cosine", "dot"):
            S = _ref_scores(Y, q, metric)
            ok = _candidates(n, q, True)
            for k in (10, 128):
                idx, cnt, sc = tr.similar(side, None, k, metric=metric)
                _check(S, ok, k, idx, cnt, sc)
            idx, cnt, sc = tr.similar(side, None, 150, metric=metric)
            _check(S, ok, 150, idx, cnt, sc)


@pytest.mark.parametrize("K", [64, 256])
def test_cutoffs_take_their_route(core, K):
    U, I = 1100, 1250
    tr, user, item = _trainer(core, U, I, K, seed=7)
    for side, Y in ((0, user), (1, item)):
        n = Y.shape[0]
        for metric in ("cosine", "dot"):
            q = np.arange(n)
            S = _ref_scores(Y, q, metric)
            ok = _candidates(n, q, True)
            for k in (1, 10, 128, 150, 1024):
                before = _launches(core)
                idx, cnt, sc = tr.similar(side, range(0, n), k, metric=metric)
                launched = _launches(core) - before
                # cosine: normalize_rows_kernel; the self mask of a range: self_mask_kernel; then
                # fused: score_tc_kernel + merge_topk_kernel, SIMT: score_tile + mask_rows + topk_rows
                expect = (metric == "cosine") + 1 + (2 if k <= 128 else 3)
                assert launched == expect, (side, metric, k, launched)
                _check(S, ok, k, idx, cnt, sc)


def test_query_forms(core):
    U, I = 200, 517
    tr, user, item = _trainer(core, U, I, 96, seed=3)
    rng = np.random.default_rng(5)
    for side, Y in ((0, user), (1, item)):
        n = Y.shape[0]
        for metric in ("cosine", "dot"):
            q = rng.integers(0, n, size=90)
            q[10] = q[3]
            q[11] = q[3]  # repeats
            for k in (10, 200):
                idx, cnt, sc = tr.similar(side, q, k, metric=metric)
                _check(_ref_scores(Y, q, metric), _candidates(n, q, True), k, idx, cnt, sc)
                assert np.array_equal(idx[10], idx[3]) and np.array_equal(sc[11], sc[3])
            b, e = 37, n - 21
            qr = np.arange(b, e)
            for k in (10, 200):
                idx, cnt, sc = tr.similar(side, range(b, e), k, metric=metric)
                _check(_ref_scores(Y, qr, metric), _candidates(n, qr, True), k, idx, cnt, sc)
                # the same rows by index: the same lists
                idx2, cnt2, sc2 = tr.similar(side, qr, k, metric=metric)
                assert np.array_equal(idx, idx2) and np.array_equal(cnt, cnt2) and np.array_equal(sc, sc2)
            idx, cnt = tr.similar(side, range(5, 5), 3, metric=metric, return_scores=False)
            assert idx.shape == (0, 3) and cnt.shape == (0,)


def test_whole_side_across_the_slab_boundary(core):
    I = SLAB + 1000
    tr, user, item = _trainer(core, 40, I, 32, seed=11)
    idx, cnt, sc = tr.similar(1, None, 10)
    assert idx.shape == (I, 10)
    rng = np.random.default_rng(2)
    q = np.concatenate([np.arange(SLAB - 4, SLAB + 4), [0, I - 1], rng.integers(0, I, size=12)])
    _check(_ref_scores(item, q, "cosine"), _candidates(I, q, True), 10, idx[q], cnt[q], sc[q])


def test_self_zero_rows_and_duplicates(core):
    U, I = 150, 300
    zeros, dups = (4, 9, 250), ((17, 5), (200, 5))
    tr, user, item = _trainer(core, U, I, 128, seed=13, item={"zero_rows": zeros, "duplicates": dups})
    q = np.array([5, 17, 4, 9, 100, 250, 200])
    for k in (10, 150):
        for excl in (True, False):
            for metric in ("cosine", "dot"):
                idx, cnt, sc = tr.similar(1, q, k, metric=metric, exclude_self=excl)
                _check(_ref_scores(item, q, metric), _candidates(I, q, excl), k, idx, cnt, sc)
        idx, cnt, sc = tr.similar(1, q, k, exclude_self=False)
        # duplicates: a tie at 1.0, broken by index; the query itself is one of them
        assert list(idx[0, :3]) == [5, 17, 200] and np.allclose(sc[0, :3], 1.0, atol=1e-6)
        assert list(idx[1, :3]) == [5, 17, 200]
        # a zero query: cosine 0 against every row, so the rows in ascending order
        assert np.array_equal(idx[2], np.arange(k)) and np.all(sc[2] == 0.0)
        idx, cnt, sc = tr.similar(1, q, k)
        assert list(idx[0, :2]) == [17, 200] and list(idx[1, :2]) == [5, 200]
        assert np.array_equal(idx[2], np.delete(np.arange(k + 1), 4))


def test_forbidden_allowed_and_short_lists(core):
    U, I = 120, 333
    tr, user, item = _trainer(core, U, I, 128, seed=17)
    rng = np.random.default_rng(9)
    q = rng.integers(0, I, size=40)
    S = {m: _ref_scores(item, q, m) for m in ("cosine", "dot")}
    forb = sps.random(40, I, density=0.05, random_state=1, format="csr", dtype=np.float32)
    forb.data[:] = 1.0
    forb[0, int(q[0])] = 1.0  # the query itself among its forbidden rows
    forb[1, 3] = 0.0  # a stored zero forbids nothing
    forb = sps.csr_matrix(forb)
    shared = np.unique(rng.choice(I, 60, replace=False)).astype(np.int32)
    per = [np.unique(rng.choice(I, 3 + r % 20, replace=False)).astype(np.int32) for r in range(40)]
    a_ip = np.concatenate([[0], np.cumsum([p.size for p in per])]).astype(np.int64)
    allowed = {"shared": (1, np.array([0, shared.size], dtype=np.int64), shared),
               "per": (40, a_ip, np.concatenate(per))}
    for metric in ("cosine", "dot"):
        for k in (10, 150):
            idx, cnt, sc = tr.similar(1, q, k, metric=metric, forbidden=forb)
            _check(S[metric], _candidates(I, q, True, forbidden=forb), k, idx, cnt, sc)
        for name, al in allowed.items():
            for excl in (True, False):
                idx, cnt, sc = tr.similar(1, q, 10, metric=metric, allowed=al, exclude_self=excl, forbidden=forb)
                ok = _candidates(I, q, excl, forbidden=forb, allowed=al)
                _check(S[metric], ok, 10, idx, cnt, sc)
            if name == "per":  # lists of 3 .. 22 rows: counts below the cutoff, padded with -1
                idx, cnt, sc = tr.similar(1, q, 128, metric=metric, allowed=al)
                assert np.all(cnt < 128) and np.all(idx[:, 100:] == -1)
                _check(S[metric], _candidates(I, q, True, allowed=al), 128, idx, cnt, sc)
            with pytest.raises(NotImplementedError):
                tr.similar(1, q, 150, metric=metric, allowed=al)
    # the whole side with forbidden lists (merged on the host) and a range without them: cutoff > candidates
    n = U
    f_all = sps.csr_matrix(np.ones((n, n), dtype=np.float32))
    idx, cnt, sc = tr.similar(0, None, 5, forbidden=f_all)
    assert np.all(cnt == 0) and np.all(idx == -1)


def test_rejected_arguments(core):
    tr, user, item = _trainer(core, 50, 80, 32, seed=19)
    bad = [
        dict(side=2), dict(side=-1), dict(metric="euclid"), dict(cutoff=0), dict(cutoff=81),
        dict(cutoff=1025), dict(indices=[0, 80]), dict(indices=[-1]), dict(indices=range(3, 81)),
        dict(indices=range(5, 2)), dict(indices=range(0, 10, 2)),
        dict(indices=[1, 2], forbidden=sps.csr_matrix((2, 79))),
        dict(indices=[1, 2], forbidden=sps.csr_matrix((3, 80))),
        dict(indices=[1, 2], allowed=(2, np.array([0, 1], np.int64), np.array([3], np.int32))),
        dict(indices=[1, 2, 3], allowed=(2, np.array([0, 1, 2], np.int64), np.array([3, 4], np.int32))),
        dict(indices=[1], allowed=(1, np.array([0, 2], np.int64), np.array([4, 3], np.int32))),
        dict(indices=[1], allowed=(1, np.array([0, 1], np.int64), np.array([80], np.int32))),
    ]
    for kw in bad:
        args = dict(side=1, indices=None, cutoff=10)
        args.update(kw)
        with pytest.raises(ValueError):
            tr.similar(args.pop("side"), args.pop("indices"), args.pop("cutoff"), **args)
    # the checks of the C ABI itself
    lib, p = core.lib, core._ptr
    idx = np.empty((2, 3), np.int32)
    cnt = np.empty(2, np.int32)
    fi, fx = np.array([0, 1, 2], np.int64), np.array([5, 80], np.int32)
    assert lib.ials_trainer_similar(tr._handle, 1, None, 0, 2, 3, 1, 1, p(fi), p(fx), 0, None, None, p(idx), None,
                                    p(cnt)) == core._lib.IALS_ERR_INVALID_ARGUMENT
    assert b"forbidden index out of range" in lib.ials_last_error()
    q = np.array([0, 1], np.int64)
    assert lib.ials_trainer_similar(tr._handle, 1, p(q), 1, 2, 3, 1, 1, None, None, 0, None, None, p(idx), None,
                                    p(cnt)) == core._lib.IALS_ERR_INVALID_ARGUMENT
    assert lib.ials_trainer_similar(tr._handle, 1, None, 0, 2, 3, 2, 1, None, None, 0, None, None, p(idx), None,
                                    p(cnt)) == core._lib.IALS_ERR_INVALID_ARGUMENT


def test_no_side_effects(core):
    U, I = 260, 390
    a, user, item = _trainer(core, U, I, 64, seed=23)
    b, _, _ = _trainer(core, U, I, 64, seed=23)
    sc = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CG).build()
    for side in (0, 1):
        for metric in ("cosine", "dot"):
            a.similar(side, None, 10, metric=metric)
            a.similar(side, np.array([3, 1, 3]), 150, metric=metric, forbidden=sps.csr_matrix(np.eye(3, U if side == 0 else I)))
    assert np.array_equal(a.user, b.user) and np.array_equal(a.item, b.item)
    assert np.array_equal(a.user, user) and np.array_equal(a.item, item)
    a.step(sc)
    b.step(sc)
    assert np.array_equal(a.user, b.user) and np.array_equal(a.item, b.item)


def test_recommender_and_id_mappers(core):
    from irspack_b200 import IALSRecommender
    from irspack_b200.id_mapping import IDMapper

    U, I = 90, 140
    rng = np.random.default_rng(29)
    X = sps.csr_matrix((rng.random((U, I)) < 0.1).astype(np.float32))
    rec = IALSRecommender(X, n_components=48, train_epochs=2).learn()
    core_tr = rec.trainer_as_ials.core_trainer
    user = core_tr.user
    # negative and boolean indices as get_score takes them
    mask = np.zeros(I, dtype=bool)
    mask[[3, 50, 139]] = True
    for got, q in ((rec.get_similar_items([-1, 3, -90], 7), [139, 3, 50]),
                   (rec.get_similar_items(mask, 7), [3, 50, 139])):
        ref = core_tr.similar(1, np.array(q), 7)
        for g, r in zip(got, ref):
            assert np.array_equal(g, r)
    idx, cnt, sc = rec.get_similar_users([0, -1], 5, metric="dot")
    _check(_ref_scores(user, np.array([0, U - 1]), "dot"), _candidates(U, np.array([0, U - 1]), True), 5, idx, cnt, sc)
    with pytest.raises(ValueError):
        rec.get_similar_items([I], 5)

    uids = [f"u{i}" for i in range(U)]
    iids = [f"i{i}" for i in range(I)]
    mapper = IDMapper(uids, iids)
    got = mapper.similar_items(rec, ["i3", "i7"], cutoff=4, forbidden_item_ids=[["i9", "zz"], []])
    f = sps.csr_matrix(([1.0], ([0], [9])), shape=(2, I))
    idx, cnt, sc = core_tr.similar(1, np.array([3, 7]), 4, forbidden=f)
    assert got == [[(iids[i], float(v)) for i, v in zip(idx[r, :cnt[r]], sc[r, :cnt[r]])] for r in range(2)]
    got = mapper.similar_items(rec, ["i3"], cutoff=20, allowed_item_ids=["i1", "i2", "i3", "i4", "nope"])
    assert sorted(x for x, _ in got[0]) == ["i1", "i2", "i4"]
    got = mapper.similar_users(rec, ["u5", "u0"], cutoff=3)
    idx, cnt, sc = core_tr.similar(0, np.array([5, 0]), 3)
    assert got == [[(uids[i], float(v)) for i, v in zip(idx[r, :cnt[r]], sc[r, :cnt[r]])] for r in range(2)]
