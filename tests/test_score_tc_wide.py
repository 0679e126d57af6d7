"""The fused tcgen05 score + mask + top-k kernel at row strides above 128 (160 .. 512): the variant
of ``score_tc_kernel`` that streams the user tile through the stages instead of parking it.

Against the CPU oracle (float64 scores + the reference's (-score, index) order,
evaluator.cpp:324-355), with the tolerances of test_score_tc.py: lists identical except that two
items whose float64 scores differ by less than 1e-5 * max|score| may swap, returned scores within
rtol = atol = 2e-5; on small-integer factors (every product and sum exact in any order) the lists
are IDENTICAL, ties included.  Also: the calls that need the fused kernel (allow-lists, users by
index with their training rows as the mask) at these strides, the route each call takes, and the
host layer (Evaluator, EvaluatorWithColdUser, IDMapper) keeping its lists on the device.
"""
import numpy as np
import pytest
import scipy.sparse as sps

import oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def core():
    import irspack_b200

    if irspack_b200.device_count() == 0:
        pytest.fail("GPU test selected but no CUDA device is visible")
    from irspack_b200 import _ials_core

    return _ials_core


def launches():
    from irspack_b200._lib import lib

    return int(lib.ials_kernel_launch_count())


# Kernels one recommend call launches when every row fits one slab (ials_kernel_launch_count,
# csrc/api_recommend.cu recommend_impl):
#   fused: per slab of 262 144 rows, launch_score_topk_tc = score_tc_kernel + merge_topk_kernel
#          (score_tc.cu); users by index add gather_rows_kernel (launch_gather_rows), embeddings add
#          pad_copy_kernel (launch_pad_copy), once per call.
#   SIMT:  per slab of 2^29 / (4 I) rows, score_tile_kernel + mask_rows_kernel (only with a mask) +
#          topk_rows_kernel (score.cu).
# A call with mask="train" also runs csr_sorted_kernel the first time (the trainer caches the
# answer), so routes are counted on a second call.
FUSED, GATHER_OR_PAD = 2, 1


def simt(masked):
    return 3 if masked else 2


def trainer(core, X, K, user, item):
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.05).build()
    g = core.IALSTrainer(cfg, X)
    g.user, g.item = user, item
    return g


def gt_all(rows, cols):  # every row is evaluated: give each one ground-truth item
    return sps.csr_matrix((np.ones(rows), (np.arange(rows), np.zeros(rows, int))), shape=(rows, cols))


def oracle_topk(user, item, k, mask=None, lists=None):
    """float64 scores, masked items and (with ``lists``: one shared or one per row) items outside
    a row's allow-list at -inf, then the oracle's top-k."""
    s = user.astype(np.float64) @ item.astype(np.float64).T
    if mask is not None:
        s[sps.csr_matrix(mask).nonzero()] = -np.inf
    if lists is not None:
        ok = np.zeros(s.shape, bool)
        for r in range(s.shape[0]):
            ok[r, np.asarray(lists[0] if len(lists) == 1 else lists[r], np.int64)] = True
        s[~ok] = -np.inf
    _, rec, cnt = oracle.topk_metrics(s, gt_all(*s.shape), k)
    return s, rec, cnt


def lists_csr(lists):
    indptr = np.zeros(len(lists) + 1, np.int64)
    np.cumsum([len(x) for x in lists], out=indptr[1:])
    flat = np.concatenate([np.asarray(x, np.int32) for x in lists]) if lists else np.zeros(0, np.int32)
    return len(lists), indptr, flat.astype(np.int32)


def check_lists(got, cnt, want, want_cnt, s64, rel=1e-5):
    np.testing.assert_array_equal(cnt, want_cnt)
    bad = np.flatnonzero((got != want).any(axis=1))
    for r in bad:
        finite = s64[r][np.isfinite(s64[r])]
        tol = rel * (np.abs(finite).max() if finite.size else 0.0) + 1e-12
        for a, b in zip(got[r], want[r]):
            if a != b:
                assert a >= 0 and b >= 0 and abs(s64[r, a] - s64[r, b]) <= tol, (r, a, b)
    return len(bad)


def check_scores(got, sc, s64):
    ok = got >= 0
    rows = np.repeat(np.arange(got.shape[0]), got.shape[1]).reshape(got.shape)
    np.testing.assert_allclose(sc[ok], s64[rows[ok], got[ok]], rtol=2e-5, atol=2e-5)


def train_matrix(U, I, seed, zeros=True):
    """0/1 training rows; with ``zeros``, a few rows hold stored zeros, which must not mask."""
    X = sps.random(U, I, density=min(0.05, 200.0 / I), random_state=seed, format="csr", dtype=np.float32)
    X.data[:] = 1.0
    if zeros:
        for r in range(1, U, 7):
            X.data[X.indptr[r]: X.indptr[r + 1]: 2] = 0.0
    return X


def effective(X):
    m = X.copy()
    m.eliminate_zeros()
    return m


# K -> row stride: 129 -> 160, 160, 200 -> 224, 256, 300 -> 320, 384, 448, 512 (padding columns
# at 129, 200 and 300); k reaches the three candidate capacities (64 / 128 / 256 keys)
@pytest.mark.parametrize("U,I,K,k", [
    (300, 5000, 256, 10),     # several catalogue splits (3 user tiles, 40 item tiles)
    (1000, 777, 129, 50),     # partial last user tile and last item tile
    (64, 100, 448, 1),        # one tile of everything
    (500, 17770, 256, 100),   # the configs[2] catalogue
    (130, 3000, 300, 128),    # k at the fused kernel's limit, 256-key buffers
    (257, 2100, 384, 50),
    (200, 1500, 160, 10),
    (333, 4000, 200, 100),
    (140, 2600, 512, 128),
])
def test_wide_topk_matches_oracle(core, U, I, K, k):
    rng = np.random.default_rng(U + I + K)
    X = train_matrix(U, I, seed=K)
    user = rng.standard_normal((U, K)).astype(np.float32)
    item = rng.standard_normal((I, K)).astype(np.float32)
    g = trainer(core, X, K, user, item)
    s64, want, want_cnt = oracle_topk(user, item, k, effective(X))
    got, cnt, sc = g.recommend(0, U, k, mask="train", return_scores=True)
    assert check_lists(got, cnt, want, want_cnt, s64) <= max(2, U // 50)
    check_scores(got, sc, s64)
    # sub-block [b, e): no mask, and a custom mask
    b, e = U // 3, U // 3 + min(U - U // 3, 77)
    s64, want, want_cnt = oracle_topk(user[b:e], item, k)
    got, cnt, sc = g.recommend(b, e, k, mask=None, return_scores=True)
    assert check_lists(got, cnt, want, want_cnt, s64) <= max(2, (e - b) // 50)
    check_scores(got, sc, s64)
    custom = sps.csr_matrix((rng.random((e - b, I)) < 0.2).astype(np.float32))
    s64, want, want_cnt = oracle_topk(user[b:e], item, k, custom)
    got, cnt, sc = g.recommend(b, e, k, mask=custom, return_scores=True)
    assert check_lists(got, cnt, want, want_cnt, s64) <= max(2, (e - b) // 50)
    check_scores(got, sc, s64)


@pytest.mark.parametrize("K", [256, 512])
def test_wide_topk_exact_on_integer_factors(core, K):
    """Small-integer factors: exact arithmetic, massive ties; the lists are the oracle's, and the
    first k columns of the SIMT route's lists at cutoff 150."""
    rng = np.random.default_rng(K)
    U, I = 300, 4000
    user = rng.integers(-2, 3, size=(U, K)).astype(np.float32)
    item = rng.integers(-2, 3, size=(I, K)).astype(np.float32)
    X = train_matrix(U, I, seed=4)
    g = trainer(core, X, K, user, item)
    simt150, simt_cnt = g.recommend(0, U, 150, mask="train")
    for k in (1, 10, 50, 100, 128):
        _, want, want_cnt = oracle_topk(user, item, k, effective(X))
        got, cnt = g.recommend(0, U, k, mask="train")
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(cnt, want_cnt)
        np.testing.assert_array_equal(got, simt150[:, :k])
        np.testing.assert_array_equal(cnt, np.minimum(simt_cnt, k))


@pytest.mark.parametrize("K", [256, 512])
def test_wide_allow_lists(core, K):
    """recommend(allowed=...) with a shared list and with per-user lists, under the training mask
    and a custom mask: the calls that raised NotImplementedError at row strides above 128."""
    rng = np.random.default_rng(11 + K)
    U, I = 200, 4500
    user = rng.integers(-1, 2, size=(U, K)).astype(np.float32)
    item = rng.integers(-1, 2, size=(I, K)).astype(np.float32)
    X = train_matrix(U, I, seed=8)
    g = trainer(core, X, K, user, item)
    shared = [np.sort(rng.choice(I, 1700, replace=False))]
    per_user = [np.sort(rng.choice(I, int(n), replace=False)) for n in rng.integers(0, 3000, size=U)]
    per_user[0] = np.zeros(0, np.int64)   # nothing recommendable
    per_user[1] = np.arange(I)            # everything
    per_user[2] = np.array([5, 4499])     # fewer than k, first and last tiles
    custom = sps.csr_matrix((rng.random((U, I)) < 0.2).astype(np.float32))
    for k in (1, 10, 50, 128):
        for lists in (shared, per_user):
            for mask, omask in (("train", effective(X)), (custom, custom)):
                _, want, want_cnt = oracle_topk(user, item, k, omask, lists)
                got, cnt = g.recommend(0, U, k, mask=mask, allowed=lists_csr(lists))
                np.testing.assert_array_equal(cnt, want_cnt)
                np.testing.assert_array_equal(got, want)
    assert cnt[0] == 0 and cnt[2] <= 2
    # sub-block: the lists are those of the block's rows
    b, e, k = 37, 171, 20
    for lists in (shared, per_user[b:e]):
        _, want, want_cnt = oracle_topk(user[b:e], item, k, effective(X[b:e]), lists)
        got, cnt = g.recommend(b, e, k, mask="train", allowed=lists_csr(lists))
        np.testing.assert_array_equal(cnt, want_cnt)
        np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("K", [256, 512])
def test_wide_allow_lists_random_factors(core, K):
    rng = np.random.default_rng(3 * K)
    U, I, k = 300, 17770, 10
    X = train_matrix(U, I, seed=5)
    user = rng.standard_normal((U, K)).astype(np.float32)
    item = rng.standard_normal((I, K)).astype(np.float32)
    g = trainer(core, X, K, user, item)
    per_user = [np.sort(rng.choice(I, int(n), replace=False)) for n in rng.integers(0, I, size=U)]
    for lists in ([np.sort(rng.choice(I, I // 3, replace=False))], per_user):
        s64, want, want_cnt = oracle_topk(user, item, k, effective(X), lists)
        got, cnt, sc = g.recommend(0, U, k, mask="train", return_scores=True, allowed=lists_csr(lists))
        assert check_lists(got, cnt, want, want_cnt, s64) <= max(2, U // 50)
        check_scores(got, sc, s64)


@pytest.mark.parametrize("K", [256, 512])
def test_wide_users_picked_by_index(core, K):
    """recommend_users: arbitrary order and repeats, each user's own training row as the mask
    (raised NotImplementedError above stride 128), custom masks, allow-lists by position."""
    rng = np.random.default_rng(17 + K)
    U, I, k = 400, 3000, 20
    user = rng.integers(-1, 2, size=(U, K)).astype(np.float32)
    item = rng.integers(-1, 2, size=(I, K)).astype(np.float32)
    X = train_matrix(U, I, seed=9)
    g = trainer(core, X, K, user, item)
    pick = np.concatenate([rng.permutation(U)[:170], [5, 5, 399, 0]])
    _, want, want_cnt = oracle_topk(user[pick], item, k, effective(X)[pick])
    got, cnt, sc = g.recommend_users(pick, k, mask="train", return_scores=True)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(cnt, want_cnt)
    custom = sps.csr_matrix((rng.random((pick.size, I)) < 0.2).astype(np.float32))
    lists = [np.sort(rng.choice(I, int(n), replace=False)) for n in rng.integers(0, 1500, pick.size)]
    for allowed in (None, [np.sort(rng.choice(I, 900, replace=False))], lists):
        for mask, omask in (("train", effective(X)[pick]), (custom, custom)):
            _, want, want_cnt = oracle_topk(user[pick], item, k, omask, allowed)
            got, cnt = g.recommend_users(pick, k, mask=mask,
                                         allowed=None if allowed is None else lists_csr(allowed))
            np.testing.assert_array_equal(cnt, want_cnt)
            np.testing.assert_array_equal(got, want)


def test_wide_embeddings(core):
    """recommend_embeddings at K = 200 (row stride 224: the padding is made on the device) with a
    mask and with allow-lists."""
    rng = np.random.default_rng(23)
    U, I, K, k = 50, 2500, 200, 15
    user = rng.integers(-1, 2, size=(U, K)).astype(np.float32)
    item = rng.integers(-1, 2, size=(I, K)).astype(np.float32)
    g = trainer(core, train_matrix(U, I, seed=2), K, user, item)
    emb = rng.integers(-2, 3, size=(333, K)).astype(np.float32)
    mask = sps.csr_matrix((rng.random((333, I)) < 0.1).astype(np.float32))
    lists = [np.sort(rng.choice(I, int(n), replace=False)) for n in rng.integers(0, 900, 333)]
    shared = [np.sort(rng.choice(I, 700, replace=False))]
    for m, allowed in ((mask, None), (None, lists), (mask, lists), (mask, shared)):
        _, want, want_cnt = oracle_topk(emb, item, k, m, allowed)
        got, cnt = g.recommend_embeddings(emb, k, mask=m, allowed=None if allowed is None else lists_csr(allowed))
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(cnt, want_cnt)
    np.testing.assert_array_equal(g.item, item)  # the model is untouched


def test_wide_routes_by_launch_count(core):
    """Which kernels each call runs at K = 256 (counts derived at the top of this file)."""
    rng = np.random.default_rng(41)
    U, I, K = 300, 3000, 256
    user = rng.integers(-1, 2, size=(U, K)).astype(np.float32)
    item = rng.integers(-1, 2, size=(I, K)).astype(np.float32)
    X = train_matrix(U, I, seed=6)
    g = trainer(core, X, K, user, item)
    custom = sps.csr_matrix((rng.random((U, I)) < 0.1).astype(np.float32))
    shared = lists_csr([np.arange(0, I, 3)])
    pick = np.array([3, 1, 3, 299])

    def count(call):
        call()  # the first mask="train" call checks that the training rows ascend, once
        n0 = launches()
        call()
        return launches() - n0

    assert count(lambda: g.recommend(0, U, 10, mask="train")) == FUSED
    assert count(lambda: g.recommend(0, U, 10, mask=None)) == FUSED
    assert count(lambda: g.recommend(0, U, 10, mask=custom)) == FUSED
    assert count(lambda: g.recommend(0, U, 10, mask="train", allowed=shared)) == FUSED
    assert count(lambda: g.recommend_users(pick, 10, mask="train")) == GATHER_OR_PAD + FUSED
    assert count(lambda: g.recommend_embeddings(user[:7], 10, allowed=shared)) == GATHER_OR_PAD + FUSED
    # cutoffs past 128 stay on the SIMT route; allow-lists and users by index with their training
    # rows as the mask have no such route and still raise
    assert count(lambda: g.recommend(0, U, 150, mask="train")) == simt(True)
    assert count(lambda: g.recommend(0, U, 150, mask=None)) == simt(False)
    with pytest.raises(NotImplementedError):
        g.recommend(0, U, 150, mask="train", allowed=shared)
    with pytest.raises(NotImplementedError):
        g.recommend_users(pick, 150, mask="train")


@pytest.mark.parametrize("K", [64, 256])
def test_unsorted_training_rows_fall_back(core, monkeypatch, K):
    """Training rows whose column ids do not ascend (a CSR handed to the C ABI as it is) cannot
    feed the fused kernel's mask cursor: block calls take the SIMT route, calls that only the
    fused kernel serves raise -- the same at row stride 128 (K = 64) and 256."""
    from irspack_b200 import _ials_core

    rng = np.random.default_rng(K + 1)
    U, I, k = 200, 1500, 10
    S = sps.csr_matrix((rng.random((U, I)) < 0.05).astype(np.float32))
    S.sort_indices()
    indices = S.indices.copy()
    for r in range(U):  # every row descending
        indices[S.indptr[r]: S.indptr[r + 1]] = indices[S.indptr[r]: S.indptr[r + 1]][::-1].copy()
    X = sps.csr_matrix((S.data, indices, S.indptr), shape=S.shape)
    monkeypatch.setattr(_ials_core, "_canonical_csr", lambda M: sps.csr_matrix(M, dtype=np.float32, copy=True))
    user = rng.integers(-1, 2, size=(U, K)).astype(np.float32)
    item = rng.integers(-1, 2, size=(I, K)).astype(np.float32)
    g = trainer(core, X, K, user, item)
    n0 = launches()
    got, cnt = g.recommend(0, U, k, mask="train")
    assert launches() - n0 == 1 + simt(True)  # csr_sorted_kernel, then the SIMT route
    _, want, want_cnt = oracle_topk(user, item, k, S)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(cnt, want_cnt)
    n0 = launches()
    g.recommend(0, U, k, mask="train")
    assert launches() - n0 == simt(True)
    with pytest.raises(NotImplementedError):
        g.recommend(0, U, k, mask="train", allowed=lists_csr([np.arange(I // 2)]))
    with pytest.raises(NotImplementedError):
        g.recommend_users(np.array([4, 2]), k, mask="train")
    # an explicit mask is sorted on the way in: the fused kernel serves it
    n0 = launches()
    got, cnt = g.recommend(0, U, k, mask=S, allowed=lists_csr([np.arange(I // 2)]))
    assert launches() - n0 == FUSED
    _, want, want_cnt = oracle_topk(user, item, k, S, [np.arange(I // 2)])
    np.testing.assert_array_equal(got, want)


# ---------------------------------------------------------------------------------------
# host layer: at K = 256 the Evaluator and the IDMapper keep their lists on the device
# ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def wide_model():
    from irspack_b200 import IALSRecommender

    rng = np.random.default_rng(51)
    U, I, K = 260, 900, 256
    X = sps.csr_matrix((rng.random((U, I)) < 0.04).astype(np.float32))
    rec = IALSRecommender(X, n_components=K, alpha0=0.1, reg=0.05, train_epochs=1).learn()
    t = rec.trainer_as_ials.core_trainer   # integer factors: no near-ties between the two paths
    t.user = rng.integers(-2, 3, size=(U, K)).astype(np.float32)
    t.item = rng.integers(-2, 3, size=(I, K)).astype(np.float32)
    return rec, X, rng


def test_wide_evaluator_lists_take_the_fused_path(wide_model, monkeypatch):
    from irspack_b200 import Evaluator, EvaluatorWithColdUser

    rec, X, rng = wide_model
    U, I = X.shape
    t = rec.trainer_as_ials.core_trainer
    te = sps.csr_matrix((rng.random((U, I)) < 0.02).astype(np.float32))

    class HostOnly:  # no recommend_block: score blocks on the host + select_topk
        X_train_all, n_users, n_items = rec.X_train_all, U, I
        get_score_block = staticmethod(rec.get_score_block)

    shared = [int(i) for i in rng.permutation(I)[:400]]                    # unsorted on purpose
    per_user = [[int(i) for i in rng.choice(I, int(n))] for n in rng.integers(0, 700, U)]  # duplicates too
    other = sps.csr_matrix((rng.random((U, I)) < 0.1).astype(np.float32))
    class ColdHost:
        n_items = I
        get_score_cold_user = staticmethod(rec.get_score_cold_user)

    warm = [Evaluator(te, cutoff=10, mb_size=64, **kw)
            for kw in (dict(recommendable_items=shared), dict(per_user_recommendable_items=per_user),
                       dict(per_user_recommendable_items=per_user, masked_interactions=other))]
    cold = [EvaluatorWithColdUser(X[:50], te[:50], cutoff=10, mb_size=16, **kw)
            for kw in (dict(per_user_recommendable_items=per_user[:50]), dict(recommendable_items=shared))]
    want = [ev.get_score(HostOnly()) for ev in warm] + [ev.get_score(ColdHost()) for ev in cold]

    def no_score_block(*a, **kw):
        raise AssertionError("the fused path must not fall back to a host score block")

    monkeypatch.setattr(type(rec), "get_score_block", no_score_block)
    monkeypatch.setattr(type(rec), "get_score_cold_user", no_score_block)
    calls = []
    for name in ("recommend", "recommend_embeddings"):
        orig = getattr(type(t), name)
        monkeypatch.setattr(type(t), name, lambda self, *a, _orig=orig, **kw:
                            calls.append(kw.get("allowed") is not None) or _orig(self, *a, **kw))
    for ev, w, tol in zip(warm + cold, want, [1e-12] * len(warm) + [1e-9] * len(cold)):
        calls.clear()
        got = ev.get_score(rec)
        assert calls and all(calls)  # every block went through the fused kernel with its lists
        for key, v in w.items():
            assert got[key] == pytest.approx(v, abs=tol), key


def test_wide_id_mapper_serves_without_a_score_block(wide_model, monkeypatch):
    from irspack_b200.id_mapping import IDMapper

    rec, X, rng = wide_model
    U, I = X.shape
    user_ids = [f"u{i}" for i in range(U)]
    item_ids = [f"i{j}" for j in range(I)]
    mapper = IDMapper(user_ids, item_ids)

    class HostOnly:  # the same model without the fused entry points
        n_users, n_items, X_train_all = U, I, rec.X_train_all
        get_score_remove_seen = staticmethod(rec.get_score_remove_seen)

    def same(got, want):
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert [i for i, _ in g] == [i for i, _ in w]
            np.testing.assert_allclose([v for _, v in g], [v for _, v in w], rtol=1e-5, atol=1e-5)

    picked = [user_ids[i] for i in (7, 3, 259, 3, 0, 88)]
    shared = [item_ids[j] for j in rng.permutation(I)[:300]] + ["no such item"]
    per_user = [[item_ids[j] for j in rng.choice(I, int(n))] for n in rng.integers(0, 400, len(picked))]
    forbidden = [[item_ids[j] for j in rng.choice(I, 50)] for _ in picked]
    cases = (dict(allowed_item_ids=shared), dict(per_user_allowed_item_ids=per_user),
             dict(forbidden_item_ids=forbidden), dict(allowed_item_ids=shared, forbidden_item_ids=forbidden),
             dict(per_user_allowed_item_ids=per_user, forbidden_item_ids=forbidden))
    want = {(i, c): mapper.recommend_for_known_user_batch(HostOnly(), picked, cutoff=c, **kw)
            for i, kw in enumerate(cases) for c in (1, 10, 128)}

    def no_score_block(*a, **kw):
        raise AssertionError("the fused path must not build a host score block")

    monkeypatch.setattr(type(rec), "get_score_remove_seen", no_score_block)
    for i, kw in enumerate(cases):
        for c in (1, 10, 128):
            same(mapper.recommend_for_known_user_batch(rec, picked, cutoff=c, **kw), want[(i, c)])
