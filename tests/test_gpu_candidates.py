"""Candidate ranking (``IALSTrainer.rank_candidates``, ``ials_trainer_rank_candidates``) and pair scores
(``candidate_scores``, ``ials_trainer_candidate_scores``) against float64 numpy on the same factors.

* Lists: the tie and score tolerances of the similar-items tests (``test_gpu_similar._check``): the float64
  order (-score, index) except between entries whose float64 scores differ by less than 1e-5 of the row's
  largest |score|; exactly equal float64 scores in ascending index order; scores within 2e-5.
* Every row stride (K = 16 .. 512), cutoffs 1, 10, 128, 129 and 1024, lists of length 0, 1, below, at and
  above the cutoff, longer than 2048 (the filter compacts more than once) and the whole catalogue.
* Shared and per-row lists; queries by range, by index (repeats, any order) and as embeddings; masks
  "train" (a stored zero masks nothing), none and explicit, a row whose candidates are all masked; one call
  over more than one slab of rows; rejected arguments; launches independent of the catalogue; no side
  effects.  Factors are set through the setters."""
import numpy as np
import pytest
import scipy.sparse as sps

from test_gpu_similar import TIE, _check

pytestmark = pytest.mark.gpu

SLAB = 262144  # kListSlabRows


@pytest.fixture(scope="module")
def core():
    import irspack_b200

    if irspack_b200.device_count() == 0:
        pytest.fail("GPU test selected but no CUDA device is visible")
    from irspack_b200 import _ials_core

    return _ials_core


def _trainer(core, U, I, K, seed=0, density=0.02):
    rng = np.random.default_rng(seed)
    X = sps.csr_matrix((rng.random((U, I)) < density).astype(np.float32))
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.05).build()
    tr = core.IALSTrainer(cfg, X)
    user = (rng.standard_normal((U, 1)) * 0.2 + rng.standard_normal((U, K)) * 0.3).astype(np.float32)
    item = (rng.standard_normal((I, 1)) * 0.2 + rng.standard_normal((I, K)) * 0.3).astype(np.float32)
    tr.user = user
    tr.item = item
    return tr, X, user, item


def _ok(n_items, lists, hidden=None):
    """Boolean [rows, n_items]: the candidates each row may receive."""
    ok = np.zeros((len(lists), n_items), dtype=bool)
    for r, lst in enumerate(lists):
        ok[r, np.asarray(lst, dtype=np.int64)] = True
    if hidden is not None:
        ok &= ~hidden
    return ok


def _csr_lists(lists):
    ip = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=ip[1:])
    ix = np.concatenate([np.asarray(x, dtype=np.int32) for x in lists]) if ip[-1] else np.empty(0, np.int32)
    return len(lists), ip, ix


def _seen(X, q):
    """The non-zeros of X's rows q (stored zeros dropped) as a boolean matrix."""
    m = sps.csr_matrix(X[q], copy=True)
    m.eliminate_zeros()
    return m.toarray() != 0


@pytest.mark.parametrize("K", [16, 64, 128, 200, 256, 512])
def test_row_strides_cutoffs_and_list_lengths(core, K):
    U, I = 120, 3000
    tr, X, user, item = _trainer(core, U, I, K, seed=K)
    rng = np.random.default_rng(K + 1)
    for k in (1, 10, 128, 129, 1024):
        lengths = [0, 1, max(k - 1, 0), k, k + 7, 2500, I]
        lists = [np.sort(rng.choice(I, n, replace=False)) for n in lengths]
        q = rng.integers(0, U, size=len(lists))
        S = user[q].astype(np.float64) @ item.astype(np.float64).T
        idx, cnt, sc = tr.rank_candidates(q, lists, k, mask=None)
        _check(S, _ok(I, lists), k, idx, cnt, sc)
    # the whole catalogue as one list: recommend's SIMT lists at k = 150, up to ties
    q = np.arange(0, 40)
    idx, cnt, sc = tr.rank_candidates(range(0, 40), [np.arange(I)], 150, mask="train")
    ridx, rcnt, rsc = tr.recommend(0, 40, 150, mask="train", return_scores=True)
    assert np.array_equal(cnt, rcnt)
    S = user[q].astype(np.float64) @ item.astype(np.float64).T
    for r in range(q.size):
        tie = TIE * np.abs(S[r]).max()
        same = idx[r] == ridx[r]
        assert np.all(same | (np.abs(S[r, idx[r]] - S[r, ridx[r]]) <= tie)), r


def test_query_forms_and_masks(core):
    U, I, K = 200, 700, 96
    tr, X, user, item = _trainer(core, U, I, K, seed=3, density=0.05)
    X = sps.csr_matrix(X, copy=True)
    u0 = 11
    z = int(X[u0].indices[0])
    X[u0, z] = 0.0  # a stored zero in the training matrix: it masks nothing
    assert X[u0, z] == 0 and z in sps.csr_matrix(X)[u0].indices
    cfg = core.IALSModelConfigBuilder().set_K(K).build()
    tr = core.IALSTrainer(cfg, X)
    X.sort_indices()
    tr.user, tr.item = user, item
    rng = np.random.default_rng(4)
    shared = np.sort(rng.choice(I, 300, replace=False))
    shared = np.union1d(shared, [z]).astype(np.int32)
    item64 = item.astype(np.float64)
    for k in (10, 200):
        # a range of users, one shared list, mask "train"
        b, e = 5, 150
        q = np.arange(b, e)
        idx, cnt, sc = tr.rank_candidates(range(b, e), [shared], k)
        _check(user[q].astype(np.float64) @ item64.T, _ok(I, [shared] * q.size, _seen(X, q)), k, idx, cnt, sc)
        # users by index (repeats, any order), per-row lists given unsorted with repeats
        q = rng.integers(0, U, size=60)
        q[7] = q[2] = u0
        lists = [rng.integers(0, I, size=int(n)) for n in rng.integers(0, 400, size=60)]
        lists[7] = lists[2]
        clean = [np.unique(x) for x in lists]
        idx, cnt, sc = tr.rank_candidates(q, lists, k)
        _check(user[q].astype(np.float64) @ item64.T, _ok(I, clean, _seen(X, q)), k, idx, cnt, sc)
        assert np.array_equal(idx[7], idx[2]) and np.array_equal(sc[7], sc[2])
        # an explicit mask, and none
        m = sps.random(60, I, density=0.1, random_state=5, format="csr", dtype=np.float32)
        m.data[:] = 1.0
        idx, cnt, sc = tr.rank_candidates(q, lists, k, mask=m)
        _check(user[q].astype(np.float64) @ item64.T, _ok(I, clean, m.toarray() != 0), k, idx, cnt, sc)
        idx, cnt, sc = tr.rank_candidates(q, _csr_lists(clean), k, mask=None)
        _check(user[q].astype(np.float64) @ item64.T, _ok(I, clean), k, idx, cnt, sc)
        # embeddings (mask None or explicit)
        emb = rng.standard_normal((40, K)).astype(np.float32)
        idx, cnt, sc = tr.rank_candidates_embeddings(emb, lists[:40], k, mask=m[:40])
        _check(emb.astype(np.float64) @ item64.T, _ok(I, clean[:40], m[:40].toarray() != 0), k, idx, cnt, sc)
        idx2, cnt2, sc2 = tr.rank_candidates_embeddings(tr.user[q[:40]], lists[:40], k)
        idx3, cnt3, sc3 = tr.rank_candidates(q[:40], lists[:40], k, mask=None)
        assert np.array_equal(idx2, idx3) and np.array_equal(sc2, sc3)
    # a row whose candidates are all masked, and an empty list: count 0, padded
    seen0 = X[u0].indices[X[u0].data != 0]
    idx, cnt = tr.rank_candidates(np.array([u0, u0]), [seen0, []], 5, return_scores=False)
    assert list(cnt) == [0, 0] and np.all(idx == -1)


def test_one_call_over_more_than_one_slab(core):
    U, I = SLAB + 300, 200
    tr, X, user, item = _trainer(core, U, I, 32, seed=5, density=0.002)
    rng = np.random.default_rng(6)
    lens = rng.integers(0, 6, size=U)
    ip = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(lens, out=ip[1:])
    ix = np.concatenate([np.sort(rng.choice(I, n, replace=False)) for n in lens]).astype(np.int32)
    idx, cnt, sc = tr.rank_candidates(range(0, U), (U, ip, ix), 3)
    q = np.concatenate([np.arange(SLAB - 5, SLAB + 5), [0, U - 1], rng.integers(0, U, size=20)])
    lists = [ix[ip[r]:ip[r + 1]] for r in q]
    _check(user[q].astype(np.float64) @ item.astype(np.float64).T, _ok(I, lists, _seen(X, q)), 3,
           idx[q], cnt[q], sc[q])


WARP_MAX = 256  # longest list the warp-per-row selection takes (kWarpTkMax)


def test_both_selection_paths(core):
    """Slabs whose longest list is <= 256 take the warp-per-row selection, longer ones the CTA per row: lists
    at and around the threshold, cutoffs below and above it, and the same rows through both paths."""
    U, I = 150, 2000
    tr, X, user, item = _trainer(core, U, I, 128, seed=31)
    rng = np.random.default_rng(32)
    S_all = user.astype(np.float64) @ item.astype(np.float64).T
    for longest in (WARP_MAX, WARP_MAX + 1):
        lengths = [0, 1, 31, 32, 33, 100, 255, WARP_MAX, longest]
        lists = [np.sort(rng.choice(I, n, replace=False)) for n in lengths]
        q = rng.integers(0, U, size=len(lists))
        for k in (1, 10, 255, 256, 257, 1024):
            idx, cnt, sc = tr.rank_candidates(q, lists, k)
            _check(S_all[q], _ok(I, lists, _seen(X, q)), k, idx, cnt, sc)
    # the same short rows alone (warp path) and next to one list of 257 (CTA path): the same bits
    lists = [np.sort(rng.choice(I, int(n), replace=False)) for n in rng.integers(0, WARP_MAX + 1, size=40)]
    q = rng.integers(0, U, size=40)
    for k in (10, 300):
        warp = tr.rank_candidates(q, lists, k)
        cta = tr.rank_candidates(np.append(q, 0), lists + [np.arange(WARP_MAX + 1)], k)
        for a, b in zip(warp, cta):
            assert np.array_equal(a, b[:40]), k


def test_unsorted_explicit_mask_and_stored_zero(core):
    """A mask row given unsorted and with repeats through the C ABI (scanned, not searched); a stored zero of
    the training matrix that is the only candidate of its row."""
    U, I = 60, 500
    tr, X, user, item = _trainer(core, U, I, 64, seed=33, density=0.05)
    rng = np.random.default_rng(34)
    q = np.array([4, 9, 4, 30], np.int64)
    lists = [np.sort(rng.choice(I, 120, replace=False)).astype(np.int32) for _ in q]
    n_lists, ip, ix = _csr_lists(lists)
    rows = [rng.choice(lst, 40) for lst in lists]  # repeats, any order
    m_ip = np.zeros(q.size + 1, np.int64)
    np.cumsum([r.size for r in rows], out=m_ip[1:])
    m_ix = np.concatenate(rows).astype(np.int32)
    k = 50
    idx, cnt, sc = np.empty((q.size, k), np.int32), np.empty(q.size, np.int32), np.empty((q.size, k), np.float32)
    p = core._ptr
    core.check(core.lib.ials_trainer_rank_candidates(tr._handle, p(q), None, 0, q.size, k, 2, p(m_ip), p(m_ix),
                                                     n_lists, p(ip), p(ix), p(idx), p(sc), p(cnt)))
    hidden = np.zeros((q.size, I), bool)
    for r, row in enumerate(rows):
        hidden[r, row] = True
    _check(user[q].astype(np.float64) @ item.astype(np.float64).T, _ok(I, lists, hidden), k, idx, cnt, sc)
    ref = tr.rank_candidates(q, lists, k, mask=sps.csr_matrix(hidden.astype(np.float32)))
    assert np.array_equal(idx, ref[0]) and np.array_equal(cnt, ref[1])
    # a stored zero in X masks nothing: its item, alone on the list, comes back with count 1
    X2 = sps.csr_matrix(X, copy=True)
    u0 = int(np.flatnonzero(np.diff(X2.indptr) > 1)[0])
    z = int(X2[u0].indices[0])
    X2[u0, z] = 0.0
    cfg = core.IALSModelConfigBuilder().set_K(64).build()
    tr2 = core.IALSTrainer(cfg, X2)
    tr2.user, tr2.item = user, item
    other = int(X2[u0].indices[1])  # a stored non-zero masks
    idx, cnt = tr2.rank_candidates(np.array([u0, u0]), [[z], [other]], 1, return_scores=False)
    assert list(cnt) == [1, 0] and idx[0, 0] == z and idx[1, 0] == -1


def test_launches_do_not_follow_the_catalogue(core):
    counts = []
    for I in (1000, 40000):
        tr, X, user, item = _trainer(core, 300, I, 128, seed=7, density=0.001)
        lists = [np.arange(0, 90, 3)] * 50
        tr.rank_candidates(range(0, 50), lists, 10)  # the first mask="train" call checks X's row order once
        n0 = int(core.lib.ials_kernel_launch_count())
        tr.rank_candidates(range(0, 50), lists, 10)
        counts.append(int(core.lib.ials_kernel_launch_count()) - n0)
    assert counts == [2, 2]  # cand_scores_kernel + topk_segments_kernel: no score_tc kernel, no dense scores


def test_candidate_scores_and_pairs(core):
    U, I = 80, 400
    tr, X, user, item = _trainer(core, U, I, 200, seed=9)
    rng = np.random.default_rng(10)
    q = np.array([3, 3, 70, 0, 3])
    lists = [rng.integers(0, I, size=n) for n in (5, 0, 9, 1, 300)]
    lists[0][1] = lists[0][3]  # a repeat
    got = tr.candidate_scores(q, lists)
    want = np.concatenate([user[u].astype(np.float64) @ item[l].astype(np.float64).T for u, l in zip(q, lists)])
    assert got.shape == want.shape and np.abs(got - want).max() <= 2e-5 * np.abs(want).max()
    assert got[1] == got[3]
    got = tr.candidate_scores(range(10, 14), [[5, 1, 5]])  # a shared list, once per row
    want = (user[10:14].astype(np.float64) @ item[[5, 1, 5]].astype(np.float64).T).reshape(-1)
    assert np.abs(got - want).max() <= 2e-5 * np.abs(want).max()


def test_agrees_with_recommend_users_allow_lists(core):
    U, I = 300, 2000
    tr, X, user, item = _trainer(core, U, I, 128, seed=11)
    rng = np.random.default_rng(12)
    q = rng.integers(0, U, size=100)
    lists = [np.sort(rng.choice(I, int(n), replace=False)).astype(np.int32) for n in rng.integers(1, 120, size=100)]
    n_lists, ip, ix = _csr_lists(lists)
    idx, cnt, sc = tr.rank_candidates(q, (n_lists, ip, ix), 10)
    ridx, rcnt, rsc = tr.recommend_users(q, 10, mask="train", return_scores=True, allowed=(n_lists, ip, ix))
    assert np.array_equal(cnt, rcnt)
    S = user[q].astype(np.float64) @ item.astype(np.float64).T
    for r in range(q.size):
        tie = TIE * np.abs(S[r]).max()
        assert np.all((idx[r] == ridx[r]) | (np.abs(S[r, idx[r]] - S[r, ridx[r]]) <= tie)), r


def test_rejected_arguments(core):
    tr, X, user, item = _trainer(core, 50, 80, 32, seed=13)
    lib, p, E = core.lib, core._ptr, core._lib.IALS_ERR_INVALID_ARGUMENT
    idx, cnt = np.empty((2, 80), np.int32), np.empty(2, np.int32)

    def rank(k=3, ip=(0, 2, 3), ix=(4, 7, 9), n_lists=2, q=(0, 1), emb=None, begin=0, end=2, mode=1):
        ip, ix = np.asarray(ip, np.int64), np.asarray(ix, np.int32)
        qa = None if q is None else np.asarray(q, np.int64)
        ea = None if emb is None else np.asarray(emb, np.float32)
        return lib.ials_trainer_rank_candidates(tr._handle, p(qa), p(ea), begin, end, k, mode, None, None, n_lists,
                                                p(ip), p(ix), p(idx), None, p(cnt))

    assert rank() == 0
    for kw in [dict(ix=(7, 4, 9)), dict(ix=(4, 4, 9)), dict(ix=(4, 7, 80)), dict(ix=(-1, 7, 9)),
               dict(n_lists=3, ip=(0, 1, 2, 3)), dict(k=0), dict(k=1025), dict(k=81),
               dict(emb=np.zeros((2, 32))), dict(emb=np.zeros((2, 32)), q=None, mode=0),
               dict(ip=(0, 2, 1), ix=(4, 7)), dict(q=(0, 50)), dict(mode=3)]:
        assert rank(**kw) == E, kw
    assert lib.ials_trainer_candidate_scores(tr._handle, None, None, 0, 1, p(np.array([0, 1], np.int64)),
                                             p(np.array([80], np.int32)), p(np.empty(1, np.float32))) == E
    for kw in [dict(cutoff=0), dict(cutoff=81), dict(mask="seen"), dict(candidates=[[1], [2], [3]]),
               dict(candidates=[[1, 80]]), dict(candidates=[[-1]]), dict(user_indices=range(0, 51)),
               dict(user_indices=[0, 50])]:
        args = dict(user_indices=[0, 1], candidates=[[1, 2]], cutoff=2)
        args.update(kw)
        with pytest.raises(ValueError):
            tr.rank_candidates(args.pop("user_indices"), args.pop("candidates"), args.pop("cutoff"), **args)
    with pytest.raises(ValueError):
        tr.rank_candidates_embeddings(np.zeros((2, 32), np.float32), [[1]], 2, mask="train")


def test_no_side_effects(core):
    a, X, user, item = _trainer(core, 260, 390, 64, seed=23)
    b, _, _, _ = _trainer(core, 260, 390, 64, seed=23)
    lists = [np.arange(0, 390, 7)] * 20
    a.rank_candidates(np.arange(20), lists, 10)
    a.rank_candidates_embeddings(user[:20], lists, 129)
    a.candidate_scores(range(0, 20), lists)
    assert np.array_equal(a.user, b.user) and np.array_equal(a.item, b.item)
    sc = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CG).build()
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
    ct = rec.trainer_as_ials.core_trainer
    lists = [[3, 9, 50, 139], [1, 2, 3]]
    for got, q in ((rec.rank_candidates([-1, 3], lists, 3), [U - 1, 3]),
                   (rec.rank_candidates(np.arange(U) < 2, lists, 3), [0, 1])):
        for g, r in zip(got, ct.rank_candidates(np.array(q), lists, 3)):
            assert np.array_equal(g, r)
    Xc = X[:4]
    got = rec.rank_candidates_cold_user(Xc, [np.arange(0, I, 2)], 5)
    ref = ct.rank_candidates_embeddings(rec.compute_user_embedding(Xc), [np.arange(0, I, 2)], 5, mask=Xc)
    for g, r in zip(got, ref):
        assert np.array_equal(g, r)
    with pytest.raises(ValueError):
        rec.rank_candidates_cold_user(Xc, [[1]], 5, mask="train")
    pairs = rec.get_score_pairs([0, 5, 0, -1], [3, 3, 3, 7])
    ref = np.array([ct.candidate_scores([u], [[i]])[0] for u, i in ((0, 3), (5, 3), (0, 3), (U - 1, 7))])
    assert np.array_equal(pairs, ref)

    uids = [f"u{i}" for i in range(U)]
    iids = [f"i{i}" for i in range(I)]
    mapper = IDMapper(uids, iids)
    got = mapper.rank_items_for_known_users(rec, ["u4", "u0"], [["i3", "nope", "i9", "i3"], ["i1"]], cutoff=2)
    idx, cnt, sc = ct.rank_candidates(np.array([4, 0]), [[3, 9], [1]], 2)
    assert got == [[(iids[i], float(v)) for i, v in zip(idx[r, :cnt[r]], sc[r, :cnt[r]])] for r in range(2)]
    got = mapper.rank_items_for_new_user(rec, ["i1", "i2"], ["i1", "i5", "i6"], cutoff=5)
    assert [x for x, _ in got] != [] and "i1" not in [x for x, _ in got]
    got_all = mapper.rank_items_for_new_user(rec, ["i1", "i2"], ["i1", "i5", "i6"], cutoff=5, remove_seen=False)
    assert sorted(x for x, _ in got_all) == ["i1", "i5", "i6"]
