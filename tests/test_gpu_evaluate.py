"""ShardedEvaluator of a world-1 row-sharded trainer (no process group) against the single-process
Evaluator on an IALSRecommender holding the same factors, and the device diversity reduction against
Metrics.as_dict.  Integer-valued factors: every score is exact, so both sides rank the same lists and
every metric agrees to the last bits a different summation order leaves."""
import numpy as np
import pytest
import scipy.sparse as sps

pytestmark = pytest.mark.gpu

KEYS = ("total_user", "valid_user", "n_items", "hit", "ndcg", "recall", "map", "precision",
        "appeared_item", "entropy", "gini_index")


def _assert_same(got, want, tol=1e-12):
    assert got.keys() == want.keys()
    for k in want:
        a, b = got[k], want[k]
        if np.isnan(b):
            assert np.isnan(a), k
        else:
            assert a == pytest.approx(b, rel=tol, abs=tol), (k, a, b)


def _model(K, U=300, I=453, seed=0):
    """(sharded trainer, IALSRecommender, X, rng): the same integer factors in both; X has a user with
    every item seen, and stored zeros (not masked)."""
    from irspack_b200 import IALSRecommender
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer

    rng = np.random.default_rng(seed + K)
    X = sps.csr_matrix((rng.random((U, I)) < 0.05).astype(np.float32))
    X = X.tolil()
    X[3, :] = 1.0               # every item seen: n_rec = 0
    X[7, 5] = 0.0
    X = sps.csr_matrix(X)
    X[8, 11] = 0.0              # a stored zero: not part of the mask
    assert X[8, 11] == 0 and X.nnz > 0
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.05).build()
    tr = ShardedIALSTrainer.from_global(cfg, X, rank=0, world=1)
    rec = IALSRecommender(X, n_components=K, alpha0=0.1, reg=0.05, train_epochs=1).learn()
    u = rng.integers(-2, 3, size=(U, K)).astype(np.float32)
    it = rng.integers(-2, 3, size=(I, K)).astype(np.float32)
    tr.user, tr.item = u, it
    rec.trainer_as_ials.core_trainer.user = u
    rec.trainer_as_ials.core_trainer.item = it
    return tr, rec, X, rng


def _ground_truth(rng, U, I):
    gt = sps.csr_matrix((rng.random((U, I)) < 0.04).astype(np.float64))
    gt = gt.tolil()
    gt[0, :] = 0                # empty ground truth: counted in total_user only
    gt[3, 2] = 1.0              # the user with nothing recommendable
    return sps.csr_matrix(gt)


@pytest.fixture(scope="module")
def m128():
    return _model(128, I=1100)  # room for cutoff 1024; not a multiple of 128


@pytest.mark.parametrize("cutoffs", [[1, 5, 10, 20, 128], [150, 1024]])
@pytest.mark.parametrize("recall_with_cutoff", [False, True])
def test_cutoffs_fused_and_simt_match_evaluator(m128, cutoffs, recall_with_cutoff):
    from irspack_b200 import Evaluator
    from irspack_b200.dist import ShardedEvaluator

    tr, rec, X, rng = m128
    U, I = X.shape
    gt = _ground_truth(np.random.default_rng(1), U, I)
    want = Evaluator(gt, recall_with_cutoff=recall_with_cutoff).get_scores(rec, cutoffs)
    sev = ShardedEvaluator.from_global(tr, gt, recall_with_cutoff=recall_with_cutoff)
    got = sev.get_scores(tr, cutoffs)
    _assert_same(got, want)
    assert got == sev.get_scores(tr, cutoffs)  # two passes: bit-identical
    assert sev.get_target_score(tr) == pytest.approx(Evaluator(gt).get_target_score(rec), rel=1e-12)


@pytest.mark.parametrize("K", [32, 64, 128, 200, 256, 512])
def test_row_strides(K):
    from irspack_b200 import Evaluator
    from irspack_b200.dist import ShardedEvaluator

    tr, rec, X, rng = _model(K, U=150, I=389)  # n_items not a multiple of 128
    gt = _ground_truth(rng, *X.shape)
    cutoffs = [3, 10, 100] if K != 512 else [7, 200]
    _assert_same(ShardedEvaluator.from_global(tr, gt).get_scores(tr, cutoffs),
                 Evaluator(gt).get_scores(rec, cutoffs))


def test_masked_interactions_and_unsorted_ground_truth(m128):
    from irspack_b200 import Evaluator
    from irspack_b200.dist import ShardedEvaluator

    tr, rec, X, rng = m128
    U, I = X.shape
    mask = sps.csr_matrix((rng.random((U, I)) < 0.1).astype(np.float32))
    mask[5, 9] = 0.0            # stored zero in the mask: not masked (scipy's .nonzero())
    mask[4, :] = 1.0            # every item masked
    gt = _ground_truth(rng, U, I).tocoo()
    order = rng.permutation(gt.nnz)  # unsorted rows, and a stored zero that IS ground truth
    gt = sps.csr_matrix((np.r_[gt.data[order], 0.0], (np.r_[gt.row[order], 1], np.r_[gt.col[order], 17])),
                        shape=(U, I))
    gt.has_sorted_indices = False
    for cutoffs in ([1, 10, 50], [300]):
        want = Evaluator(gt, masked_interactions=mask).get_scores(rec, cutoffs)
        got = ShardedEvaluator.from_global(tr, gt, masked_interactions=mask).get_scores(tr, cutoffs)
        _assert_same(got, want)


def test_device_ground_truth(m128):
    import torch

    from irspack_b200 import Evaluator
    from irspack_b200.dist import ShardedEvaluator

    tr, rec, X, rng = m128
    gt = _ground_truth(rng, *X.shape)
    trip = tuple(torch.from_numpy(np.asarray(a)).cuda() for a in (gt.indptr.astype(np.int64),
                                                                  gt.indices.astype(np.int32),
                                                                  gt.data.astype(np.float32)))
    _assert_same(ShardedEvaluator(tr, trip).get_scores(tr, [5, 20]), Evaluator(gt).get_scores(rec, [5, 20]))


def test_allow_lists(m128):
    from irspack_b200 import Evaluator
    from irspack_b200.dist import ShardedEvaluator

    tr, rec, X, rng = m128
    U, I = X.shape
    gt = _ground_truth(rng, U, I)
    shared = sorted(rng.choice(I, 120, replace=False).tolist())
    per_user = [sorted(rng.choice(I, int(rng.integers(0, 60)), replace=False).tolist()) for _ in range(U)]
    for kw in ({"recommendable_items": shared}, {"per_user_recommendable_items": per_user}):
        want = Evaluator(gt, **kw).get_scores(rec, [5, 20, 128])
        sev = ShardedEvaluator.from_global(tr, gt, **kw)
        _assert_same(sev.get_scores(tr, [5, 20, 128]), want)
        with pytest.raises(NotImplementedError):
            sev.get_scores(tr, [150])


def test_reference_evaluator_on_the_same_scores(m128):
    import oracle
    from irspack_b200.dist import ShardedEvaluator

    if oracle.build_ref() is None:
        pytest.skip("oracle/_ref is not built and /root/reference is absent")
    tr, rec, X, rng = m128
    U, I = X.shape
    gt = _ground_truth(rng, U, I)
    gt.eliminate_zeros()
    scores = tr.user.astype(np.float64) @ tr.item.astype(np.float64).T
    Xm = X.copy()
    Xm.eliminate_zeros()
    scores[Xm.nonzero()] = -np.inf
    for cutoff in (1, 10, 37):
        want = oracle.ref_evaluator_metrics(scores, gt, cutoff)
        got = ShardedEvaluator.from_global(tr, gt, cutoff=cutoff).get_score(tr)
        for k in KEYS:
            assert got[k] == pytest.approx(want[k], rel=1e-12, abs=1e-12), (cutoff, k, got[k], want[k])


def test_rejections_match_evaluator(m128):
    from irspack_b200 import Evaluator
    from irspack_b200.dist import ShardedEvaluator

    tr, rec, X, rng = m128
    U, I = X.shape
    gt = _ground_truth(rng, U, I)
    ev, sev = Evaluator(gt), ShardedEvaluator.from_global(tr, gt)
    for cutoffs in ([0], [I + 1], [1025]):
        with pytest.raises(ValueError) as want:
            ev.get_scores(rec, cutoffs)
        with pytest.raises(ValueError) as got:
            sev.get_scores(tr, cutoffs)
        assert str(got.value) == str(want.value)
    with pytest.raises(ValueError, match="different n_items"):
        ShardedEvaluator(tr, sps.csr_matrix((U, I + 1)))
    with pytest.raises(ValueError, match="user rows"):
        ShardedEvaluator(tr, sps.csr_matrix((U - 1, I)))
    with pytest.raises(ValueError, match="inconsistent shapes"):
        ShardedEvaluator(tr, gt, per_user_recommendable_items=[[1]] * (U - 1))


def _device_diversity(hist):
    """Metrics.as_dict's (appeared_item, entropy, gini_index) of one histogram, by the device kernel."""
    import ctypes

    from irspack_b200 import _ials_core as core
    from irspack_b200._lib import check, lib
    from irspack_b200.dist import ShardedEvaluator, ShardedIALSTrainer

    I = hist.shape[0]
    X = sps.csr_matrix(([1.0], ([0], [0])), shape=(1, I), dtype=np.float32)
    tr = ShardedIALSTrainer.from_global(core.IALSModelConfigBuilder().set_K(32).build(), X, rank=0, world=1)
    sev = ShardedEvaluator(tr, sps.csr_matrix((1, I)))
    h = sev._set_for(tr, (1,))
    _, _, view = sev._views(h)
    view.copy_(__import__("torch").from_numpy(hist.astype(np.int64)))
    out = np.empty(3, np.float64)
    check(lib.ials_eval_set_diversity(h, ctypes.c_void_p(0), out.ctypes.data_as(ctypes.c_void_p)))
    return tuple(out)


@pytest.mark.parametrize("case", ["zeros", "single", "equal", "ties_2m", "skewed"])
def test_diversity_kernel_matches_as_dict(case):
    from irspack_b200.evaluation import Metrics

    rng = np.random.default_rng(3)
    hist = {"zeros": lambda: np.zeros(1000, np.int64),
            "single": lambda: np.eye(1, 777, 300, dtype=np.int64)[0] * 5,
            "equal": lambda: np.full(4096, 7, np.int64),
            "ties_2m": lambda: rng.integers(0, 4, size=2_000_000),
            "skewed": lambda: (rng.pareto(1.2, size=50_000) * 10).astype(np.int64)}[case]()
    got = _device_diversity(hist)
    want = Metrics.diversity(hist)
    for a, b in zip(got, want):
        assert a == pytest.approx(b, rel=1e-12, abs=1e-300), (case, got, want)
