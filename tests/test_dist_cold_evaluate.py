"""ShardedEvaluatorWithColdUser and ShardedIALSTrainer.transform_user / transform_item on 1, 2 and 3
gloo ranks on one device (and a one-rank-per-device NCCL twin).  Every rank must return the identical
dict, equal to the single-process EvaluatorWithColdUser on an IALSRecommender with the same factors,
from the same lists; the fold-in must equal IALSTrainer.transform_*; an evaluation between epochs must
not change the next epoch; early stopping on the cold score must pick the single loop's epoch.
Bounded joins: a rank left blocked in a collective fails the test."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sps

from test_dist_evaluate import _assert_same, _dict_same_on_every_rank
from test_dist_features import _close, _init, _n_devices, _same_on_every_rank, _spawn

pytestmark = pytest.mark.gpu

ALPHA0, REG, NU = 0.1, 0.05, 1.0
TOL_STEP = 2e-4  # one solve of the same rows with reordered float sums (test_gpu_feature_routes.py)


def _cold_problem(seed, U=360, I=301, C=150):
    """Training matrix, the cold users' input and ground truth (row 0 with two stored zeros, row 1
    empty, row 2 with a negative value, ground-truth rows 3..5 empty) and item factors."""
    rng = np.random.default_rng(seed)
    X = sps.csr_matrix((rng.random((U, I)) < 0.05).astype(np.float32))
    dense = (rng.random((C, I)) < 0.06).astype(np.float32) * rng.integers(1, 4, size=(C, I)).astype(np.float32)
    dense[0, :5] = 1.0
    dense[1] = 0.0
    Xc = sps.csr_matrix(dense)
    Xc.data[Xc.indptr[0]: Xc.indptr[0] + 2] = 0.0  # stored zeros: in the fold-in, not in the mask
    Xc.data[Xc.indptr[2]] = -0.5
    assert Xc.nnz == int((dense != 0).sum())
    gt = (rng.random((C, I)) < 0.04).astype(np.float32)
    gt[3:6] = 0.0
    item = (rng.standard_normal((I, 1)) * 0.3 + rng.standard_normal((I, 128)) * 0.2).astype(np.float32)
    return X, Xc, sps.csr_matrix(gt), item


def _configs(core, K, solver):
    st = core.SolverType[solver]
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(ALPHA0).set_reg(REG).set_nu(NU).build()
    # the prediction-time solver of ials.IALSTrainer: 5 CG steps, 7 iALS++ iterations
    sc = core.IALSSolverConfigBuilder().set_solver_type(st).set_max_cg_steps(5).set_ialspp_iteration(7) \
        .set_ialspp_subspace_dimension(64).build()
    return cfg, sc


def _reference(X, item, K, solver):
    """An IALSRecommender holding the item factors, with the same model and fold-in configuration."""
    from irspack_b200 import IALSRecommender

    rec = IALSRecommender(X, n_components=K, alpha0=ALPHA0, reg=REG, nu=NU, solver_type=solver,
                          ialspp_subspace_dimension=64, train_epochs=1).learn()
    rec.trainer_as_ials.core_trainer.item = item
    return rec


def _share(C, rank, world, empty_last):
    """Contiguous share of the C cold users; ``empty_last``: the last rank gets none."""
    from irspack_b200.dist import balanced_bounds

    b = balanced_bounds(np.ones(C), world - 1 if empty_last else world)
    b = np.concatenate([b, [C]]) if empty_last else b
    return int(b[rank]), int(b[rank + 1])


def _pass_lists(tr, sev, k):
    """The lists the cold pass ranks, one user at a time: with cutoffs 1..k the histogram of cutoff c
    minus that of cutoff c - 1 holds the user's c-th item (-1: the list ended, or the user has no
    ground truth: the metrics skip such users, evaluator.cpp:319-321)."""
    from irspack_b200._lib import check, lib

    h = sev._set_for(tr, tuple(range(1, k + 1)))
    stream = ctypes.c_void_p(tr._core._stream_of(tr._device))
    out = np.full((sev._ev.n_users, k), -1, dtype=np.int64)
    for r in range(sev._ev.n_users):
        check(lib.ials_eval_set_reset(h, stream))
        tr._use_current_stream()
        check(lib.ials_trainer_evaluate_cold(tr._handle, h, ctypes.byref(sev._sc), r, r + 1))
        hist = sev._views(h)[2].cpu().numpy().reshape(k, -1)
        prev = np.zeros(hist.shape[1], dtype=np.int64)
        for c in range(k):
            nz = np.flatnonzero(hist[c] - prev)
            assert nz.size <= 1
            if nz.size:
                out[r, c] = nz[0]
            prev = hist[c]
    return out


def _worker_cold(rank, world, port):
    _init(rank, world, port)
    import torch.distributed as dist

    from irspack_b200 import EvaluatorWithColdUser
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluatorWithColdUser, ShardedIALSTrainer

    X, Xc, gt, item = _cold_problem(world)
    U, I = X.shape
    C = Xc.shape[0]
    lo, hi = _share(C, rank, world, empty_last=world == 3)
    rng = np.random.default_rng(3)
    mask = sps.csr_matrix((rng.random((C, I)) < 0.1).astype(np.float32))
    lists = [sorted(np.random.default_rng(u).choice(I, 5 + u % 60, replace=False).tolist()) for u in range(C)]
    shared = sorted(rng.choice(I, 120, replace=False).tolist())
    variants = [{}, {"masked_interactions": mask}, {"recommendable_items": shared},
                {"per_user_recommendable_items": lists}]

    def mine(kw):
        out = dict(kw)
        if "masked_interactions" in kw:
            out["masked_interactions"] = mask[lo:hi]
        if "per_user_recommendable_items" in kw:
            out["per_user_recommendable_items"] = lists[lo:hi]
        return out

    for solver in ("CG", "IALSPP"):
        K = 128
        cfg, sc = _configs(core, K, solver)
        tr = ShardedIALSTrainer.from_global(cfg, X)
        tr.item = item
        dist.barrier()
        rec = _reference(X, item, K, solver)
        for kw in variants:
            cutoffs = [1, 5, 20]
            sev = ShardedEvaluatorWithColdUser(tr, Xc[lo:hi], gt[lo:hi], sc, recall_with_cutoff=True, **mine(kw))
            got = sev.get_scores(tr, cutoffs)
            assert _dict_same_on_every_rank(got)
            assert got == sev.get_scores(tr, cutoffs)  # two passes, bit-identical
            want = EvaluatorWithColdUser(Xc, gt, recall_with_cutoff=True, **kw).get_scores(rec, cutoffs)
            _assert_same(got, want)
            # the lists behind the dicts: this rank's users, ranked by the pass and by the recommender
            m = mine(kw)
            allowed = sev._ev._allowed_for(0, hi - lo, canonical=True)
            want_idx, _ = rec.recommend_cold_block(Xc[lo:hi], 10, mask=m.get("masked_interactions", "input"),
                                                   allowed=allowed)
            valid = np.diff(gt[lo:hi].indptr) > 0
            assert valid.sum() >= (hi - lo) // 2
            assert np.array_equal(_pass_lists(tr, sev, 10)[valid], want_idx[valid]), (solver, sorted(kw))
            del sev
        dist.barrier()
        del tr

    # the fold-in itself: bit for bit against the single trainer with the same factors
    for solver, K in (("CG", 128), ("CG", 200), ("CHOLESKY", 64)):
        cfg, sc = _configs(core, K, solver)
        tr = ShardedIALSTrainer.from_global(cfg, X)
        r = np.random.default_rng(K)
        tr.user = (r.standard_normal((U, K)) * 0.2).astype(np.float32)
        tr.item = (r.standard_normal((I, K)) * 0.2).astype(np.float32)
        dist.barrier()
        single = core.IALSTrainer(cfg, X)
        single.user, single.item = tr.user, tr.item
        # 128-column rows: the same deterministic kernels (tensor-core Gram included) on both sides; wider
        # rows form P with the SIMT Gram, whose float sums may be added in another order
        same = (lambda a, b: np.array_equal(a, b)) if K <= 128 else (lambda a, b: _close(a, b, TOL_STEP))
        got = tr.transform_user(Xc[lo:hi], sc)
        assert got.shape == (hi - lo, K)
        assert same(got, single.transform_user(Xc[lo:hi], sc)), (solver, K)
        Xi = sps.csr_matrix((r.random((U, 7)) < 0.1).astype(np.float32))
        assert same(tr.transform_item(Xi, sc), single.transform_item(Xi, sc)), (solver, K)
        dist.barrier()
        del tr
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2, 3])
def test_every_rank_returns_the_single_process_cold_dict(world):
    _spawn(_worker_cold, world)


def _expect(call, mine_fails, match, exc=ValueError):
    with pytest.raises((exc, RuntimeError)) as e:
        call()
    if mine_fails:
        assert isinstance(e.value, exc) and match in str(e.value), str(e.value)
    else:
        assert "peer rank failed" in str(e.value), str(e.value)


def _worker_rejections(rank, world, port):
    _init(rank, world, port)
    import torch.distributed as dist

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluatorWithColdUser, ShardedIALSTrainer

    X, Xc, gt, item = _cold_problem(11)
    C, I = Xc.shape
    lo, hi = _share(C, rank, world, empty_last=False)
    cfg, sc = _configs(core, 32, "CG")
    tr = ShardedIALSTrainer.from_global(cfg, X)
    last = rank == world - 1
    wide = sps.hstack([Xc[lo:hi], sps.csr_matrix((hi - lo, 1))]).tocsr() if last else Xc[lo:hi]
    _expect(lambda: ShardedEvaluatorWithColdUser(tr, wide, gt[lo:hi], sc), last, "training items")
    short = gt[lo:hi - 1] if last else gt[lo:hi]
    _expect(lambda: ShardedEvaluatorWithColdUser(tr, Xc[lo:hi], short, sc), last, "same number of rows")
    _expect(lambda: ShardedEvaluatorWithColdUser(tr, Xc[lo:hi], gt[lo:hi], "CG" if last else sc), last,
            "IALSSolverConfig", TypeError)
    sev = ShardedEvaluatorWithColdUser(tr, Xc[lo:hi], gt[lo:hi], sc, cutoff=0)
    with pytest.raises(ValueError, match="greather than 0"):
        sev.get_score(tr)
    with pytest.raises(ValueError, match="exeeed"):
        sev.get_scores(tr, [5, I + 1])
    allow = ShardedEvaluatorWithColdUser(tr, Xc[lo:hi], gt[lo:hi], sc, recommendable_items=list(range(0, I, 2)))
    with pytest.raises(NotImplementedError):
        allow.get_scores(tr, [10, 129])
    assert _dict_same_on_every_rank(allow.get_scores(tr, [10, 128]))  # the collectives are still in step
    # cutoff 1025 needs a catalogue past the device selection's 1024 keys
    rng = np.random.default_rng(1)
    X2 = sps.csr_matrix((rng.random((40, 1100)) < 0.02).astype(np.float32))
    C2 = sps.csr_matrix((rng.random((9, 1100)) < 0.02).astype(np.float32))
    tr2 = ShardedIALSTrainer.from_global(cfg, X2)
    sev2 = ShardedEvaluatorWithColdUser.from_global(tr2, C2, C2, sc)
    with pytest.raises(ValueError, match="1024"):
        sev2.get_scores(tr2, [10, 1025])
    assert _dict_same_on_every_rank(sev2.get_scores(tr2, [10, 1024]))
    dist.barrier()
    del sev, allow, sev2, tr, tr2
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_cold_rejections_raise_on_every_rank(world):
    _spawn(_worker_rejections, world)


def _early_stop_problem():
    """Interactions drawn from a planted rank-3 preference, split into training and held-out entries; the
    last 300 users are cold (input: their training entries, ground truth: their held-out entries).  From
    the seeded start, one CG step per epoch, checked every 4 epochs, the cold ndcg@10 falls from its first
    check on, by more than 5e-3 per check: the loop keeps epoch 4 and stops after epoch 16."""
    rng = np.random.default_rng(9)
    U, I, n_cold, K = 1000, 220, 300, 32
    pref = rng.standard_normal((U, 3)) @ rng.standard_normal((3, I))
    p = 1.0 / (1.0 + np.exp(-(pref - 2.5)))
    full = rng.random((U, I)) < p
    test = rng.random((U, I)) < 0.2
    X = sps.csr_matrix((full & ~test).astype(np.float32))
    held = sps.csr_matrix((full & test).astype(np.float32))
    return sps.csr_matrix(X[:U - n_cold]), sps.csr_matrix(X[U - n_cold:]), sps.csr_matrix(held[U - n_cold:]), K


def _worker_epochs(rank, world, port, max_epoch, validate_epoch, degradation, out_path):
    _init(rank, world, port)
    import torch.distributed as dist

    from irspack_b200 import EvaluatorWithColdUser, IALSRecommender
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluatorWithColdUser, ShardedIALSTrainer

    X, Xc, held, K = _early_stop_problem()
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.5).set_reg(1e-3).set_nu(NU).set_init_stdev(0.1) \
        .set_random_seed(42).build()
    train_sc = core.IALSSolverConfigBuilder().set_max_cg_steps(1).build()
    pred_sc = core.IALSSolverConfigBuilder().set_max_cg_steps(5).set_ialspp_iteration(7).build()

    # an evaluation between two epochs leaves the second epoch bit-identical
    a, b = ShardedIALSTrainer.from_global(cfg, X), ShardedIALSTrainer.from_global(cfg, X)
    dist.barrier()
    sevs = [ShardedEvaluatorWithColdUser.from_global(a, Xc, held, s) for s in (
        pred_sc, core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP).build())]
    a.step(train_sc)
    for sev in sevs:
        sev.get_scores(a, [1, 10])
    a.step(train_sc)
    b.step(train_sc)
    b.step(train_sc)
    assert np.array_equal(a.user, b.user) and np.array_equal(a.item, b.item)
    del sevs, a, b

    # early stopping on the cold score: the epoch IALSRecommender.learn_with_optimizer picks
    scores = []

    class Recording(EvaluatorWithColdUser):
        def get_target_score(self, model):
            scores.append(super().get_target_score(model))
            return scores[-1]

    rec = IALSRecommender(X, n_components=K, alpha0=0.5, reg=1e-3, nu=NU, init_std=0.1, random_seed=42,
                          max_cg_steps=1)
    rec.learn_with_optimizer(Recording(Xc, held, cutoff=10), max_epoch=max_epoch, validate_epoch=validate_epoch,
                             score_degradation_max=degradation)
    want_epoch = rec.learnt_config["train_epochs"]
    want_u, want_i = rec.trainer_as_ials.core_trainer.user, rec.trainer_as_ials.core_trainer.item
    tr = ShardedIALSTrainer.from_global(cfg, X)
    dist.barrier()
    sev = ShardedEvaluatorWithColdUser.from_global(tr, Xc, held, pred_sc, cutoff=10)
    got = tr.learn_with_optimizer(train_sc, sev, max_epoch=max_epoch, validate_epoch=validate_epoch,
                                  score_degradation_max=degradation)
    assert got == want_epoch, (got, want_epoch, scores)
    u, it = tr.user, tr.item
    assert _same_on_every_rank([u, it])
    assert _close(u, want_u, 1e-4) and _close(it, want_i, 1e-4)
    if rank == 0 and out_path:
        np.save(out_path, np.array(scores + [want_epoch, max_epoch]))
    dist.barrier()
    del sev, tr
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_cold_early_stopping_picks_the_recommender_epoch(world, tmp_path):
    out = str(tmp_path / "scores.npy")
    _spawn(_worker_epochs, world, 40, 4, 3, out)
    s = np.load(out)
    scores, best = s[:-2], int(s[-2])
    assert 0 < best < 40 and scores.size < 10  # the loop stopped early
    # the decisions are not near-ties: the validation scores differ clearly from one another
    gaps = np.abs(scores[:, None] - scores[None, :])[np.triu_indices(scores.size, 1)]
    assert gaps.min() > 1e-4, scores


def _worker_nccl(rank, world, port):
    _init(rank, world, port, backend="nccl")
    import torch.distributed as dist

    from irspack_b200 import EvaluatorWithColdUser
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluatorWithColdUser, ShardedIALSTrainer

    X, Xc, gt, item = _cold_problem(4)
    cfg, sc = _configs(core, 128, "CG")
    tr = ShardedIALSTrainer.from_global(cfg, X)
    tr.item = item
    dist.barrier()
    got = ShardedEvaluatorWithColdUser.from_global(tr, Xc, gt, sc).get_scores(tr, [10, 100])
    assert _dict_same_on_every_rank(got)
    if rank == 0:
        _assert_same(got, EvaluatorWithColdUser(Xc, gt).get_scores(_reference(X, item, 128, "CG"), [10, 100]))
    dist.barrier()
    del tr
    dist.destroy_process_group()


@pytest.mark.skipif(_n_devices() < 2, reason="needs two GPUs")
def test_one_rank_per_device_nccl_cold_matches_single_process():
    _spawn(_worker_nccl, min(_n_devices(), 4))
