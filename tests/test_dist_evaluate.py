"""ShardedEvaluator and ShardedIALSTrainer.learn_with_optimizer on 1, 2 and 3 gloo ranks on one device
(and a one-rank-per-device NCCL twin).  Every rank must return the identical dict, equal to the
single-process Evaluator on the gathered model; early stopping must pick the single loop's epoch and
leave every replica on every rank equal to the best epoch's factors.  Bounded joins: a rank left
blocked in a collective fails the test."""
import numpy as np
import pytest
import scipy.sparse as sps

from test_dist_features import _close, _init, _n_devices, _same_on_every_rank, _spawn

pytestmark = pytest.mark.gpu


def _dict_same_on_every_rank(d):
    import torch
    import torch.distributed as dist

    t = torch.tensor([d[k] for k in sorted(d)], dtype=torch.float64)
    if dist.get_backend() == "nccl":
        t = t.cuda()
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return torch.equal(lo, hi)


def _assert_same(got, want, tol=1e-12):
    assert got.keys() == want.keys()
    for k in want:
        if np.isnan(want[k]):
            assert np.isnan(got[k]), k
        else:
            assert got[k] == pytest.approx(want[k], rel=tol, abs=tol), (k, got[k], want[k])


def _problem(seed, U=360, I=301, density=0.05):
    rng = np.random.default_rng(seed)
    X = sps.csr_matrix((rng.random((U, I)) < density).astype(np.float32))
    gt = sps.csr_matrix((rng.random((U, I)) < 0.03).astype(np.float32))
    return X, gt, rng


def _reference(X, u, it, K):
    """An IALSRecommender holding the factors (the single-process model)."""
    from irspack_b200 import IALSRecommender

    rec = IALSRecommender(X, n_components=K, alpha0=0.1, reg=0.05, train_epochs=1).learn()
    rec.trainer_as_ials.core_trainer.user = u
    rec.trainer_as_ials.core_trainer.item = it
    return rec


def _worker_metrics(rank, world, port, scenario):
    _init(rank, world, port)
    import torch.distributed as dist

    from irspack_b200 import Evaluator
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluator, ShardedIALSTrainer, balanced_bounds

    K = 64
    X, gt, rng = _problem(world)
    U, I = X.shape
    feats = {}
    if scenario == "features":
        feats = dict(user_feature=sps.random(U, 5, density=0.5, random_state=1, format="csr", dtype=np.float32),
                     item_feature=rng.standard_normal((I, 4)).astype(np.float32))
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.05).set_lambda_user_feature(0.3) \
        .set_lambda_item_feature(0.2).build()
    tr = ShardedIALSTrainer.from_global(cfg, X, **feats)
    ub, ue = tr.user_range
    if scenario == "empty_rank":  # the last rank's ground-truth rows are all empty
        gt = gt.tolil()
        gt[int(balanced_bounds(np.diff(X.indptr) + 1, world)[world - 1]):] = 0
        gt = sps.csr_matrix(gt)
    rng_f = np.random.default_rng(5)
    tr.user = rng_f.integers(-2, 3, size=(U, K)).astype(np.float32)
    tr.item = rng_f.integers(-2, 3, size=(I, K)).astype(np.float32)
    if scenario == "features":
        sc = core.IALSSolverConfigBuilder().build()
        tr.step(sc)  # a real feature-aware epoch; then the gathered factors are the model
    dist.barrier()
    kw = {}
    if scenario == "per_user":
        lists = [sorted(np.random.default_rng(u).choice(I, 1 + u % 40, replace=False).tolist()) for u in range(U)]
        kw = {"per_user_recommendable_items": lists}
    cutoffs = [1, 5, 20] if scenario == "per_user" else [1, 5, 20, 200]
    sev = ShardedEvaluator.from_global(tr, gt, **kw)
    got = sev.get_scores(tr, cutoffs)
    assert _dict_same_on_every_rank(got)
    assert got == sev.get_scores(tr, cutoffs)  # two passes, bit-identical
    want = Evaluator(gt, **kw).get_scores(_reference(X, tr.user, tr.item, K), cutoffs)
    _assert_same(got, want)
    if scenario == "per_user":  # the union over every rank's lists, not this rank's
        assert sev._ev.n_recommendable_items == len({i for x in kw["per_user_recommendable_items"] for i in x})
    dist.barrier()
    del sev, tr
    dist.destroy_process_group()


@pytest.mark.parametrize("world,scenario", [
    (1, "plain"), (2, "plain"), (3, "plain"), (2, "empty_rank"), (3, "per_user"), (2, "features"),
])
def test_every_rank_returns_the_gathered_evaluator_dict(world, scenario):
    _spawn(_worker_metrics, world, scenario)


def _worker_bad_shape(rank, world, port):
    _init(rank, world, port)
    import torch.distributed as dist

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluator, ShardedIALSTrainer

    X, gt, _ = _problem(9)
    tr = ShardedIALSTrainer.from_global(core.IALSModelConfigBuilder().set_K(32).build(), X)
    ub, ue = tr.user_range
    mine = sps.csr_matrix(gt)[ub:ue]
    if rank == world - 1:
        mine = mine[:-1]  # one row short on one rank only
    with pytest.raises((ValueError, RuntimeError)) as e:
        ShardedEvaluator(tr, mine)
    assert ("user rows" in str(e.value)) == (rank == world - 1), str(e.value)
    sev = ShardedEvaluator.from_global(tr, gt)  # the collectives are still in step
    assert _dict_same_on_every_rank(sev.get_score(tr))
    dist.barrier()
    del sev, tr
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_wrong_ground_truth_shape_raises_on_every_rank(world):
    _spawn(_worker_bad_shape, world)


def _early_stop_problem():
    from irspack_b200.synth import init_factors

    # interactions drawn from a planted rank-3 preference, split into training and held-out entries:
    # from a random start, one CG step per epoch and a small regulariser, the held-out ndcg rises over
    # the first checks and falls once the 32 factors fit the training noise
    rng = np.random.default_rng(17)
    U, I, K = 500, 220, 32
    pref = rng.standard_normal((U, 3)) @ rng.standard_normal((3, I))
    p = 1.0 / (1.0 + np.exp(-(pref - 2.5)))
    full = rng.random((U, I)) < p
    test = rng.random((U, I)) < 0.2
    X = sps.csr_matrix((full & ~test).astype(np.float32))
    held = sps.csr_matrix((full & test).astype(np.float32))
    return X, held, init_factors(U, K, 1), init_factors(I, K, 2), K


def _single_best_epoch(max_epoch, validate_epoch, degradation):
    """The loop of IALSRecommender.learn_with_optimizer on the single trainer, with the same start:
    (best epoch, its factors, the validation scores)."""
    from irspack_b200 import Evaluator
    from irspack_b200 import _ials_core as core

    X, held, u0, i0, K = _early_stop_problem()
    rec = _reference(X, u0, i0, K)
    t = rec.trainer_as_ials.core_trainer
    cfg_reg = 1e-3
    single = core.IALSTrainer(core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.5).set_reg(cfg_reg).build(), X)
    single.user, single.item = u0, i0
    sc = core.IALSSolverConfigBuilder().set_max_cg_steps(1).build()
    ev = Evaluator(held, cutoff=10)
    best, best_epoch, best_f, n_deg, scores = -np.inf, 0, None, 0, []
    for epoch in range(max_epoch):
        single.step(sc)
        if (epoch + 1) % validate_epoch:
            continue
        t.user, t.item = single.user, single.item
        s = ev.get_target_score(rec)
        scores.append(s)
        if s > best:
            best, best_epoch, best_f, n_deg = s, epoch + 1, (single.user, single.item), 0
        else:
            n_deg += 1
            if n_deg >= degradation:
                break
    return best_epoch, best_f, scores, cfg_reg


def _worker_early_stop(rank, world, port, max_epoch, validate_epoch, degradation, out_path):
    _init(rank, world, port)
    import torch.distributed as dist

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluator, ShardedIALSTrainer

    X, held, u0, i0, K = _early_stop_problem()
    want_epoch, want_f, scores, reg = _single_best_epoch(max_epoch, validate_epoch, degradation)
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.5).set_reg(reg).build()
    sc = core.IALSSolverConfigBuilder().set_max_cg_steps(1).build()
    tr = ShardedIALSTrainer.from_global(cfg, X)
    tr.user, tr.item = u0, i0
    dist.barrier()
    sev = ShardedEvaluator.from_global(tr, held, cutoff=10)
    got = tr.learn_with_optimizer(sc, sev, max_epoch=max_epoch, validate_epoch=validate_epoch,
                                  score_degradation_max=degradation)
    assert got == want_epoch, (got, want_epoch, scores)
    assert 0 < want_epoch < max_epoch  # the loop stopped early, past its first check
    u, it = tr.user, tr.item
    assert _same_on_every_rank([u, it])
    assert _close(u, want_f[0], 1e-4) and _close(it, want_f[1], 1e-4)
    # evaluator=None: every epoch, and the model is the last one
    tr2 = ShardedIALSTrainer.from_global(cfg, X)
    tr2.user, tr2.item = u0, i0
    dist.barrier()
    assert tr2.learn_with_optimizer(sc, None, max_epoch=3) == 3
    single = core.IALSTrainer(cfg, X)
    single.user, single.item = u0, i0
    for _ in range(3):
        single.step(sc)
    assert _close(tr2.user, single.user, 1e-4) and _close(tr2.item, single.item, 1e-4)
    if rank == 0 and out_path:
        np.save(out_path, np.array(scores))
    dist.barrier()
    del sev, tr, tr2
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_early_stopping_picks_the_single_trainer_epoch(world, tmp_path):
    out = str(tmp_path / "scores.npy")
    _spawn(_worker_early_stop, world, 40, 2, 3, out)
    s = np.load(out)
    # the decisions are not near-ties: the validation scores differ clearly from one another
    gaps = np.abs(s[:, None] - s[None, :])[np.triu_indices(s.size, 1)]
    assert gaps.min() > 1e-4, s


def _worker_nccl(rank, world, port, out_path):
    _init(rank, world, port, backend="nccl")
    import torch.distributed as dist

    from irspack_b200 import Evaluator
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluator, ShardedIALSTrainer

    X, gt, rng = _problem(4, U=3000, I=900)
    K = 128
    tr = ShardedIALSTrainer.from_global(core.IALSModelConfigBuilder().set_K(K).build(), X)
    r = np.random.default_rng(2)
    tr.user = r.integers(-2, 3, size=X.shape[:1] + (K,)).astype(np.float32)
    tr.item = r.integers(-2, 3, size=(X.shape[1], K)).astype(np.float32)
    dist.barrier()
    got = ShardedEvaluator.from_global(tr, gt).get_scores(tr, [10, 100])
    assert _dict_same_on_every_rank(got)
    if rank == 0:
        want = Evaluator(gt).get_scores(_reference(X, tr.user, tr.item, K), [10, 100])
        _assert_same(got, want)
    dist.barrier()
    del tr
    dist.destroy_process_group()


@pytest.mark.skipif(_n_devices() < 2, reason="needs two GPUs")
def test_one_rank_per_device_nccl_matches_single_process(tmp_path):
    _spawn(_worker_nccl, min(_n_devices(), 4), str(tmp_path / "x"))
