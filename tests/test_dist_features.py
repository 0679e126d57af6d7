"""Feature-aware iALS and compute_loss on the row-sharded trainer (irspack_b200/dist.py).

1, 2 and 3 gloo ranks on one device (CUDA-IPC peer replicas exactly as on several devices) must
reproduce the single-process ``IALSTrainer(cfg, X, user_feature, item_feature)`` epoch by epoch:
factors, feature weights and the loss.  Every rank must hold the same replicas and weights, and a
rejected epoch must raise the single trainer's exception on every rank without touching the model.
The workers run under a bounded join: a rank left blocked in a collective fails the test."""
import os
import socket
import sys
import time

import numpy as np
import pytest
import scipy.sparse as sps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TIMEOUT_S = 600


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _spawn(fn, world, *args):
    """Run fn(rank, world, port, *args) on `world` processes; kill them all and fail on timeout."""
    import torch.multiprocessing as mp

    ctx = mp.start_processes(fn, args=(world, _free_port()) + args, nprocs=world, join=False,
                             start_method="spawn")
    deadline = time.monotonic() + TIMEOUT_S
    while not ctx.join(timeout=5):  # raises when a worker failed (and terminates the others)
        if time.monotonic() > deadline:
            for p in ctx.processes:
                if p.is_alive():
                    p.kill()
            for p in ctx.processes:
                p.join()
            pytest.fail(f"sharded workers did not finish within {TIMEOUT_S} s (a rank blocked in a collective?)")


def _init(rank, world, port, backend="gloo"):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist

    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    else:
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)


def _problem(seed, U=400, I=260, layout="user_csr"):
    """Interactions with a few empty users, user / item features of which one side is CSR and the
    other dense ("user_csr": 6 sparse user columns, 5 dense item columns; "item_csr": a dense user
    side with 0 columns, 7 sparse item columns)."""
    rng = np.random.default_rng(seed)
    X = sps.random(U, I, density=0.06, random_state=seed, format="csr", dtype=np.float32)
    X.data[:] = rng.choice([0.5, 1.0, 2.0, 3.0], size=X.nnz).astype(np.float32)
    X = sps.csr_matrix(X.toarray() * (rng.random((U, 1)) > 0.04))
    X.sort_indices()

    def feats(n, f):
        return (rng.standard_normal((n, f)) * (rng.random((n, f)) < 0.6)).astype(np.float32)

    if layout == "user_csr":
        return X, sps.csr_matrix(feats(U, 6)), feats(I, 5)
    return X, np.zeros((U, 0), np.float32), sps.csr_matrix(feats(I, 7))


def _config(core, K, warmup, loss="IALSPP", alpha0=0.1, reg=0.05, nu=1.0):
    return (core.IALSModelConfigBuilder().set_K(K).set_alpha0(alpha0).set_reg(reg).set_nu(nu)
            .set_loss_type(getattr(core.LossType, loss)).set_lambda_user_feature(0.3)
            .set_lambda_item_feature(0.2).set_feature_warmup_epochs(warmup).build())


def _state(t):
    return [t.user, t.item, t.user_feature_weight, t.item_feature_weight]


def _same_on_every_rank(arrays):
    import torch
    import torch.distributed as dist

    t = torch.from_numpy(np.concatenate([np.asarray(a, np.float64).ravel() for a in arrays]))
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return torch.equal(lo, hi)


def _close(a, b, tol):
    return np.abs(a - b).max(initial=0.0) <= tol * (np.abs(b).max(initial=0.0) + 1e-30)


def _worker_epochs(rank, world, port, solver, K, warmup, loss, layout):
    _init(rank, world, port)
    import torch
    import torch.distributed as dist

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer
    from irspack_b200.synth import init_factors

    X, uf, itf = _problem(K + world, layout=layout)
    U, I = X.shape
    cfg = _config(core, K, warmup, loss)
    sc = core.IALSSolverConfigBuilder().set_solver_type(getattr(core.SolverType, solver)).build()
    rng = np.random.default_rng(1)
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    w0 = [(rng.standard_normal((F.shape[1], K)) * 0.05).astype(np.float32) for F in (uf, itf)]

    tr = ShardedIALSTrainer.from_global(cfg, X, user_feature=uf, item_feature=itf)
    tr.user, tr.item = u0, i0
    tr.user_feature_weight, tr.item_feature_weight = w0
    single = core.IALSTrainer(cfg, X, uf, itf)
    single.user, single.item = u0, i0
    single.user_feature_weight, single.item_feature_weight = w0
    dist.barrier()
    for epoch in range(4):
        tr.step(sc)
        single.step(sc)
        got, want = _state(tr), _state(single)
        for a, b, what in zip(got, want, ("user", "item", "user weight", "item weight")):
            assert a.shape == b.shape, (what, a.shape, b.shape)
            assert _close(a, b, 1e-4), (epoch, what, np.abs(a - b).max(), np.abs(b).max())
        for w, w_init in zip(got[2:], w0):  # the feature path ran exactly from the warm-up on
            assert np.array_equal(w, w_init) == (epoch < warmup or w.size == 0), (epoch, w.size)
        assert _same_on_every_rank(got), f"replicas or weights diverged after epoch {epoch}"

    # the loss: the same float on every rank, equal to the single trainer's on the same model
    loss_sh = tr.compute_loss(sc)
    assert _same_on_every_rank([np.array([loss_sh])])
    ref = core.IALSTrainer(cfg, X, uf, itf)
    ref.user, ref.item = got[0], got[1]
    ref.user_feature_weight, ref.item_feature_weight = got[2], got[3]
    assert loss_sh == pytest.approx(ref.compute_loss(sc), rel=1e-6)
    plain = ShardedIALSTrainer.from_global(cfg, X)  # and without features
    plain.user, plain.item = got[0], got[1]
    dist.barrier()
    plain_ref = core.IALSTrainer(cfg, X)
    plain_ref.user, plain_ref.item = got[0], got[1]
    loss_plain = plain.compute_loss(sc)
    assert _same_on_every_rank([np.array([loss_plain])])
    assert loss_plain == pytest.approx(plain_ref.compute_loss(sc), rel=1e-6)
    assert loss_plain != loss_sh

    # step_io on host-resident shards == set + step + get
    saved = _state(tr)
    tr.step(sc)
    want = _state(tr)
    tr.user, tr.item = saved[0], saved[1]
    tr.user_feature_weight, tr.item_feature_weight = saved[2], saved[3]
    dist.barrier()
    (ub, ue), (ib, ie) = tr.user_range, tr.item_range
    hu = torch.from_numpy(saved[0][ub:ue].copy()).pin_memory()
    hi = torch.from_numpy(saved[1][ib:ie].copy()).pin_memory()
    tr.step_io(sc, hu, hi)
    got = _state(tr)
    # bit for bit with 128-column rows; the SIMT Gram of wider rows and the refit's F^T sums add with
    # atomics, whose last bits vary from run to run
    same = np.array_equal if K <= 128 else (lambda a, b: _close(a, b, 1e-5))
    assert same(hu.numpy(), want[0][ub:ue]) and same(hi.numpy(), want[1][ib:ie])
    assert same(got[0], want[0]) and same(got[1], want[1])
    for a, b in zip(got[2:], want[2:]):
        assert _close(a, b, 1e-5)
    assert _same_on_every_rank(got)
    dist.barrier()
    del tr, plain
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("world,solver,K,warmup,loss,layout", [
    (1, "CG", 128, 0, "IALSPP", "user_csr"),
    (2, "CG", 200, 2, "ORIGINAL", "item_csr"),
    (3, "CG", 128, 2, "IALSPP", "item_csr"),
    (2, "CHOLESKY", 64, 0, "ORIGINAL", "user_csr"),
    (3, "CHOLESKY", 256, 2, "IALSPP", "user_csr"),
    (1, "CHOLESKY", 256, 0, "ORIGINAL", "item_csr"),
])
def test_sharded_feature_epochs_match_single_process(world, solver, K, warmup, loss, layout):
    _spawn(_worker_epochs, world, solver, K, warmup, loss, layout)


def _expect_rejection(tr, call, single_call, dist):
    """call() must raise what single_call() raises, on every rank, and leave the model untouched."""
    before = _state(tr)
    with pytest.raises(Exception) as want:
        single_call()
    with pytest.raises(type(want.value)) as got:
        call()
    assert str(got.value) == str(want.value), (str(got.value), str(want.value))
    dist.barrier()
    after = _state(tr)
    for a, b in zip(after, before):
        assert np.array_equal(a, b)


def _worker_rejections(rank, world, port):
    _init(rank, world, port)
    import torch
    import torch.distributed as dist

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer, balanced_bounds
    from irspack_b200.synth import init_factors

    X, uf, itf = _problem(5)
    U, I = X.shape
    K = 32
    cfg = _config(core, K, 0)
    cg = core.IALSSolverConfigBuilder().build()
    tr = ShardedIALSTrainer.from_global(cfg, X, user_feature=uf, item_feature=itf)
    single = core.IALSTrainer(cfg, X, uf, itf)
    tr.user, tr.item = init_factors(U, K, 1), init_factors(I, K, 2)
    single.user, single.item = tr.user, tr.item
    tr.step(cg)
    single.step(cg)

    ialspp = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.IALSPP).build()
    _expect_rejection(tr, lambda: tr.step(ialspp), lambda: single.step(ialspp), dist)
    good = tr.user_feature_weight
    bad = np.zeros((good.shape[0] + 1, K), np.float32)
    tr.user_feature_weight = bad
    single.user_feature_weight = bad
    _expect_rejection(tr, lambda: tr.step(cg), lambda: single.step(cg), dist)
    _expect_rejection(tr, lambda: tr.compute_loss(cg), lambda: single.compute_loss(cg), dist)
    hu = torch.zeros((tr.user_range[1] - tr.user_range[0], K)).pin_memory()
    hi = torch.zeros((tr.item_range[1] - tr.item_range[0], K)).pin_memory()
    _expect_rejection(tr, lambda: tr.step_io(cg, hu, hi), lambda: single.step(cg), dist)
    tr.user_feature_weight = good
    tr.step(cg)  # the trainer is still usable
    del tr

    # alpha0 = 0 and a vanishing regulariser: an empty user row in ONE rank's shard (the last one)
    # must stop the epoch on every rank
    Xf = X.tolil()
    for u in range(U):  # every other row and column has an interaction
        if Xf.rows[u] == []:
            Xf[u, u % I] = 1.0
    for i in np.flatnonzero(np.asarray((Xf.tocsr() != 0).sum(axis=0)).ravel() == 0):
        Xf[int(i) % U, int(i)] = 1.0
    Xf = Xf.tocsr()
    victim = int(balanced_bounds(np.diff(Xf.indptr) + 1, world)[world - 1])
    Xf[victim] = 0
    Xf.eliminate_zeros()
    ub = balanced_bounds(np.diff(Xf.indptr) + 1, world)
    owners = [r for r in range(world) if ub[r] <= victim < ub[r + 1]]
    assert len(owners) == 1 and np.count_nonzero(np.diff(Xf.indptr) == 0) == 1
    cfg0 = _config(core, K, 0, alpha0=0.0, reg=0.0)
    tr = ShardedIALSTrainer.from_global(cfg0, Xf, user_feature=uf, item_feature=itf)
    single = core.IALSTrainer(cfg0, Xf, uf, itf)
    tr.user, tr.item = init_factors(U, K, 1), init_factors(I, K, 2)
    dist.barrier()
    _expect_rejection(tr, lambda: tr.step(cg), lambda: single.step(cg), dist)
    assert "not uniquely defined" in str(pytest.raises(ValueError, single.step, cg).value)
    dist.barrier()
    del tr
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 3])
def test_sharded_feature_rejections_raise_on_every_rank(world):
    _spawn(_worker_rejections, world)


# ---------------------------------------------------------------------------------------------
# one rank per GPU, NCCL, peer stores over NVLink: the feature-aware twin of test_dist.py's
# test_one_rank_per_device_nccl_matches_single_process.  Skipped with fewer than two GPUs.


def _worker_multi_device(rank, world, port, out_path):
    _init(rank, world, port, backend="nccl")
    import torch
    import torch.distributed as dist

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer
    from irspack_b200.synth import init_factors, synth_csr

    K, U, I = 128, 6000, 700
    X = synth_csr(U, I, 900000, seed=11)
    rng = np.random.default_rng(2)
    uf = sps.random(U, 20, density=0.2, random_state=3, format="csr", dtype=np.float32)
    itf = rng.standard_normal((I, 30)).astype(np.float32)
    cfg = _config(core, K, 1)
    sc = core.IALSSolverConfigBuilder().build()
    tr = ShardedIALSTrainer.from_global(cfg, X, user_feature=uf, item_feature=itf)
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    tr.user, tr.item = u0, i0
    dist.barrier()
    for _ in range(2):
        tr.step(sc)
    for _ in range(2):
        tr.step_async(sc)
    tr.sync()
    got = _state(tr)
    loss = tr.compute_loss(sc)
    if rank == 0:
        single = core.IALSTrainer(cfg, X, uf, itf)
        single.user, single.item = u0, i0
        for _ in range(4):
            single.step(sc)
        want = _state(single)
        np.savez(out_path, *got, *want, loss=loss, ref_loss=single.compute_loss(sc))
    t = torch.from_numpy(np.concatenate([a.ravel() for a in got] + [np.array([loss], np.float32)])).cuda()
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), "replicas or weights diverged"
    dist.barrier()
    del tr
    dist.destroy_process_group()


def _n_devices() -> int:
    try:
        import torch

        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_n_devices() < 2, reason="needs two GPUs")
def test_one_rank_per_device_nccl_feature_aware_matches_single_process(tmp_path):
    out = str(tmp_path / "res.npz")
    _spawn(_worker_multi_device, min(_n_devices(), 4), out)
    r = np.load(out)
    for j in range(4):
        a, b = r[f"arr_{j}"], r[f"arr_{j + 4}"]
        assert _close(a, b, 2e-4), j
    assert float(r["loss"]) == pytest.approx(float(r["ref_loss"]), rel=1e-4)
