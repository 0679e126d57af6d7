"""Row-sharded multi-GPU path (irspack_b200/dist.py).

CPU (``-m "not gpu"``): the host logic -- nnz-balanced partitioning, the
collective that builds every rank's rows of X^T and the agreement of ranks on a
failure -- on world_size-2 and -3 ``gloo``.
GPU (``-m gpu``): two ranks on ONE device (gloo control plane, CUDA-IPC peer
replicas exactly as on two devices) must reproduce the single-process trainer.
The workers run under a bounded join: a rank left blocked in a collective fails the test.
"""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sps

from test_dist_features import _n_devices, _spawn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _init(rank, world, port):
    """gloo without selecting a CUDA device: the CPU workers must run on a machine without one."""
    import torch.distributed as dist

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _matrix(seed=3, U=300, I=170, nnz=6000):
    # (no irspack_b200 import on the CPU path of this helper: synth is pure numpy)
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, U, nnz)
    cols = (rng.pareto(1.2, nnz) * 7).astype(np.int64) % I  # skewed item popularity
    X = sps.csr_matrix((np.ones(nnz, np.float32), (rows, cols)), shape=(U, I))
    X.sum_duplicates()
    X.data = rng.integers(1, 5, X.nnz).astype(np.float32)
    X.sort_indices()
    return X


def _dist_module():
    """irspack_b200.dist without triggering the CUDA library load (host logic only)."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("_ials_dist_host", os.path.join(ROOT, "irspack_b200", "dist.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_balanced_bounds():
    d = _dist_module()
    w = np.array([5, 1, 1, 1, 1, 1, 10, 0, 0, 4], dtype=np.int64)
    b = d.balanced_bounds(w, 3)
    assert b[0] == 0 and b[-1] == len(w) and np.all(np.diff(b) >= 0)
    parts = [w[b[i]:b[i + 1]].sum() for i in range(3)]
    assert max(parts) <= w.sum() / 3 + w.max()
    assert list(d.balanced_bounds(np.zeros(0), 2)) == [0, 0, 0]
    assert list(d.balanced_bounds(np.ones(3), 1)) == [0, 3]
    big = d.balanced_bounds(np.ones(1000), 8)
    assert np.all(np.abs(np.diff(big) - 125) <= 1)


def _csr_to_torch(X):
    import torch

    return (torch.from_numpy(X.indptr.astype(np.int64)), torch.from_numpy(X.indices.astype(np.int32)),
            torch.from_numpy(X.data.astype(np.float32)))


def _worker_exchange(rank, world, port):
    """The collective on CPU tensors: every rank's rows of X^T equal scipy's."""
    _init(rank, world, port)
    import torch.distributed as dist

    d = _dist_module()
    X = _matrix()
    U, I = X.shape
    ub = d.balanced_bounds(np.diff(X.indptr) + 1, world)
    mine = X[ub[rank]:ub[rank + 1]]
    ip, ix, dt = _csr_to_torch(mine)
    ib = d.global_item_bounds(ix, I)
    assert np.array_equal(ib, d.balanced_bounds(np.bincount(X.indices, minlength=I) + 1, world))
    t_ip, t_ix, t_dt = d.exchange_transposed_shards(ip, ix, dt, int(ub[rank]), U, ib)
    want = sps.csr_matrix(X.T)[ib[rank]:ib[rank + 1]]
    want.sort_indices()
    assert np.array_equal(t_ip.numpy(), want.indptr)
    assert np.array_equal(t_ix.numpy(), want.indices)
    assert np.array_equal(t_dt.numpy(), want.data)
    dist.barrier()
    dist.destroy_process_group()


def test_exchange_transposed_shards_torch_gloo_world2():
    _spawn(_worker_exchange, 2)


def test_exchange_transposed_shards_torch_gloo_world3():
    _spawn(_worker_exchange, 3)


def test_exchange_transposed_shards_torch_single_process():
    d = _dist_module()
    X = _matrix(seed=8, U=120, I=90, nnz=2500)
    ip, ix, dt = _csr_to_torch(X)
    t_ip, t_ix, t_dt = d.exchange_transposed_shards(ip, ix, dt, 0, X.shape[0], [0, X.shape[1]])
    want = sps.csr_matrix(X.T)
    want.sort_indices()
    assert np.array_equal(t_ip.numpy(), want.indptr) and np.array_equal(t_ix.numpy(), want.indices)
    assert np.array_equal(t_dt.numpy(), want.data)


def _worker_agreement(rank, world, port):
    _init(rank, world, port)
    import torch.distributed as dist

    d = _dist_module()
    # one rank raises: it gets its own exception, every other rank a RuntimeError naming a peer
    for i, kind in enumerate((ValueError, TypeError, KeyError, RuntimeError, NotImplementedError)):
        culprit = i % world
        mine = kind(f"rank {rank} failed")
        with pytest.raises(Exception) as got:
            with d._agreement(None):
                if rank == culprit:
                    raise mine
        if rank == culprit:
            assert got.value is mine
        else:
            assert type(got.value) is RuntimeError and "peer rank failed" in str(got.value)
    # no rank raises: the piggybacked integers come back as their maximum over the ranks
    values = [rank, 10 * (world - 1 - rank), -rank]
    with d._agreement(None, values):
        pass
    assert values == [world - 1, 10 * (world - 1), 0]
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_agreement_raises_on_every_rank_gloo(world):
    _spawn(_worker_agreement, world)


def test_synth_user_block_device_is_a_well_formed_power_law_block():
    d = _dist_module()
    n_u, n_i, nnz = 2000, 700, 40000
    ip, ix, dt = d.synth_user_block_device(n_u, n_i, nnz, seed=5, device="cpu", item_seed=1)
    ip2, ix2, _ = d.synth_user_block_device(n_u, n_i, nnz, seed=5, device="cpu", item_seed=1)
    assert np.array_equal(ip.numpy(), ip2.numpy()) and np.array_equal(ix.numpy(), ix2.numpy())
    ip, ix = ip.numpy(), ix.numpy()
    assert ip[0] == 0 and ip[-1] == nnz == ix.size == dt.numel() and np.all(np.diff(ip) >= 0)
    assert ix.min() >= 0 and ix.max() < n_i
    X = sps.csr_matrix((dt.numpy(), ix, ip), shape=(n_u, n_i))
    assert X.has_canonical_format  # ascending, duplicate-free rows
    # another rank (other seed) shares the item popularity law: the same head items
    _, jx, _ = d.synth_user_block_device(n_u, n_i, nnz, seed=6, device="cpu", item_seed=1)
    top_a = set(np.argsort(-np.bincount(ix, minlength=n_i))[:20])
    top_b = set(np.argsort(-np.bincount(jx.numpy(), minlength=n_i))[:20])
    assert len(top_a & top_b) >= 12
    deg = np.sort(np.bincount(ix, minlength=n_i))[::-1]
    assert deg[0] > 20 * max(np.median(deg), 1)  # a head, not a uniform law
    with pytest.raises(ValueError):
        d.synth_user_block_device(3, 3, 10, seed=1, device="cpu")


# ---------------------------------------------------------------------------------------------


def _worker_gpu(rank, world, port, solver, out_path):
    _init(rank, world, port)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(0)
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer
    from irspack_b200.synth import init_factors, synth_csr

    K = 32 if solver == "CHOLESKY" else 128
    X = synth_csr(900, 500, 30000, seed=5, values="counts")
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.03).build()
    st = getattr(core.SolverType, solver)
    sc = core.IALSSolverConfigBuilder().set_solver_type(st).build()
    tr = ShardedIALSTrainer.from_global(cfg, X)
    u0, i0 = init_factors(900, K, 1), init_factors(500, K, 2)
    tr.user, tr.item = u0, i0
    dist.barrier()
    for _ in range(3):
        tr.step(sc)
    user, item = tr.user, tr.item
    if rank == 0:
        single = core.IALSTrainer(cfg, X)
        single.user, single.item = u0, i0
        for _ in range(3):
            single.step(sc)
        np.savez(out_path, user=user, item=item, ref_user=single.user, ref_item=single.item)
    # every rank's replica must hold the same thing
    t = torch.from_numpy(np.concatenate([user.ravel(), item.ravel()]))
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), "replicas diverged"
    dist.barrier()
    del tr
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("solver", ["CG", "CHOLESKY", "IALSPP"])
def test_two_ranks_one_device_match_single_process(tmp_path, solver):
    out = str(tmp_path / "res.npz")
    _spawn(_worker_gpu, 2, solver, out)
    r = np.load(out)
    # same kernels, same row arithmetic; only the Gram is summed in a different order, and three
    # epochs of unconverged CG amplify that rounding (TOL_STEP of test_gpu_parity.py is 2e-4)
    for a, b in ((r["user"], r["ref_user"]), (r["item"], r["ref_item"])):
        assert np.abs(a - b).max() <= 1e-4 * np.abs(b).max()


@pytest.mark.gpu
def test_get_factors_into_rejects_a_buffer_of_the_wrong_layout():
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer

    K = 32
    X = _matrix()
    tr = ShardedIALSTrainer.from_global(core.IALSModelConfigBuilder().set_K(K).build(), X, rank=0, world=1)
    for side, n in ((0, X.shape[0]), (1, X.shape[1])):
        for bad in (np.empty((n - 1, K), np.float32), np.empty((n, K + 1), np.float32),
                    np.empty((n, K), np.float64), np.empty((K, n), np.float32).T):
            with pytest.raises(ValueError):
                tr.get_factors_into(side, bad)
        out = np.empty((n, K), np.float32)
        tr.get_factors_into(side, out)
        assert np.array_equal(out, tr.user if side == 0 else tr.item)


# ---------------------------------------------------------------------------------------------
# real multi-device run: one rank per GPU, NCCL, peer stores over NVLink.  Skipped on boxes with
# fewer than two GPUs (the driver's `-m gpu` tier has one; `gpurun --gpus 2` runs it).


def _worker_multi_device(rank, world, port, out_path):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer
    from irspack_b200.synth import init_factors, synth_csr

    K, U, I = 128, 6000, 700
    X = synth_csr(U, I, 900000, seed=11)     # items average ~1300 neighbours: heavy + light rows
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.03).build()
    sc = core.IALSSolverConfigBuilder().build()
    tr = ShardedIALSTrainer.from_global(cfg, X)
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    tr.user, tr.item = u0, i0
    dist.barrier()
    for _ in range(2):
        tr.step(sc)
    for _ in range(3):                        # back-to-back epochs: the all-reduce is the only fence
        tr.step_async(sc)
    tr.sync()
    user, item = tr.user, tr.item
    if rank == 0:
        single = core.IALSTrainer(cfg, X)
        single.user, single.item = u0, i0
        for _ in range(5):
            single.step(sc)
        np.savez(out_path, user=user, item=item, ref_user=single.user, ref_item=single.item)
    t = torch.from_numpy(np.concatenate([user.ravel(), item.ravel()])).cuda()
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), "replicas diverged"
    dist.barrier()
    # own rows down from the host + NVLink push into every peer's replica, own rows back
    for side, n in ((0, U), (1, I)):
        b, e = tr.shard_range(side)
        rows = (np.arange((e - b) * K, dtype=np.float32).reshape(e - b, K) % 997.0) + 1000.0 * (rank + 1)
        tr.set_shard_rows(side, rows)
        tr.sync()  # stream sync + barrier: every rank's copies have landed everywhere
        ranges = [None] * world
        dist.all_gather_object(ranges, (b, e))
        full = tr.user if side == 0 else tr.item
        assert full.shape == (n, K)
        for r, (rb, re_) in enumerate(ranges):
            want = (np.arange((re_ - rb) * K, dtype=np.float32).reshape(re_ - rb, K) % 997.0) + 1000.0 * (r + 1)
            assert np.array_equal(full[rb:re_], want), (side, r)
        back = np.empty_like(rows)
        tr.get_shard_rows(side, back)
        assert np.array_equal(back, rows)
        dist.barrier()
    # step_io on host-resident shards == set rows + step + get rows
    tr.user, tr.item = u0, i0
    dist.barrier()
    tr.step(sc)
    want_u, want_i = tr.user, tr.item
    tr.user, tr.item = u0, i0
    dist.barrier()
    (ub, ue), (ib, ie) = tr.user_range, tr.item_range
    hu = torch.from_numpy(u0[ub:ue].copy()).pin_memory()
    hi = torch.from_numpy(i0[ib:ie].copy()).pin_memory()
    tr.step_io(sc, hu, hi)
    assert np.array_equal(hu.numpy(), want_u[ub:ue]) and np.array_equal(hi.numpy(), want_i[ib:ie])
    assert np.array_equal(tr.user, want_u) and np.array_equal(tr.item, want_i)
    dist.barrier()
    del tr
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(_n_devices() < 2, reason="needs two GPUs (gpurun --gpus 2)")
def test_one_rank_per_device_nccl_matches_single_process(tmp_path):
    out = str(tmp_path / "res.npz")
    _spawn(_worker_multi_device, min(_n_devices(), 4), out)
    r = np.load(out)
    for a, b in ((r["user"], r["ref_user"]), (r["item"], r["ref_item"])):
        assert np.abs(a - b).max() <= 2e-4 * np.abs(b).max()
