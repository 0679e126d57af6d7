"""Device-resident shard construction (irspack_b200/dist.py, BASELINE configs[3] / [4] plumbing):
a block generated, transposed and handed to ``ials_trainer_create_sharded`` without touching the
host must train exactly like the same matrix uploaded from scipy.  (The collective itself is
covered on CPU tensors by tests/test_dist.py, world_size 2 and 3 on gloo.)"""
import numpy as np
import pytest
import scipy.sparse as sps


@pytest.mark.gpu
def test_sharded_trainer_from_device_csr_matches_host_csr():
    import torch

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import (ShardedIALSTrainer, exchange_transposed_shards,
                                   global_item_bounds, synth_user_block_device)
    from irspack_b200.synth import init_factors

    dev = torch.device("cuda:0")
    torch.cuda.set_device(0)
    U, I, nnz, K = 3000, 900, 60000, 128
    ip, ix, dt = synth_user_block_device(U, I, nnz, seed=3, device=dev, item_seed=1)
    assert ip.is_cuda and int(ip[-1]) == nnz
    bounds = global_item_bounds(ix, I)
    assert list(bounds) == [0, I]
    t_ip, t_ix, t_dt = exchange_transposed_shards(ip, ix, dt, 0, U, bounds)
    X = sps.csr_matrix((dt.cpu().numpy(), ix.cpu().numpy(), ip.cpu().numpy()), shape=(U, I))
    Xt = sps.csr_matrix(X.T)
    Xt.sort_indices()
    assert np.array_equal(t_ip.cpu().numpy(), Xt.indptr)
    assert np.array_equal(t_ix.cpu().numpy(), Xt.indices)

    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.03).build()
    sc = core.IALSSolverConfigBuilder().build()
    a = ShardedIALSTrainer(cfg, (ip, ix, dt), 0, U, (t_ip, t_ix, t_dt), 0, I)
    b = ShardedIALSTrainer(cfg, X, 0, U, Xt, 0, I)
    assert a.user_range == (0, U) and a.item_range == (0, I) and a.nnz_local == nnz
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    for t in (a, b):
        t.user, t.item = u0, i0
        for _ in range(2):
            t.step(sc)
    # same arrays, same plan, same kernels: bit-identical
    assert np.array_equal(a.user, b.user) and np.array_equal(a.item, b.item)
    single = core.IALSTrainer(cfg, X)
    single.user, single.item = u0, i0
    for _ in range(2):
        single.step(sc)
    for x, y in ((a.user, single.user), (a.item, single.item)):
        assert np.abs(x - y).max() <= 1e-4 * np.abs(y).max()
    with pytest.raises(ValueError):
        ShardedIALSTrainer(cfg, (ip, ix, dt), 0, U, Xt, 0, I)
    with pytest.raises(ValueError):
        ShardedIALSTrainer(cfg, (ip.cpu(), ix.cpu(), dt.cpu()), 0, U, (t_ip, t_ix, t_dt), 0, I)
