"""ShardedIALSTrainer.rank_candidates on 1, 2 and 3 gloo ranks on one device: rank-local on the full item
replica, no collective.  Every rank's lists must equal the single-process IALSTrainer's on the same factors
bit for bit, for the users of its own shard (mask "train") and for users of other shards (an explicit
mask); mask "train" on another shard's users is rejected.  Bounded joins: a rank that does not finish fails
the test."""
import numpy as np
import pytest
import scipy.sparse as sps

from test_dist_features import _init, _spawn

pytestmark = pytest.mark.gpu


def _worker_candidates(rank, world, port):
    _init(rank, world, port)
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer

    rng = np.random.default_rng(4)
    U, I, K = 310, 1277, 96
    X = sps.csr_matrix((rng.random((U, I)) < 0.05).astype(np.float32))
    user = rng.standard_normal((U, K)).astype(np.float32)
    item = rng.standard_normal((I, K)).astype(np.float32)
    cfg = core.IALSModelConfigBuilder().set_K(K).build()
    single = core.IALSTrainer(cfg, X)
    single.user, single.item = user, item
    tr = ShardedIALSTrainer.from_global(cfg, X)
    tr.user, tr.item = user, item
    b, e = tr.shard_range(0)
    own = np.arange(b, e)[::-1]
    foreign = np.concatenate([np.arange(0, b), np.arange(e, U)])[::5]
    for k in (10, 200):
        lists = [rng.choice(I, int(n), replace=False) for n in rng.integers(0, 400, size=own.size)]
        for args, kw in (((range(b, e), [np.arange(0, I, 2)]), {}), ((own, lists), {})):
            got = tr.rank_candidates(*args, k, **kw)
            ref = single.rank_candidates(*args, k, **kw)
            for g, r in zip(got, ref):
                assert np.array_equal(g, r), (rank, k)
        if foreign.size:
            lists = [rng.choice(I, int(n), replace=False) for n in rng.integers(0, 400, size=foreign.size)]
            mask = X[foreign]
            got = tr.rank_candidates(foreign, lists, k, mask=mask)
            ref = single.rank_candidates(foreign, lists, k, mask="train")
            for g, r in zip(got, ref):
                assert np.array_equal(g, r), (rank, k)
            with pytest.raises(ValueError):
                tr.rank_candidates(foreign, lists, k, mask="train")


@pytest.mark.parametrize("world", [1, 2, 3])
def test_every_rank_matches_the_single_trainer(world):
    _spawn(_worker_candidates, world)
