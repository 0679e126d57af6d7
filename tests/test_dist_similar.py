"""ShardedIALSTrainer.similar on 1, 2 and 3 gloo ranks on one device: rank-local on the full replicas,
no collective.  Every rank's lists, for the rows of its own shard and for rows of other shards, must
equal the single-process IALSTrainer's on the same factors bit for bit.  Bounded joins: a rank that
does not finish fails the test."""
import numpy as np
import pytest
import scipy.sparse as sps

from test_dist_features import _init, _spawn

pytestmark = pytest.mark.gpu


def _worker_similar(rank, world, port):
    _init(rank, world, port)
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer

    rng = np.random.default_rng(4)
    U, I, K = 310, 277, 96
    X = sps.csr_matrix((rng.random((U, I)) < 0.05).astype(np.float32))
    user = rng.standard_normal((U, K)).astype(np.float32)
    item = rng.standard_normal((I, K)).astype(np.float32)
    item[7] = 0.0
    cfg = core.IALSModelConfigBuilder().set_K(K).build()
    single = core.IALSTrainer(cfg, X)
    single.user, single.item = user, item
    tr = ShardedIALSTrainer.from_global(cfg, X)
    tr.user, tr.item = user, item
    for side in (0, 1):
        n = U if side == 0 else I
        b, e = tr.shard_range(side)
        foreign = np.concatenate([np.arange(0, b), np.arange(e, n)])[::7]
        forb = sps.csr_matrix((np.arange(foreign.size) % 3 == 0).astype(np.float32)[:, None]
                              * (rng.random((1, n)) < 0.1).astype(np.float32))
        cases = [((range(b, e),), {}), ((foreign,), {}), ((foreign,), {"forbidden": forb}),
                 ((foreign[::-1],), {"metric": "dot", "exclude_self": False})]
        for args, kw in cases:
            for k in (10, 150):
                got = tr.similar(side, *args, cutoff=k, **kw)
                ref = single.similar(side, *args, cutoff=k, **kw)
                for g, r in zip(got, ref):
                    assert np.array_equal(g, r), (rank, side, k, kw)


@pytest.mark.parametrize("world", [1, 2, 3])
def test_every_rank_matches_the_single_trainer(world):
    _spawn(_worker_similar, world)
