"""ShardedIALSTrainer.explain / explain_history on 1, 2 and 3 gloo ranks on one device: rank-local on the
replicas, no collective.  Every rank's explanations of its own rows (both sides) and of cold rows must equal
the single-process IALSTrainer's on the same factors bit for bit; a foreign row by index is rejected.
Bounded joins: a rank that does not finish fails the test."""
import numpy as np
import pytest
import scipy.sparse as sps

from test_dist_features import _init, _spawn

pytestmark = pytest.mark.gpu


def _same(got, ref, what):
    for g, r in zip(got, ref):
        assert np.array_equal(g, r), what


def _worker_explain(rank, world, port):
    _init(rank, world, port)
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer

    rng = np.random.default_rng(7)
    U, I, K = 310, 577, 64
    X = sps.csr_matrix((rng.random((U, I)) < 0.05) * rng.integers(1, 4, size=(U, I)), dtype=np.float32)
    user = (rng.standard_normal((U, K)) * 0.05).astype(np.float32)
    item = (rng.standard_normal((I, K)) * 0.05).astype(np.float32)
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.02).build()
    single = core.IALSTrainer(cfg, X)
    single.user, single.item = user, item
    tr = ShardedIALSTrainer.from_global(cfg, X)
    tr.user, tr.item = user, item
    for side, n_other in ((0, I), (1, U)):
        b, e = tr.shard_range(side)
        own = np.arange(b, e)[::-1]
        targets = [rng.integers(0, n_other, size=int(n)) for n in rng.integers(0, 12, size=own.size)]
        _same(tr.explain(side, own, targets, n_top=5), single.explain(side, own, targets, n_top=5), (rank, side))
        targets = [rng.integers(0, n_other, size=3) for _ in range(e - b)]
        _same(tr.explain(side, range(b, e), targets, n_top=1024),
              single.explain(side, range(b, e), targets, n_top=1024), (rank, side, "range"))
        foreign = np.concatenate([np.arange(0, b), np.arange(e, U if side == 0 else I)])
        if foreign.size:
            with pytest.raises(ValueError):
                tr.explain(side, foreign[:1], [[0]])
    cold = sps.csr_matrix((rng.random((9, I)) < 0.1) * rng.integers(1, 4, size=(9, I)), dtype=np.float32)
    targets = [rng.integers(0, I, size=4) for _ in range(9)]
    _same(tr.explain_history(0, cold, targets, n_top=10), single.explain_history(0, cold, targets, n_top=10),
          (rank, "cold"))


@pytest.mark.parametrize("world", [1, 2, 3])
def test_every_rank_matches_the_single_trainer(world):
    _spawn(_worker_explain, world)
