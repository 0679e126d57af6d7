"""Similar items / users on the host side, without a GPU: the ID mappers' translation of ids, unknown
ids and allow / forbid lists against a recommender stub, and the argument checks made before the
library is called."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sps


class _Stub:
    """Records the calls of the mappers; the lists it answers are query + 1, query + 2, ..."""

    def __init__(self, n_users, n_items):
        self.n_users, self.n_items = n_users, n_items
        self.calls = []

    def _lists(self, n, q, cutoff):
        q = np.asarray(q)
        idx = (q[:, None] + 1 + np.arange(cutoff)[None, :]) % n
        cnt = np.full(q.size, cutoff, dtype=np.int32)
        idx[:, cutoff - 1:] = -1  # one entry short
        cnt[:] = cutoff - 1
        return idx.astype(np.int32), cnt, (1.0 / (1 + np.arange(cutoff)[None, :] + q[:, None])).astype(np.float32)

    def get_similar_items(self, q, cutoff, **kw):
        self.calls.append(("items", np.asarray(q).copy(), cutoff, kw))
        return self._lists(self.n_items, q, cutoff)

    def get_similar_users(self, q, cutoff, **kw):
        self.calls.append(("users", np.asarray(q).copy(), cutoff, kw))
        return self._lists(self.n_users, q, cutoff)


def _mapper():
    from irspack_b200.id_mapping import IDMapper

    return IDMapper([f"u{i}" for i in range(6)], [f"i{i}" for i in range(8)])


def test_similar_items_translates_ids():
    m, rec = _mapper(), _Stub(6, 8)
    got = m.similar_items(rec, ["i2", "i7"], cutoff=3)
    kind, q, cutoff, kw = rec.calls[-1]
    assert kind == "items" and list(q) == [2, 7] and cutoff == 3
    assert kw["forbidden"] is None and kw["allowed"] is None and kw["return_scores"]
    assert got == [[("i3", pytest.approx(1 / 3)), ("i4", pytest.approx(1 / 4))],
                   [("i0", pytest.approx(1 / 8)), ("i1", pytest.approx(1 / 9))]]
    m.similar_items(rec, ["i1"], cutoff=50)  # the cutoff is clipped to the catalogue
    assert rec.calls[-1][2] == 8
    assert m.similar_items(rec, [], cutoff=3) == []


def test_similar_items_lists():
    m, rec = _mapper(), _Stub(6, 8)
    m.similar_items(rec, ["i2", "i5"], cutoff=2, allowed_item_ids=["i6", "nope", "i1", "i6"],
                    forbidden_item_ids=[["i3", "zz", "i3"], []])
    kw = rec.calls[-1][3]
    n_lists, ip, ix = kw["allowed"]
    assert n_lists == 1 and list(ip) == [0, 2] and list(ix) == [1, 6]
    f = sps.csr_matrix(kw["forbidden"])
    assert f.shape == (2, 8) and f.toarray().nonzero() == ((0,), (3,))
    m.similar_items(rec, ["i2", "i5"], cutoff=2, per_item_allowed_item_ids=[["i4", "i0"], ["bad"]])
    n_lists, ip, ix = rec.calls[-1][3]["allowed"]
    assert n_lists == 2 and list(ip) == [0, 2, 2] and list(ix) == [0, 4]


def test_similar_users_translates_ids():
    m, rec = _mapper(), _Stub(6, 8)
    got = m.similar_users(rec, ["u5", "u0"], cutoff=2)
    kind, q, cutoff, _ = rec.calls[-1]
    assert kind == "users" and list(q) == [5, 0] and cutoff == 2
    assert got == [[("u0", pytest.approx(1 / 6))], [("u1", pytest.approx(1.0))]]


def test_unknown_ids_and_recommenders():
    m, rec = _mapper(), _Stub(6, 8)
    with pytest.raises(RuntimeError, match="Item with item_id nope not found"):
        m.similar_items(rec, ["i1", "nope"])
    with pytest.raises(RuntimeError, match="User with user_id 17 not found"):
        m.similar_users(rec, [17])
    with pytest.raises(ValueError):
        m.similar_items(_Stub(6, 9), ["i1"])
    with pytest.raises(ValueError):
        m.similar_users(_Stub(5, 8), ["u1"])

    class NoSimilar:
        n_users, n_items = 6, 8

    with pytest.raises(NotImplementedError):
        m.similar_items(NoSimilar(), ["i1"])
    with pytest.raises(NotImplementedError):
        m.similar_users(NoSimilar(), ["u1"])


@pytest.mark.parametrize("kw", [
    dict(side=2), dict(side=-1), dict(metric="euclidean"), dict(cutoff=0), dict(cutoff=11),
    dict(indices=range(0, 11)), dict(indices=range(4, 2)), dict(indices=range(0, 6, 2)),
    dict(indices=range(2, 4), forbidden=sps.csr_matrix((2, 9))),
    dict(indices=[1, 2, 3], forbidden=sps.csr_matrix((2, 10))),
    dict(indices=[1], allowed=(1, np.array([0, 3]), np.array([1, 2]))),
    dict(indices=[1], allowed=(2, np.array([0, 1]), np.array([1]))),
])
def test_argument_checks_before_the_library(kw):
    from irspack_b200 import _ials_core

    args = dict(side=1, indices=None, cutoff=5, metric="cosine", exclude_self=True, forbidden=None,
                allowed=None, return_scores=True)
    args.update(kw)
    with pytest.raises(ValueError):  # a null handle: nothing may reach the library
        _ials_core._similar(ctypes.c_void_p(0), 0, 10, args.pop("side"), args.pop("indices"), args.pop("cutoff"),
                            args.pop("metric"), args.pop("exclude_self"), args.pop("forbidden"),
                            args.pop("allowed"), args.pop("return_scores"))
