"""Explanations on the host side, without a GPU: the ID mappers' translation of ids, unknown ids and result
shapes against a recommender stub, and the argument checks made before the library is called."""
import numpy as np
import pytest
import scipy.sparse as sps


class _Stub:
    """Records the mappers' calls; target t of row r scores t + r / 10 and lists history items 0 and 1
    with contributions t and -1."""

    def __init__(self, n_users, n_items):
        self.n_users, self.n_items = n_users, n_items
        self.calls = []

    def _explain(self, lists, n_top):
        from irspack_b200._ials_core import Explanation

        ip = np.zeros(len(lists) + 1, dtype=np.int64)
        np.cumsum([len(x) for x in lists], out=ip[1:])
        pairs = int(ip[-1])
        idx = np.full((pairs, n_top), -1, dtype=np.int32)
        con = np.full((pairs, n_top), -np.inf, dtype=np.float32)
        cnt = np.zeros(pairs, dtype=np.int32)
        score = np.zeros(pairs, dtype=np.float32)
        for r, lst in enumerate(lists):
            for q, t in enumerate(lst):
                p = ip[r] + q
                score[p] = t + r / 10
                n = min(2, n_top)
                idx[p, :n] = [0, 1][:n]
                con[p, :n] = [t, -1][:n]
                cnt[p] = n
        return Explanation(ip, score, np.zeros(pairs, np.float32), idx, con, cnt)

    def explain(self, u, lists, n_top=10):
        self.calls.append(("known", np.asarray(u).copy(), lists, n_top))
        return self._explain(lists, n_top)

    def explain_cold_user(self, X, lists, n_top=10):
        self.calls.append(("new", X, lists, n_top))
        return self._explain(lists, n_top)


def _mapper():
    from irspack_b200.id_mapping import IDMapper

    return IDMapper([f"u{i}" for i in range(6)], [f"i{i}" for i in range(8)])


def test_known_users_translate_ids():
    m, rec = _mapper(), _Stub(6, 8)
    got = m.explain_for_known_users(rec, ["u2", "u5"], [["i3", "nope", "i6"], []], n_top=5)
    kind, u, lists, n_top = rec.calls[-1]
    assert kind == "known" and list(u) == [2, 5] and lists == [[3, 6], []] and n_top == 5
    assert got == [[("i3", pytest.approx(3.0), [("i0", 3.0), ("i1", -1.0)]),
                    ("i6", pytest.approx(6.0), [("i0", 6.0), ("i1", -1.0)])], []]
    got = m.explain_for_known_users(rec, ["u0"], [["i7"]], n_top=1)
    assert got == [[("i7", pytest.approx(7.0), [("i0", 7.0)])]]
    assert m.explain_for_known_users(rec, [], []) == []
    with pytest.raises(RuntimeError):
        m.explain_for_known_users(rec, ["u9"], [["i1"]])
    with pytest.raises(ValueError):
        m.explain_for_known_users(rec, ["u1"], [["i1"], ["i2"]])


def test_new_user_translates_ids():
    m, rec = _mapper(), _Stub(6, 8)
    got = m.explain_for_new_user(rec, ["i0", "i4", "unknown"], ["i7", "zz", "i2"], n_top=3)
    kind, X, lists, n_top = rec.calls[-1]
    assert kind == "new" and X.shape == (1, 8) and sorted(X.indices.tolist()) == [0, 4] and lists == [[7, 2]]
    assert got == [("i7", pytest.approx(7.0), [("i0", 7.0), ("i1", -1.0)]),
                   ("i2", pytest.approx(2.0), [("i0", 2.0), ("i1", -1.0)])]
    assert m.explain_for_new_user(rec, {"i1": 2.0}, ["nope"]) == []


def test_recommender_without_the_method():
    m = _mapper()

    class Bare:
        n_users, n_items = 6, 8

    with pytest.raises(NotImplementedError):
        m.explain_for_known_users(Bare(), ["u0"], [["i1"]])
    with pytest.raises(NotImplementedError):
        m.explain_for_new_user(Bare(), ["i0"], ["i1"])


def test_python_side_argument_checks():
    from irspack_b200._ials_core import _explain, _target_lists

    ip, ix = _target_lists([[3, 1, 3], [], [0]], 3, 5)
    assert ip.tolist() == [0, 3, 3, 4] and ix.tolist() == [3, 1, 3, 0] and ix.dtype == np.int32
    ip, ix = _target_lists((np.array([0, 1, 1]), np.array([4])), 2, 5)
    assert ip.tolist() == [0, 1, 1] and ix.tolist() == [4]
    for bad, rows in (([[5]], 1), ([[-1]], 1), ([[0]], 2), ([[0.5]], 1),
                      ((np.array([0, 2]), np.array([1])), 1), ((np.array([1, 1]), np.array([1])), 1)):
        with pytest.raises(ValueError):
            _target_lists(bad, rows, 5)
    # checked before any library call: the handle is never touched
    for kw in (dict(side=2), dict(n_top=0), dict(n_top=1025), dict(indices=range(0, 9))):
        args = dict(side=0, indices=[0], X=None, targets=[[0]], n_top=1)
        args.update(kw)
        with pytest.raises(ValueError):
            _explain(None, 0, (6, 8), **args)
    with pytest.raises(TypeError):
        _explain(None, 0, (6, 8), 0, None, np.ones((1, 8)), [[0]], 1)
    with pytest.raises(ValueError):
        _explain(None, 0, (6, 8), 0, None, sps.csr_matrix((1, 7)), [[0]], 1)
