"""Candidate ranking on the host side, without a GPU: the ID mappers' translation of ids and unknown ids
against a recommender stub, the sorting and de-duplication of candidate lists, and the argument checks
made before the library is called."""
import ctypes

import numpy as np
import pytest


class _Stub:
    """Records the calls of the mappers; ranks each row's candidates in descending index order."""

    def __init__(self, n_users, n_items):
        self.n_users, self.n_items = n_users, n_items
        self.calls = []

    def _rank(self, rows, lists, cutoff):
        if len(lists) == 1:
            lists = list(lists) * rows
        idx = np.full((rows, cutoff), -1, dtype=np.int32)
        sc = np.full((rows, cutoff), -np.inf, dtype=np.float32)
        cnt = np.zeros(rows, dtype=np.int32)
        for r, lst in enumerate(lists):
            best = sorted(set(lst), reverse=True)[:cutoff]
            idx[r, :len(best)] = best
            sc[r, :len(best)] = [i / 10 for i in best]
            cnt[r] = len(best)
        return idx, cnt, sc

    def rank_candidates(self, u, lists, cutoff, **kw):
        self.calls.append(("known", np.asarray(u).copy(), lists, cutoff, kw))
        return self._rank(len(u), lists, cutoff)

    def rank_candidates_cold_user(self, X, lists, cutoff, **kw):
        self.calls.append(("new", X, lists, cutoff, kw))
        return self._rank(X.shape[0], lists, cutoff)


def _mapper():
    from irspack_b200.id_mapping import IDMapper

    return IDMapper([f"u{i}" for i in range(6)], [f"i{i}" for i in range(8)])


def test_known_users_translate_ids():
    m, rec = _mapper(), _Stub(6, 8)
    got = m.rank_items_for_known_users(rec, ["u2", "u5"], [["i1", "i6", "nope", "i6"], []], cutoff=5)
    kind, u, lists, cutoff, kw = rec.calls[-1]
    assert kind == "known" and list(u) == [2, 5] and lists == [[1, 6, 6], []]
    assert cutoff == 3 and kw == {"mask": "train", "return_scores": True}  # no list holds more than 3
    assert got == [[("i6", pytest.approx(0.6)), ("i1", pytest.approx(0.1))], []]
    m.rank_items_for_known_users(rec, ["u0"], [["i3"]], cutoff=50, remove_seen=False)
    assert rec.calls[-1][3] == 1 and rec.calls[-1][4]["mask"] is None
    assert m.rank_items_for_known_users(rec, [], [], cutoff=3) == []


def test_new_user_translates_ids():
    m, rec = _mapper(), _Stub(6, 8)
    got = m.rank_items_for_new_user(rec, ["i0", "i4"], ["i7", "i2", "zz"], cutoff=1)
    kind, X, lists, cutoff, kw = rec.calls[-1]
    assert kind == "new" and X.shape == (1, 8) and sorted(X.indices) == [0, 4]
    assert lists == [[7, 2]] and cutoff == 1 and kw["mask"] == "input"
    assert got == [("i7", pytest.approx(0.7))]
    m.rank_items_for_new_user(rec, {"i1": 2.0}, ["i1"], remove_seen=False)
    assert rec.calls[-1][4]["mask"] is None


def test_unknown_ids_and_recommenders():
    m, rec = _mapper(), _Stub(6, 8)
    with pytest.raises(RuntimeError, match="User with user_id nope not found"):
        m.rank_items_for_known_users(rec, ["u1", "nope"], [[], []])
    with pytest.raises(ValueError):
        m.rank_items_for_known_users(rec, ["u1"], [[], []])
    with pytest.raises(ValueError):
        m.rank_items_for_known_users(_Stub(6, 9), ["u1"], [[]])
    with pytest.raises(ValueError):
        m.rank_items_for_new_user(_Stub(6, 9), [], [])

    class NoRanking:
        n_users, n_items = 6, 8

    with pytest.raises(NotImplementedError):
        m.rank_items_for_known_users(NoRanking(), ["u1"], [["i1"]])
    with pytest.raises(NotImplementedError):
        m.rank_items_for_new_user(NoRanking(), [], ["i1"])


def test_lists_are_sorted_and_deduplicated():
    from irspack_b200._ials_core import _candidate_lists

    n, ip, ix = _candidate_lists([[5, 1, 5, 3], [], [2, 2]], 3, 10)
    assert n == 3 and list(ip) == [0, 3, 3, 4] and list(ix) == [1, 3, 5, 2] and ix.dtype == np.int32
    n, ip, ix = _candidate_lists((2, np.array([0, 3, 5]), np.array([9, 0, 9, 4, 1])), 2, 10)
    assert list(ip) == [0, 2, 4] and list(ix) == [0, 9, 1, 4]
    n, ip, ix = _candidate_lists([[4, 0, 4]], 7, 10)  # one list shared by 7 rows
    assert n == 1 and list(ip) == [0, 2] and list(ix) == [0, 4]
    n, ip, ix = _candidate_lists([[4, 0, 4]], 1, 10, rank=False)  # pair scores keep the input order
    assert list(ix) == [4, 0, 4]
    for bad in ([[1], [2]], [[10]], [[-1]], [[1.5]], [[2**32 + 1]],
                (1, np.array([0, 3]), np.array([4, 10, 2], np.int32)), (1, np.array([0, 2]), np.array([-3, 1], np.int32)), (2, np.array([0, 1]), np.array([1])),
                (1, np.array([0, 2]), np.array([1])), (2, np.array([0, 2, 1]), np.array([1]))):
        with pytest.raises(ValueError):
            _candidate_lists(bad, 3, 10)


@pytest.mark.parametrize("kw", [
    dict(cutoff=0), dict(cutoff=11), dict(cutoff=1025), dict(users=range(0, 7)), dict(users=range(3, 1)),
    dict(users=range(0, 4, 2)), dict(mask="seen"), dict(candidates=[[1], [2]]), dict(candidates=[[10]]),
    dict(users=None, embeddings=np.zeros((2, 3), np.float32)),
    dict(users=None, embeddings=np.zeros((2, 4), np.float32), mask="train"),
])
def test_argument_checks_before_the_library(kw):
    from irspack_b200 import _ials_core

    args = dict(users=[0, 1, 2], embeddings=None, candidates=[[1, 2]], cutoff=2, mask="train")
    args.update(kw)
    with pytest.raises(ValueError):  # a null handle: nothing may reach the library
        _ials_core._rank_candidates(ctypes.c_void_p(0), 0, 6, 10, 4, args["users"], args["embeddings"],
                                    args["candidates"], args["cutoff"], args["mask"], True)
