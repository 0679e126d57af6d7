"""Serving top-k with allow / forbid lists (SURVEY.md §8 f3).

Mirrors ``irspack.utils.id_mapping`` (/root/reference/src/irspack/utils/id_mapping.py:29-453):
``retrieve_recommend_from_score``, ``ItemIDMapper`` and ``IDMapper`` keep the reference's
names, arguments and error behaviour.  The selection itself
(``retrieve_recommend_from_score<Real>``, /root/reference/cpp_source/util.hpp:426-504) runs on
the GPU through ``ials_retrieve_recommend`` (``include/ials_b200.h``): allow-list scatter +
block radix select; only ``cutoff`` (index, score) pairs per row come back to the host.
With an ``IALSRecommender`` the ``recommend_for_*`` calls do not even build the score block:
the fused scoring kernel takes the users (by index, or folded in from their profiles), the
seen and forbidden items as its mask and the allowed items as its allow-lists
(``ItemIDMapper._fused_serving`` -> ``ials_trainer_recommend_users``).
There is no CPU fallback.

Differences, all on points the reference leaves open: ties are returned in ascending index
order (the reference's comparator only looks at the score); a duplicate inside an allow-list
is one candidate; float64 scores are selected at float32 resolution on the device, then the
candidates that tie with the last selected one at that resolution are ranked with their
float64 values (``evaluation._rerank_f64``): the lists equal an all-float64 selection.
"""
from __future__ import annotations

from typing import (Any, Dict, Generic, Iterable, List, Optional, Sequence, Tuple, TypeVar, Union)

import numpy as np
import scipy.sparse as sps

from . import evaluation
from ._threading import get_n_threads

UserIdType = TypeVar("UserIdType")
ItemIdType = TypeVar("ItemIdType")
Profile = Union[List[Any], Dict[Any, float]]


def _lists_to_csr(lists: Sequence[Sequence[int]]) -> Tuple[np.ndarray, np.ndarray]:
    indptr = np.zeros(len(lists) + 1, dtype=np.int64)
    if lists:
        np.cumsum([len(x) for x in lists], out=indptr[1:])
    flat = np.fromiter((int(i) for x in lists for i in x), dtype=np.int64, count=int(indptr[-1]))
    return indptr, flat


def retrieve_recommend_from_score(score: np.ndarray, allowed_item_indices: List[List[int]],
                                  cutoff: int, n_threads: int = 1) -> List[List[Tuple[int, float]]]:
    """Best ``cutoff`` (item index, score) pairs of every row (id_mapping.py:29-46 ->
    util.hpp:426-504).  ``allowed_item_indices``: ``[]`` (all items), one list (shared) or one
    list per row; indices outside ``[0, n_items)`` are ignored; ``-inf`` is never returned."""
    score = np.asarray(score)
    if score.dtype not in (np.float32, np.float64):
        raise ValueError("Only float32 or float64 are allowed.")  # id_mapping.py:44-45
    if score.ndim != 2:
        raise ValueError("score must be 2-D")
    if n_threads <= 0:
        raise ValueError("n_threads must not be 0.")  # util.hpp:434
    if cutoff < 0:
        raise ValueError("cutoff must not be negative")
    rows, n_items = score.shape
    n_lists = len(allowed_item_indices)
    if n_lists not in (0, 1, rows):  # fail like the reference even when rows == 0 (util.hpp:436-439)
        raise ValueError("allowed_indices, if not empty, must have a size equal to X.rows()")
    k = min(int(cutoff), n_items)
    if rows == 0 or k == 0:
        return [[] for _ in range(rows)]
    s32 = np.ascontiguousarray(score, dtype=np.float32)
    indptr, flat = _lists_to_csr(allowed_item_indices)
    idx, val, cnt = evaluation._device_retrieve(s32, k, n_lists, indptr, flat)
    exact = score.dtype == np.float64
    if exact:  # candidates that tie at float32 resolution are ranked with their float64 values
        idx, cnt = evaluation._rerank_f64(score, s32, idx, val, cnt,
                                          evaluation._allowed_matrix(rows, n_items, n_lists, indptr, flat))
    out: List[List[Tuple[int, float]]] = []
    for r in range(rows):
        ids = idx[r, : cnt[r]]
        if exact:
            out.append([(int(i), float(score[r, i])) for i in ids])
        else:
            out.append([(int(i), float(v)) for i, v in zip(ids, val[r, : cnt[r]])])
    return out


class ItemIDMapper(Generic[ItemIdType]):
    """Item ids <-> column indices (id_mapping.py:52-349)."""

    def __init__(self, item_ids: List[ItemIdType]):
        self.item_ids = item_ids
        self.item_id_to_index = {iid: i for i, iid in enumerate(item_ids)}
        if len(self.item_id_to_index) != len(item_ids):
            raise ValueError("Duplicates in item_ids.")

    def _check_recommender_n_items(self, rec: Any) -> None:
        if rec.n_items != len(self.item_ids):
            raise ValueError("`n_items` of the recommender is inconsistent.")

    def _check_score_shape(self, score: np.ndarray) -> None:
        if score.shape[1] != len(self.item_ids):
            raise ValueError("`score.shape[1]` inconsistent with `len(self.item_ids)`")

    def _item_id_list_to_index_list(self, ids: Iterable[ItemIdType]) -> List[int]:
        known = self.item_id_to_index
        return [known[i] for i in ids if i in known]  # unknown ids are dropped silently

    def _user_profile_to_data_col(self, profile: Profile) -> Tuple[List[float], List[int]]:
        if isinstance(profile, list):
            cols = self._item_id_list_to_index_list(profile)
            return [1.0] * len(cols), cols
        data: List[float] = []
        cols = []
        for iid, rating in profile.items():
            if iid in self.item_id_to_index:
                data.append(rating)
                cols.append(self.item_id_to_index[iid])
        return data, cols

    def list_of_user_profile_to_matrix(self, users_info: Sequence[Profile]) -> sps.csr_matrix:
        """Interaction histories -> CSR with one row per profile (id_mapping.py:102-132)."""
        data: List[float] = []
        cols: List[int] = []
        indptr = [0]
        for profile in users_info:
            d, c = self._user_profile_to_data_col(profile)
            data.extend(d)
            cols.extend(c)
            indptr.append(len(cols))
        return sps.csr_matrix((data, cols, indptr), shape=(len(users_info), len(self.item_ids)))

    # ---- device-resident serving (B200): an IALSRecommender scores, masks, filters and selects
    # in one fused kernel (``ials_trainer_recommend_users`` / ``_recommend_allowed``); no score
    # block crosses the bus.  Anything the kernel does not take (cutoff > 128, other recommenders)
    # goes the reference's way: host score block -> ``retrieve_recommend_from_score``.
    _FUSED_MAX_CUTOFF = 128

    def _index_lists_csr(self, rows: int, lists: Sequence[Iterable[ItemIdType]]) -> sps.csr_matrix:
        """One list of item ids per row as a 0/1 CSR (unknown ids dropped, repeats merged)."""
        idx = [self._item_id_list_to_index_list(x) for x in lists]
        indptr, flat = _lists_to_csr(idx)
        m = sps.csr_matrix((np.ones(flat.size, dtype=np.float32), flat, indptr),
                           shape=(rows, len(self.item_ids)))
        m.sum_duplicates()
        m.data[:] = 1.0
        return m

    def _fused_serving(self, call: Any, rows: int, cutoff: int, seen: Any,
                       allowed_item_ids: Optional[List[ItemIdType]],
                       per_user_allowed_item_ids: Optional[List[List[ItemIdType]]],
                       forbidden_item_ids: Optional[List[List[ItemIdType]]]
                       ) -> Optional[List[List[Tuple[ItemIdType, float]]]]:
        """``call(cutoff, mask, allowed) -> (indices, counts, scores)`` of the recommender's fused
        path.  ``seen``: callable giving the rows' seen items as a CSR (needed only to merge the
        forbidden lists into the mask; without them the kernel masks with its own copy).
        Returns None where the fused kernel does not apply."""
        n_items = len(self.item_ids)
        k = min(int(cutoff), n_items)
        if rows == 0 or k < 1 or k > self._FUSED_MAX_CUTOFF:
            return None
        if forbidden_item_ids is not None:
            assert len(forbidden_item_ids) == rows
        if per_user_allowed_item_ids is not None:
            assert len(per_user_allowed_item_ids) == rows
        mask: Any = None
        if forbidden_item_ids is not None:
            mask = (sps.csr_matrix(seen()) != 0).astype(np.float32) + self._index_lists_csr(rows, forbidden_item_ids)
        allowed = self._allow_lists(rows, allowed_item_ids, per_user_allowed_item_ids)
        try:
            idx, cnt, sc = call(k, mask, allowed)
        except NotImplementedError:
            return None
        return self._id_lists(self.item_ids, idx, cnt, sc)

    def _allow_lists(self, rows: int, allowed_item_ids: Optional[List[ItemIdType]],
                     per_row_allowed_item_ids: Optional[List[List[ItemIdType]]]) -> Any:
        """``(n_lists, indptr, indices)`` allow-lists of the fused kernel (None: every item)."""
        if per_row_allowed_item_ids is not None:
            a = self._index_lists_csr(rows, per_row_allowed_item_ids)
            a.sort_indices()
            return (rows, a.indptr.astype(np.int64), a.indices.astype(np.int32))
        if allowed_item_ids is not None:
            a = np.unique(np.asarray(self._item_id_list_to_index_list(allowed_item_ids), dtype=np.int32))
            return (1, np.array([0, a.size], dtype=np.int64), a)
        return None

    @staticmethod
    def _id_lists(ids: List[Any], idx: np.ndarray, cnt: np.ndarray, sc: np.ndarray) -> List[List[Tuple[Any, float]]]:
        return [[(ids[i], float(v)) for i, v in zip(idx[r, :cnt[r]], sc[r, :cnt[r]])] for r in range(len(cnt))]

    @staticmethod
    def _query_indices(id_to_index: Dict[Any, int], ids: Iterable[Any], what: str) -> np.ndarray:
        out = []
        for i in ids:
            if i not in id_to_index:
                raise RuntimeError(f"{what} with {what.lower()}_id {i} not found.")
            out.append(id_to_index[i])
        return np.asarray(out, dtype=np.int64)

    def similar_items(self, recommender: Any, item_ids: List[ItemIdType], cutoff: int = 20,
                      allowed_item_ids: Optional[List[ItemIdType]] = None,
                      per_item_allowed_item_ids: Optional[List[List[ItemIdType]]] = None,
                      forbidden_item_ids: Optional[List[List[ItemIdType]]] = None
                      ) -> List[List[Tuple[ItemIdType, float]]]:
        """B200 extension: for each of ``item_ids``, the ``cutoff`` most similar other items (cosine
        similarity of the item factors) as [(item id, score)], best first; ties in ascending index
        order.  ``allowed_item_ids`` (shared) / ``per_item_allowed_item_ids`` restrict the candidates,
        ``forbidden_item_ids`` (one list per queried item) hides items; unknown ids in those lists are
        ignored, an unknown queried id raises ``RuntimeError``.  The recommender must provide
        ``get_similar_items`` (an ``IALSRecommender``): there is no host path."""
        self._check_recommender_n_items(recommender)
        if not hasattr(recommender, "get_similar_items"):
            raise NotImplementedError("similar_items needs a recommender with get_similar_items")
        q = self._query_indices(self.item_id_to_index, item_ids, "Item")
        rows = q.size
        if forbidden_item_ids is not None:
            assert len(forbidden_item_ids) == rows
        if per_item_allowed_item_ids is not None:
            assert len(per_item_allowed_item_ids) == rows
        if rows == 0:
            return []
        forbidden = None if forbidden_item_ids is None else self._index_lists_csr(rows, forbidden_item_ids)
        idx, cnt, sc = recommender.get_similar_items(
            q, min(int(cutoff), len(self.item_ids)), forbidden=forbidden,
            allowed=self._allow_lists(rows, allowed_item_ids, per_item_allowed_item_ids), return_scores=True)
        return self._id_lists(self.item_ids, idx, cnt, sc)

    def _candidate_cutoff(self, cutoff: int, lists: Sequence[Sequence[int]]) -> int:
        """The cutoff a ranking call needs: no list returns more items than it holds."""
        return min(int(cutoff), len(self.item_ids), max([len(x) for x in lists] + [1]))

    def rank_items_for_new_user(self, recommender: Any, user_profile: Profile,
                                candidate_item_ids: List[ItemIdType], cutoff: int = 20,
                                remove_seen: bool = True) -> List[Tuple[ItemIdType, float]]:
        """B200 extension: order the items ``candidate_item_ids`` for a user who is not in the model
        (folded in from ``user_profile``) as [(item id, score)], best first, at most ``cutoff``; ties in
        ascending index order.  Unknown and repeated candidate ids are ignored; with ``remove_seen`` the
        profile's items are dropped.  The recommender must provide ``rank_candidates_cold_user`` (an
        ``IALSRecommender``): there is no host path."""
        self._check_recommender_n_items(recommender)
        if not hasattr(recommender, "rank_candidates_cold_user"):
            raise NotImplementedError("rank_items_for_new_user needs a recommender with rank_candidates_cold_user")
        X = self.list_of_user_profile_to_matrix([user_profile])
        lists = [self._item_id_list_to_index_list(candidate_item_ids)]
        idx, cnt, sc = recommender.rank_candidates_cold_user(
            X, lists, self._candidate_cutoff(cutoff, lists), mask="input" if remove_seen else None,
            return_scores=True)
        return self._id_lists(self.item_ids, idx, cnt, sc)[0]

    def _explanations(self, e: Any, rows: int, lists: Sequence[Sequence[int]]
                      ) -> List[List[Tuple[ItemIdType, float, List[Tuple[ItemIdType, float]]]]]:
        """Per query row, per target: (item id, score, [(history item id, contribution), ...])."""
        ids = self.item_ids
        out = []
        for r in range(rows):
            row = []
            for p in range(int(e.indptr[r]), int(e.indptr[r + 1])):
                because = [(ids[int(e.indices[p, k])], float(e.contributions[p, k])) for k in range(int(e.counts[p]))]
                row.append((ids[lists[r][p - int(e.indptr[r])]], float(e.score[p]), because))
            out.append(row)
        return out

    def explain_for_new_user(self, recommender: Any, user_profile: Profile, item_ids: List[ItemIdType],
                             n_top: int = 10) -> List[Tuple[ItemIdType, float, List[Tuple[ItemIdType, float]]]]:
        """B200 extension: why a user who is not in the model (``user_profile``) scores each of
        ``item_ids``: [(item id, score, [(history item id, contribution), ...])], the ``n_top`` largest
        contributions first.  Unknown item and profile ids are ignored.  The recommender must provide
        ``explain_cold_user`` (an ``IALSRecommender``): there is no host path."""
        self._check_recommender_n_items(recommender)
        if not hasattr(recommender, "explain_cold_user"):
            raise NotImplementedError("explain_for_new_user needs a recommender with explain_cold_user")
        X = self.list_of_user_profile_to_matrix([user_profile])
        lists = [self._item_id_list_to_index_list(item_ids)]
        return self._explanations(recommender.explain_cold_user(X, lists, n_top=n_top), 1, lists)[0]

    def recommend_for_new_user(self, recommender: Any, user_profile: Profile, cutoff: int = 20,
                               allowed_item_ids: Optional[List[ItemIdType]] = None,
                               forbidden_item_ids: Optional[List[ItemIdType]] = None
                               ) -> List[Tuple[ItemIdType, float]]:
        self._check_recommender_n_items(recommender)
        X = self.list_of_user_profile_to_matrix([user_profile])
        if hasattr(recommender, "recommend_cold_block"):
            got = self._fused_serving(
                lambda k, mask, allowed: recommender.recommend_cold_block(
                    X, k, mask="input" if mask is None else mask, allowed=allowed, return_scores=True),
                1, cutoff, lambda: X, allowed_item_ids, None,
                None if forbidden_item_ids is None else [forbidden_item_ids])
            if got is not None:
                return got[0]
        score = recommender.get_score_cold_user_remove_seen(X)[0]
        return self.score_to_recommended_items(score, cutoff, allowed_item_ids, forbidden_item_ids)

    def recommend_for_new_user_batch(self, recommender: Any, user_profiles: Sequence[Profile],
                                     cutoff: int = 20,
                                     allowed_item_ids: Optional[List[ItemIdType]] = None,
                                     per_user_allowed_item_ids: Optional[List[List[ItemIdType]]] = None,
                                     forbidden_item_ids: Optional[List[List[ItemIdType]]] = None,
                                     n_threads: Optional[int] = None
                                     ) -> List[List[Tuple[ItemIdType, float]]]:
        self._check_recommender_n_items(recommender)
        X = self.list_of_user_profile_to_matrix(user_profiles)
        if hasattr(recommender, "recommend_cold_block"):
            got = self._fused_serving(
                lambda k, mask, allowed: recommender.recommend_cold_block(
                    X, k, mask="input" if mask is None else mask, allowed=allowed, return_scores=True),
                X.shape[0], cutoff, lambda: X, allowed_item_ids, per_user_allowed_item_ids,
                forbidden_item_ids)
            if got is not None:
                return got
        score = recommender.get_score_cold_user_remove_seen(X)
        return self.score_to_recommended_items_batch(
            score, cutoff, allowed_item_ids, per_user_allowed_item_ids, forbidden_item_ids, n_threads)

    def score_to_recommended_items(self, score: np.ndarray, cutoff: int,
                                   allowed_item_ids: Optional[List[ItemIdType]] = None,
                                   forbidden_item_ids: Optional[List[ItemIdType]] = None
                                   ) -> List[Tuple[ItemIdType, float]]:
        """One score row -> [(item id, score)] (id_mapping.py:225-256): infinite scores (either
        sign, ``np.isinf``) and forbidden ids are skipped without counting towards ``cutoff``."""
        score = np.asarray(score)
        self._check_score_shape(score[None, :])
        s = np.array(score, dtype=np.float32 if score.dtype != np.float64 else np.float64, copy=True)
        s[np.isinf(s)] = -np.inf
        if forbidden_item_ids is not None:
            s[self._item_id_list_to_index_list(forbidden_item_ids)] = -np.inf
        allowed = [] if allowed_item_ids is None else [self._item_id_list_to_index_list(allowed_item_ids)]
        (pairs,) = retrieve_recommend_from_score(s[None, :], allowed, cutoff, 1)
        return [(self.item_ids[i], v) for i, v in pairs]

    def score_to_recommended_items_batch(self, score: np.ndarray, cutoff: int,
                                         allowed_item_ids: Optional[List[ItemIdType]] = None,
                                         per_user_allowed_item_ids: Optional[List[List[ItemIdType]]] = None,
                                         forbidden_item_ids: Optional[List[List[ItemIdType]]] = None,
                                         n_threads: Optional[int] = None
                                         ) -> List[List[Tuple[ItemIdType, float]]]:
        """Score block -> per-row [(item id, score)] (id_mapping.py:249-324).  The forbidden
        entries are set to ``-inf`` in ``score`` itself, as the reference does (:306-310)."""
        self._check_score_shape(score)
        if forbidden_item_ids is not None:
            assert len(forbidden_item_ids) == score.shape[0]
        if per_user_allowed_item_ids is not None:
            assert len(per_user_allowed_item_ids) == score.shape[0]
        allowed: List[List[int]] = []
        if per_user_allowed_item_ids is not None:
            allowed = [self._item_id_list_to_index_list(x) for x in per_user_allowed_item_ids]
        elif allowed_item_ids is not None:
            allowed = [self._item_id_list_to_index_list(allowed_item_ids)]
        if forbidden_item_ids is not None:
            for u, ids in enumerate(forbidden_item_ids):
                score[u, self._item_id_list_to_index_list(ids)] = -np.inf
        raw = retrieve_recommend_from_score(score, allowed, cutoff, get_n_threads(n_threads))
        return [[(self.item_ids[i], v) for i, v in row] for row in raw]


class IDMapper(Generic[UserIdType, ItemIdType], ItemIDMapper[ItemIdType]):
    """User and item ids <-> indices (id_mapping.py:352-453)."""

    def __init__(self, user_ids: List[UserIdType], item_ids: List[ItemIdType]):
        super().__init__(item_ids)
        self.user_ids = user_ids
        self.user_id_to_index = {uid: i for i, uid in enumerate(user_ids)}
        if len(self.user_id_to_index) != len(user_ids):
            raise ValueError("Duplicates in user_ids.")

    def _check_recommender_n_users(self, rec: Any) -> None:
        if rec.n_users != len(self.user_ids):
            raise ValueError("`n_users` of the recommender is inconsistent.")

    def recommend_for_known_user_id(self, recommender: Any, user_id: UserIdType, cutoff: int = 20,
                                    allowed_item_ids: Optional[List[ItemIdType]] = None,
                                    forbidden_item_ids: Optional[List[ItemIdType]] = None
                                    ) -> List[Tuple[ItemIdType, float]]:
        self._check_recommender_n_users(recommender)
        self._check_recommender_n_items(recommender)
        if user_id not in self.user_id_to_index:
            raise RuntimeError(f"User with user_id {user_id} not found.")
        u = np.asarray([self.user_id_to_index[user_id]], dtype=np.int64)
        if hasattr(recommender, "recommend_users"):
            got = self._fused_serving(
                lambda k, mask, allowed: recommender.recommend_users(
                    u, k, mask="train" if mask is None else mask, allowed=allowed),
                1, cutoff, lambda: recommender.X_train_all[u], allowed_item_ids, None,
                None if forbidden_item_ids is None else [forbidden_item_ids])
            if got is not None:
                return got[0]
        score = recommender.get_score_remove_seen(u)[0, :]
        return self.score_to_recommended_items(score, cutoff, allowed_item_ids, forbidden_item_ids)

    def recommend_for_known_user_batch(self, recommender: Any, user_ids: List[UserIdType],
                                       cutoff: int = 20,
                                       allowed_item_ids: Optional[List[ItemIdType]] = None,
                                       per_user_allowed_item_ids: Optional[List[List[ItemIdType]]] = None,
                                       forbidden_item_ids: Optional[List[List[ItemIdType]]] = None,
                                       n_threads: Optional[int] = None
                                       ) -> List[List[Tuple[ItemIdType, float]]]:
        self._check_recommender_n_users(recommender)
        self._check_recommender_n_items(recommender)
        u = np.asarray([self.user_id_to_index[uid] for uid in user_ids], dtype=np.int64)
        if hasattr(recommender, "recommend_users"):
            got = self._fused_serving(
                lambda k, mask, allowed: recommender.recommend_users(
                    u, k, mask="train" if mask is None else mask, allowed=allowed),
                u.size, cutoff, lambda: recommender.X_train_all[u], allowed_item_ids,
                per_user_allowed_item_ids, forbidden_item_ids)
            if got is not None:
                return got
        score = recommender.get_score_remove_seen(u)
        return self.score_to_recommended_items_batch(
            score, cutoff, allowed_item_ids, per_user_allowed_item_ids, forbidden_item_ids, n_threads)

    def rank_items_for_known_users(self, recommender: Any, user_ids: List[UserIdType],
                                   candidate_item_ids: List[List[ItemIdType]], cutoff: int = 20,
                                   remove_seen: bool = True) -> List[List[Tuple[ItemIdType, float]]]:
        """B200 extension: for each of ``user_ids``, order that user's list in ``candidate_item_ids`` as
        [(item id, score)], best first, at most ``cutoff``; ties in ascending index order.  Unknown and
        repeated candidate ids are ignored, an unknown user id raises ``RuntimeError``; with
        ``remove_seen`` the users' training items are dropped.  The recommender must provide
        ``rank_candidates`` (an ``IALSRecommender``): there is no host path."""
        self._check_recommender_n_users(recommender)
        self._check_recommender_n_items(recommender)
        if not hasattr(recommender, "rank_candidates"):
            raise NotImplementedError("rank_items_for_known_users needs a recommender with rank_candidates")
        u = self._query_indices(self.user_id_to_index, user_ids, "User")
        if len(candidate_item_ids) != u.size:
            raise ValueError("candidate_item_ids must hold one list per user")
        if u.size == 0:
            return []
        lists = [self._item_id_list_to_index_list(x) for x in candidate_item_ids]
        idx, cnt, sc = recommender.rank_candidates(u, lists, self._candidate_cutoff(cutoff, lists),
                                                   mask="train" if remove_seen else None, return_scores=True)
        return self._id_lists(self.item_ids, idx, cnt, sc)

    def explain_for_known_users(self, recommender: Any, user_ids: List[UserIdType],
                                item_ids_per_user: List[List[ItemIdType]], n_top: int = 10
                                ) -> List[List[Tuple[ItemIdType, float, List[Tuple[ItemIdType, float]]]]]:
        """B200 extension: for each of ``user_ids``, why that user scores each item of their list in
        ``item_ids_per_user``: [(item id, score, [(history item id, contribution), ...])], the ``n_top``
        largest contributions of the user's training items first.  Unknown item ids are ignored, an
        unknown user id raises ``RuntimeError``.  The recommender must provide ``explain`` (an
        ``IALSRecommender``): there is no host path."""
        self._check_recommender_n_users(recommender)
        self._check_recommender_n_items(recommender)
        if not hasattr(recommender, "explain"):
            raise NotImplementedError("explain_for_known_users needs a recommender with explain")
        u = self._query_indices(self.user_id_to_index, user_ids, "User")
        if len(item_ids_per_user) != u.size:
            raise ValueError("item_ids_per_user must hold one list per user")
        if u.size == 0:
            return []
        lists = [self._item_id_list_to_index_list(x) for x in item_ids_per_user]
        return self._explanations(recommender.explain(u, lists, n_top=n_top), u.size, lists)

    def similar_users(self, recommender: Any, user_ids: List[UserIdType], cutoff: int = 20
                      ) -> List[List[Tuple[UserIdType, float]]]:
        """B200 extension, the user twin of ``similar_items``: for each of ``user_ids``, the ``cutoff``
        most similar other users (cosine similarity of the user factors) as [(user id, score)].  The
        recommender must provide ``get_similar_users``."""
        self._check_recommender_n_users(recommender)
        if not hasattr(recommender, "get_similar_users"):
            raise NotImplementedError("similar_users needs a recommender with get_similar_users")
        q = self._query_indices(self.user_id_to_index, user_ids, "User")
        if q.size == 0:
            return []
        idx, cnt, sc = recommender.get_similar_users(q, min(int(cutoff), len(self.user_ids)), return_scores=True)
        return self._id_lists(self.user_ids, idx, cnt, sc)
