"""Evaluator for the B200 iALS path.

Mirror of the hot-user ``Evaluator`` flow of the reference
(/root/reference/src/irspack/evaluation/evaluator.py:98-205, 400-441) with the
per-chunk work re-cut for the GPU:

* the score GEMM, the seen-item mask and the top-``cutoff`` selection run on the
  device (``IALSTrainer.recommend`` -- fused, the U x I score matrix never
  reaches the host -- or ``ials_topk_scores`` for any other recommender's
  float32 score block);
* only ``cutoff`` indices per user come back, and the metric arithmetic of
  ``Metrics::update`` / ``as_dict`` (cpp_source/evaluator.cpp:87-166) is done
  here on the host in float64, vectorised with numpy.

Also mirrored, on the same device kernels: ``recommendable_items`` /
``per_user_recommendable_items`` (allow-lists, ``ials_retrieve_recommend``),
``get_score(s)_from_score_matrix`` / ``get_score(s)_from_score_chunks``
(evaluator.py:228-398), float64 score blocks (selected on the device at float32
resolution, then the candidates that tie at that resolution are ranked with their
float64 values -- the same lists an all-float64 selection returns) and
``EvaluatorWithColdUser`` (evaluator.py:470-657; fold-in, score, mask and top-k of a
block of cold users stay on the device for an ``IALSRecommender``).
``cold_item_features`` belongs to the feature-aware model, which is outside the
hot path (SURVEY.md 8): ``NotImplementedError``.
"""
from __future__ import annotations

import ctypes
from collections import OrderedDict
from enum import Enum, auto
from typing import Any, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import scipy.sparse as sps

from ._ials_core import _current_device_and_stream, _ptr

MAX_DEVICE_CUTOFF = 1024  # ials_trainer_recommend / ials_topk_scores / ials_retrieve_recommend
from ._lib import check, lib
from ._threading import get_n_threads


class TargetMetric(Enum):  # evaluator.py:17-22
    ndcg = auto()
    recall = auto()
    hit = auto()
    map = auto()
    precision = auto()


METRIC_NAMES = [  # evaluator.py:25-35
    "hit", "recall", "ndcg", "map", "precision", "gini_index", "entropy", "appeared_item",
    "catalog_coverage",
]


class Metrics:
    """Accumulator equal to the reference's ``Metrics`` (evaluator.cpp:49-179)."""

    def __init__(self, n_item: int) -> None:
        self.n_item = int(n_item)
        self.valid_user = 0
        self.total_user = 0
        self.hit = 0.0
        self.recall = 0.0
        self.ndcg = 0.0
        self.precision = 0.0
        self.map = 0.0
        self.item_cnt = np.zeros(self.n_item, dtype=np.int64)

    def merge(self, other: "Metrics") -> None:  # evaluator.cpp:76-85
        self.hit += other.hit
        self.recall += other.recall
        self.ndcg += other.ndcg
        self.total_user += other.total_user
        self.valid_user += other.valid_user
        self.item_cnt += other.item_cnt
        self.precision += other.precision
        self.map += other.map

    # blocks with at least this many (user, position) pairs are accumulated on the device
    # (ials_metrics_accumulate, csrc/metrics.cu: one warp per user); the numpy form below takes
    # ~3 s for the 138 493 x 10 lists of configs[1], next to 8 ms of scoring
    DEVICE_MIN_PAIRS = 1 << 16

    def update_block(self, rec: np.ndarray, n_rec: np.ndarray, gt: sps.csr_matrix,
                     recall_with_cutoff: bool) -> None:
        """``get_metrics_local`` bookkeeping + ``Metrics::update`` for a block of users
        (evaluator.cpp:308-361, 127-166).  ``rec`` int32 [rows, cutoff] (-1 padded),
        ``n_rec`` valid entries per row, ``gt`` the block's ground-truth rows."""
        rows, cutoff = rec.shape
        if rows * cutoff >= self.DEVICE_MIN_PAIRS:
            self._update_block_device(rec, n_rec, gt, recall_with_cutoff)
            return
        self.total_user += rows
        if rows == 0:
            return
        n_gt = np.diff(gt.indptr).astype(np.int64)
        valid = n_gt > 0  # users with empty ground truth are skipped, :319-321
        self.valid_user += int(valid.sum())
        use = valid & (n_rec > 0)  # Metrics::update returns early when nothing is recommendable
        if not use.any():
            return
        rec = rec[use].astype(np.int64)
        n_rec = n_rec[use].astype(np.int64)
        n_gt = n_gt[use]
        r = rec.shape[0]
        pos = np.arange(cutoff)
        in_list = pos[None, :] < n_rec[:, None]
        # membership of every recommended (user, item) pair in the ground truth
        gt_use = gt[np.flatnonzero(use)]
        gt_keys = (np.repeat(np.arange(r, dtype=np.int64), np.diff(gt_use.indptr)) * self.n_item
                   + gt_use.indices.astype(np.int64))
        rec_keys = np.arange(r, dtype=np.int64)[:, None] * self.n_item + np.where(in_list, rec, 0)
        if gt_use.has_sorted_indices and gt_keys.size:  # the keys ascend: one binary search per pair
            at = np.minimum(np.searchsorted(gt_keys, rec_keys), gt_keys.size - 1)
            hits = (gt_keys[at] == rec_keys) & in_list
        else:
            hits = np.isin(rec_keys, gt_keys) & in_list
        discount = 1.0 / np.log2(2.0 + pos)  # prepare_dcg_discount, :42-48
        cum_discount = np.cumsum(discount)
        dcg = (hits * discount[None, :]).sum(axis=1)
        idcg = cum_discount[np.minimum(n_gt, n_rec) - 1]
        cum_hit = np.cumsum(hits, axis=1)
        ap = (hits * (cum_hit / (pos[None, :] + 1.0))).sum(axis=1)
        total_hit = cum_hit[:, -1]
        self.hit += float((total_hit > 0).sum())
        self.precision += float((total_hit / n_rec).sum())
        denom = np.minimum(n_gt, n_rec) if recall_with_cutoff else n_gt
        self.recall += float((total_hit / denom).sum())
        self.ndcg += float((dcg / idcg).sum())
        self.map += float((ap / n_gt).sum())
        self.item_cnt += np.bincount(rec[in_list], minlength=self.n_item)

    @staticmethod
    def diversity(item_cnt: np.ndarray) -> Tuple[float, float, float]:
        """(appeared_item, entropy, gini_index) of an item-count histogram (evaluator.cpp:87-123)."""
        cnt = np.sort(item_cnt)
        total_item = float(cnt.sum())
        nz = cnt > 0
        appeared = float(nz.sum())
        entropy = 0.0
        gini = 0.0
        n = cnt.shape[0]
        if appeared:
            p = cnt[nz] / total_item
            entropy = float((-np.log(p) * p).sum())
            idx = np.flatnonzero(nz).astype(np.float64)
            gini = float(((2 * idx - n + 1) * cnt[nz]).sum())
        if total_item > 0:
            gini /= n * total_item
        return appeared, entropy, gini

    def _update_block_device(self, rec: np.ndarray, n_rec: np.ndarray, gt: sps.csr_matrix,
                             recall_with_cutoff: bool) -> None:
        rows, cutoff = rec.shape
        g = sps.csr_matrix(gt)
        if not g.has_sorted_indices:
            g = g.copy()
            g.sort_indices()
        rec32 = np.ascontiguousarray(rec, dtype=np.int32)
        cnt32 = np.ascontiguousarray(np.minimum(n_rec, cutoff), dtype=np.int32)
        gi = np.ascontiguousarray(g.indptr, dtype=np.int64)
        gx = np.ascontiguousarray(g.indices, dtype=np.int32)
        discount = 1.0 / np.log2(2.0 + np.arange(cutoff))  # prepare_dcg_discount, :42-48
        acc = np.zeros(5, dtype=np.float64)
        valid = np.zeros(1, dtype=np.int64)
        dev, stream = _current_device_and_stream()
        check(lib.ials_metrics_accumulate(
            _ptr(rec32), _ptr(cnt32), rows, cutoff, _ptr(gi), _ptr(gx), self.n_item,
            int(bool(recall_with_cutoff)), _ptr(discount), dev, ctypes.c_void_p(stream),
            _ptr(acc), _ptr(valid), _ptr(self.item_cnt)))
        self.total_user += rows
        self.valid_user += int(valid[0])
        self.hit += float(acc[0])
        self.recall += float(acc[1])
        self.ndcg += float(acc[2])
        self.map += float(acc[3])
        self.precision += float(acc[4])

    def as_dict(self, diversity: Optional[Tuple[float, float, float]] = None) -> Dict[str, float]:
        """evaluator.cpp:87-123.  ``diversity``: (appeared_item, entropy, gini_index) when they were
        reduced elsewhere (``ShardedEvaluator``: on the device, from the histogram merged over ranks);
        None reduces ``item_cnt`` here."""
        if diversity is None:
            diversity = self.diversity(self.item_cnt)
        appeared, entropy, gini = diversity
        den = self.valid_user if self.valid_user > 0 else 1
        return {
            "total_user": float(self.total_user), "valid_user": float(self.valid_user),
            "n_items": float(self.n_item), "hit": self.hit / den, "ndcg": self.ndcg / den,
            "recall": self.recall / den, "map": self.map / den,
            "precision": self.precision / den, "appeared_item": appeared, "entropy": entropy,
            "gini_index": gini,
        }


def _mask_csr(mask: Any) -> Tuple[np.ndarray, np.ndarray]:
    m = sps.csr_matrix(mask, copy=True)
    m.eliminate_zeros()  # scipy's .nonzero() drops stored zeros (evaluator.py:432)
    m.sort_indices()
    return (np.ascontiguousarray(m.indptr, dtype=np.int64),
            np.ascontiguousarray(m.indices, dtype=np.int32))


def _device_topk(s32: np.ndarray, cutoff: int, mask: Optional[Tuple[np.ndarray, np.ndarray]]
                 ) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """``ials_topk_scores`` on a float32 host block: (idx, score, count)."""
    rows, n_items = s32.shape
    idx = np.empty((rows, cutoff), dtype=np.int32)
    val = np.empty((rows, cutoff), dtype=np.float32)
    cnt = np.empty((rows,), dtype=np.int32)
    mi, mx = mask if mask is not None else (None, None)
    dev, stream = _current_device_and_stream()
    check(lib.ials_topk_scores(_ptr(s32), rows, n_items, int(cutoff), _ptr(mi), _ptr(mx), dev,
                               ctypes.c_void_p(stream), _ptr(idx), _ptr(val), _ptr(cnt)))
    return idx, val, cnt


def _device_retrieve(s32: np.ndarray, cutoff: int, n_lists: int, indptr: np.ndarray,
                     flat: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """``ials_retrieve_recommend`` on a float32 host block with allow-lists."""
    rows, n_items = s32.shape
    idx = np.empty((rows, cutoff), dtype=np.int32)
    val = np.empty((rows, cutoff), dtype=np.float32)
    cnt = np.empty((rows,), dtype=np.int32)
    dev, stream = _current_device_and_stream()
    check(lib.ials_retrieve_recommend(_ptr(s32), rows, n_items, int(cutoff), int(n_lists),
                                      _ptr(indptr), _ptr(flat), dev, ctypes.c_void_p(stream),
                                      _ptr(idx), _ptr(val), _ptr(cnt)))
    return idx, val, cnt


def _rerank_f64(scores: np.ndarray, s32: np.ndarray, idx: np.ndarray, val: np.ndarray,
                cnt: np.ndarray, allowed: Optional[np.ndarray]) -> Tuple[np.ndarray, np.ndarray]:
    """Turn a float32-resolution selection into the float64 one.

    Rounding to float32 is monotone, so the float64 top-k of a row is contained in
    {items whose float32 score >= the k-th selected float32 score}: the device's list plus
    the candidates that tie with its last entry.  Rows without such excluded ties only
    need their list re-ordered by (-float64 score, index)."""
    rows, k = idx.shape
    if rows == 0 or k == 0:
        return idx, cnt
    pos = np.arange(k)[None, :]
    live = pos < cnt[:, None]
    safe = np.where(live, idx, 0).astype(np.int64)
    v64 = np.where(live, np.take_along_axis(scores, safe, axis=1), -np.inf)
    order = np.lexsort((np.where(live, idx, np.iinfo(np.int32).max), -v64), axis=-1)
    out = np.take_along_axis(idx, order, axis=1)
    full = np.flatnonzero(cnt == k)
    if full.size:
        thr = val[full, k - 1]
        ties_sel = (val[full] == thr[:, None]).sum(axis=1)
        tie_all = s32[full] == thr[:, None]
        if allowed is not None:
            tie_all &= allowed if allowed.ndim == 1 else allowed[full]
        for j in np.flatnonzero(tie_all.sum(axis=1) > ties_sel):
            r = full[j]
            cand = np.union1d(idx[r].astype(np.int64), np.flatnonzero(tie_all[j]))
            o = np.lexsort((cand, -scores[r, cand]))[:k]
            out[r] = cand[o].astype(np.int32)
    return out, cnt


def _allowed_matrix(rows: int, n_items: int, n_lists: int, indptr: np.ndarray, flat: np.ndarray
                    ) -> Optional[np.ndarray]:
    if n_lists == 0:
        return None
    ok = (flat >= 0) & (flat < n_items)
    if n_lists == 1:
        a = np.zeros(n_items, dtype=bool)
        a[flat[ok]] = True
        return a
    a = np.zeros((rows, n_items), dtype=bool)
    r = np.repeat(np.arange(rows), np.diff(indptr))
    a[r[ok], flat[ok]] = True
    return a


def select_topk(scores: np.ndarray, cutoff: int, mask: Optional[sps.spmatrix] = None,
                allowed: Optional[Tuple[int, np.ndarray, np.ndarray]] = None
                ) -> Tuple[np.ndarray, np.ndarray]:
    """Best ``cutoff`` items of every row of a host score block, selected on the device with
    the reference's ordering (descending score, ties to the smaller index, ``-inf``
    excluded; evaluator.cpp:324-355).  ``mask``: entries to exclude (evaluator.py:426-432).
    ``allowed``: ``(n_lists, indptr, flat)`` with ``n_lists`` 1 (shared list) or ``rows``.
    Returns (indices int32 [rows, min(cutoff, n_items)] -1 padded, counts int32 [rows])."""
    scores = np.asarray(scores)
    if scores.dtype not in (np.float32, np.float64):
        raise ValueError("score must be either float32 or float64.")  # evaluator.py:183
    if scores.ndim != 2:
        raise ValueError("score block must be 2-D")
    rows, n_items = scores.shape
    k = min(int(cutoff), n_items)
    if rows == 0 or k == 0:
        return np.full((rows, k), -1, dtype=np.int32), np.zeros((rows,), dtype=np.int32)
    s32 = np.ascontiguousarray(scores, dtype=np.float32)
    csr = _mask_csr(mask) if mask is not None else None
    if allowed is None or allowed[0] == 0:
        idx, val, cnt = _device_topk(s32, k, csr)
        allow_m = None
    else:
        if csr is not None:  # the allow-list kernel takes no mask: scatter it like the reference
            if np.shares_memory(s32, scores):
                s32 = s32.copy()
            r = np.repeat(np.arange(rows), np.diff(csr[0]))
            s32[r, csr[1]] = -np.inf
        n_lists, indptr, flat = allowed
        idx, val, cnt = _device_retrieve(s32, k, n_lists, indptr, flat)
        allow_m = _allowed_matrix(rows, n_items, n_lists, indptr, flat)
    if scores.dtype == np.float64:
        if csr is not None and allow_m is None:  # ties must not resurrect masked entries
            r = np.repeat(np.arange(rows), np.diff(csr[0]))
            s32[r, csr[1]] = -np.inf
        idx, cnt = _rerank_f64(scores, s32, idx, val, cnt, allow_m)
    return idx, cnt


def topk_scores(scores: np.ndarray, cutoff: int, mask: Optional[sps.spmatrix] = None
                ) -> Tuple[np.ndarray, np.ndarray]:
    """Device top-``cutoff`` of a host score block (see ``select_topk``)."""
    return select_topk(scores, cutoff, mask)


def _csr_row_block(m: sps.csr_matrix, begin: int, end: int) -> sps.csr_matrix:
    """Rows ``[begin, end)`` of a CSR matrix as views of its arrays (scipy's ``m[begin:end]`` copies
    them: 25 of the 27 ms of host work in an Evaluator pass over configs[1]'s users)."""
    lo, hi = int(m.indptr[begin]), int(m.indptr[end])
    out = sps.csr_matrix((end - begin, m.shape[1]), dtype=m.dtype)
    out.data, out.indices = m.data[lo:hi], m.indices[lo:hi]  # (the constructor would copy offset views)
    out.indptr = m.indptr[begin: end + 1] - m.indptr[begin]
    out.has_sorted_indices = m.has_sorted_indices
    return out


def _lists_to_csr(lists: Sequence[Sequence[int]]) -> Tuple[np.ndarray, np.ndarray]:
    indptr = np.zeros(len(lists) + 1, dtype=np.int64)
    if len(lists):
        np.cumsum([len(x) for x in lists], out=indptr[1:])
    flat = np.fromiter((int(i) for x in lists for i in x), dtype=np.int64, count=int(indptr[-1]))
    return indptr, flat


def _canonical_lists(indptr: np.ndarray, flat: np.ndarray, n_items: int
                     ) -> Tuple[np.ndarray, np.ndarray]:
    """Every list sorted, de-duplicated and cut to ``[0, n_items)``: the set the host path's
    allow matrix holds (``_allowed_matrix``), as the strictly ascending int32 CSR that
    ``ials_trainer_recommend_allowed`` takes."""
    n = len(indptr) - 1
    rows = np.repeat(np.arange(n, dtype=np.int64), np.diff(indptr))
    ok = (flat >= 0) & (flat < n_items)
    key = np.unique(rows[ok] * max(n_items, 1) + flat[ok])
    out = np.zeros(n + 1, dtype=np.int64)
    if n:
        np.cumsum(np.bincount(key // max(n_items, 1), minlength=n), out=out[1:])
    return out, (key % max(n_items, 1)).astype(np.int32)


class Evaluator:
    """See the module docstring; arguments as in evaluator.py:98-161."""

    def __init__(self, ground_truth: Any, offset: int = 0, cutoff: int = 10,
                 target_metric: str = "ndcg", recommendable_items: Optional[List[int]] = None,
                 per_user_recommendable_items: Any = None, masked_interactions: Any = None,
                 n_threads: Optional[int] = None, recall_with_cutoff: bool = False,
                 mb_size: int = 4096) -> None:
        gt = sps.csr_matrix(ground_truth).astype(np.float64)
        gt.sort_indices()
        # evaluator.py:115-136: [] (every item), one shared list, or one list per user
        if recommendable_items is None:
            if per_user_recommendable_items is None:
                lists: List[List[int]] = []
            else:
                if sps.issparse(per_user_recommendable_items):
                    per_user = sps.csr_matrix(per_user_recommendable_items)
                    lists = [[int(j) for j in row.nonzero()[1]] for row in per_user]
                else:
                    lists = per_user_recommendable_items
                if len(lists) != gt.shape[0]:
                    raise ValueError(
                        "ground_truth and per_user_recommendable_items have inconsistent shapes.")
        else:
            lists = [recommendable_items]
        self.recommendable_items = lists
        # EvaluatorCore keeps a single-element list as the shared list (evaluator.cpp:340-347),
        # also when there is exactly one user
        self._n_lists = len(lists)
        if not gt.has_sorted_indices:  # the device metrics search a user's ground-truth row
            gt = gt.copy()
            gt.sort_indices()
        self._allow_indptr, self._allow_flat = _lists_to_csr(lists)
        # the fused kernel walks a list with a cursor: ascending, unique, in-range ids
        self._allow_sorted_indptr, self._allow_sorted_flat = _canonical_lists(
            self._allow_indptr, self._allow_flat, gt.shape[1])
        self.ground_truth = gt
        if not lists:
            self.n_recommendable_items = gt.shape[1]
        elif len(lists) == 1:
            self.n_recommendable_items = len(lists[0])
        else:
            self.n_recommendable_items = len({i for user_items in lists for i in user_items})
        self.offset = offset
        self.n_users, self.n_items = gt.shape
        self.n_cold_items = 0
        self.target_metric = TargetMetric[target_metric]
        self.cutoff = cutoff
        self.target_metric_name = f"{self.target_metric.name}@{self.cutoff}"
        self.n_threads = get_n_threads(n_threads)
        # the reference defaults to 128-row chunks sized for CPU caches; the GPU
        # path only ships `cutoff` indices per user, so bigger chunks are free
        self.mb_size = mb_size
        if masked_interactions is None:
            self.masked_interactions = None
        else:
            if masked_interactions.shape != gt.shape:
                raise ValueError("ground_truth and masked_interactions have different shapes. ")
            self.masked_interactions = sps.csr_matrix(masked_interactions)
        self.recall_with_cutoff = recall_with_cutoff

    # -- public entry points (evaluator.py:186-324) --
    def get_target_score(self, model: Any) -> float:
        return self.get_score(model)[self.target_metric.name]

    def get_score(self, model: Any) -> Dict[str, float]:
        return self._get_scores_as_list(model, [self.cutoff])[0]

    def get_scores(self, model: Any, cutoffs: List[int]) -> Dict[str, float]:
        return self._flatten(cutoffs, self._get_scores_as_list(model, cutoffs))

    def get_score_from_score_matrix(self, scores: np.ndarray) -> Dict[str, float]:
        return self._get_scores_from_score_matrix_as_list(scores, [self.cutoff])[0]

    def get_scores_from_score_matrix(self, scores: np.ndarray, cutoffs: List[int]
                                     ) -> Dict[str, float]:
        return self._flatten(cutoffs, self._get_scores_from_score_matrix_as_list(scores, cutoffs))

    def get_score_from_score_chunks(self, score_chunks: Iterable[np.ndarray]) -> Dict[str, float]:
        return self._get_scores_from_score_chunks_as_list(score_chunks, [self.cutoff])[0]

    def get_scores_from_score_chunks(self, score_chunks: Iterable[np.ndarray], cutoffs: List[int]
                                     ) -> Dict[str, float]:
        return self._flatten(cutoffs, self._get_scores_from_score_chunks_as_list(score_chunks, cutoffs))

    @staticmethod
    def _flatten(cutoffs: List[int], per_cutoff: List[Dict[str, float]]) -> Dict[str, float]:
        result: Dict[str, float] = OrderedDict()
        for cutoff, score in zip(cutoffs, per_cutoff):
            for name in METRIC_NAMES:
                result[f"{name}@{cutoff}"] = score[name]
        return result

    def _metrics_as_dict(self, metrics: Metrics, diversity: Optional[Tuple[float, float, float]] = None
                         ) -> Dict[str, float]:  # evaluator.py:326-334
        result = metrics.as_dict(diversity)
        result["catalog_coverage"] = (
            result["appeared_item"] / self.n_recommendable_items
            if self.n_recommendable_items else float("nan"))
        return result

    # -- helpers --
    def _check_cutoffs(self, cutoffs: List[int]) -> int:
        for c in cutoffs:  # EvaluatorCore::get_metrics, evaluator.cpp:265-266
            if c <= 0:
                raise ValueError("cutoff must be strictly greather than 0.")
            if c > self.n_items:
                raise ValueError("cutoff must not exeeed the number of items.")
            if c > MAX_DEVICE_CUTOFF:  # the device selection (score_tc.cu / score.cu) keeps <= 1024 keys per row
                raise ValueError(f"cutoff > {MAX_DEVICE_CUTOFF} is not supported by the B200 top-k kernels "
                                 "(the reference's partial_sort takes any cutoff <= n_items).")
        return max(cutoffs)

    def _allowed_for(self, gt_begin: int, gt_end: int, canonical: bool = False
                     ) -> Optional[Tuple[int, np.ndarray, np.ndarray]]:
        """Allow-lists of the ground-truth rows ``[gt_begin, gt_end)`` in the C ABI's layout
        (``canonical``: the sorted int32 form of the fused kernel)."""
        if self._n_lists == 0:
            return None
        indptr, flat = ((self._allow_sorted_indptr, self._allow_sorted_flat) if canonical
                        else (self._allow_indptr, self._allow_flat))
        if self._n_lists == 1:
            return 1, indptr, flat
        ip = indptr[gt_begin: gt_end + 1]
        return gt_end - gt_begin, np.ascontiguousarray(ip - ip[0]), \
            np.ascontiguousarray(flat[ip[0]: ip[-1]])

    def _update(self, metrics: List[Metrics], cutoffs: List[int], rec: np.ndarray, n_rec: np.ndarray,
                gt_begin: int, gt_end: int) -> None:
        gt = _csr_row_block(self.ground_truth, gt_begin, gt_end)
        for m, c in zip(metrics, cutoffs):  # a shorter list is a prefix of the longest one
            m.update_block(rec[:, :c], np.minimum(n_rec, c), gt, self.recall_with_cutoff)

    def _get_score_matrix_mask(self) -> Optional[sps.csr_matrix]:  # evaluator.py:336-337
        return self.masked_interactions

    def _block_topk(self, model: Any, begin: int, end: int, cutoff: int, fused: bool = True
                    ) -> Tuple[np.ndarray, np.ndarray]:
        """Top-``cutoff`` of users ``[begin, end)``.  ``fused``: ask the model's
        ``recommend_block`` (IALSRecommender: scores, mask, allow-lists and top-k in one kernel,
        nothing but the indices leaves the device); with allow-lists it raises
        NotImplementedError where that kernel does not apply and the caller retries unfused."""
        custom = None
        if self.masked_interactions is not None:
            custom = self.masked_interactions[begin - self.offset: end - self.offset]
        if fused and hasattr(model, "recommend_block"):
            mask = "train" if custom is None else custom
            if self._n_lists == 0:
                return model.recommend_block(begin, end, cutoff, mask=mask)
            return model.recommend_block(begin, end, cutoff, mask=mask, allowed=self._allowed_for(
                begin - self.offset, end - self.offset, canonical=True))
        allowed = self._allowed_for(begin - self.offset, end - self.offset)
        try:
            scores = model.get_score_block(begin, end)
        except NotImplementedError:
            scores = model.get_score(np.arange(begin, end))
        mask = model.X_train_all[begin:end] if custom is None else custom
        return select_topk(np.asarray(scores), cutoff, mask, allowed)

    def _get_scores_as_list(self, model: Any, cutoffs: List[int]) -> List[Dict[str, float]]:
        if self.offset + self.n_users > model.n_users:  # evaluator.py:403-406
            raise ValueError("evaluator offset + n_users exceeds the model's n_users.")
        if self.n_items != model.n_items:
            raise ValueError("The model and evaluator assume different n_items.")
        cmax = self._check_cutoffs(cutoffs)
        metrics = [Metrics(self.n_items) for _ in cutoffs]
        block_end = self.offset + self.n_users
        # mb_size bounds the HOST score block of evaluator.py:415-420.  The fused device path never
        # materialises one (its scratch is a few hundred bytes per user), and a call of 4096 users
        # is two short waves of CTAs: it takes 32768 users per call (tools/time_recommend.py:
        # 29.6 ms in blocks of 4096 against 8.2 ms in one call for the 138 493 users of configs[1])
        fused = hasattr(model, "recommend_block")
        b = self.offset
        while b < block_end:
            e = min(b + (max(self.mb_size, 32768) if fused else self.mb_size), block_end)
            # one top-max(cutoffs) pass serves every cutoff
            try:
                rec, n_rec = self._block_topk(model, b, e, cmax, fused)
            except NotImplementedError:
                if not (fused and self._n_lists):
                    raise
                fused = False  # allow-lists outside the fused kernel's shapes: host score blocks
                continue
            self._update(metrics, cutoffs, rec, n_rec, b - self.offset, e - self.offset)
            b = e
        return [self._metrics_as_dict(m) for m in metrics]

    def _get_scores_from_score_matrix_as_list(self, scores: np.ndarray, cutoffs: List[int]
                                              ) -> List[Dict[str, float]]:  # evaluator.py:339-356
        scores = np.asarray(scores)
        if scores.ndim != 2 or scores.shape != (self.n_users, self.n_items):
            raise ValueError(f"score matrix must have shape ({self.n_users}, {self.n_items}), "
                             f"but got {scores.shape}.")
        if scores.dtype not in (np.dtype("float32"), np.dtype("float64")):
            raise ValueError("score matrix must have dtype float32 or float64.")
        chunks = (scores[b: b + self.mb_size] for b in range(0, self.n_users, self.mb_size))
        return self._get_scores_from_score_chunks_as_list(chunks, cutoffs)

    def _get_scores_from_score_chunks_as_list(self, score_chunks: Iterable[np.ndarray],
                                              cutoffs: List[int]) -> List[Dict[str, float]]:
        """evaluator.py:358-398.  The caller's arrays are never modified: the mask goes to
        the device as a CSR (or is scattered into the float32 staging copy)."""
        cmax = self._check_cutoffs(cutoffs)
        mask = self._get_score_matrix_mask()
        metrics = [Metrics(self.n_items) for _ in cutoffs]
        start = 0
        for chunk in score_chunks:
            if not isinstance(chunk, np.ndarray) or chunk.ndim != 2:
                raise ValueError(f"each score chunk must be a 2-D ndarray, got {type(chunk).__name__}.")
            if chunk.shape[1] != self.n_items:
                raise ValueError(f"score chunk must have n_items={self.n_items} columns, "
                                 f"got {chunk.shape[1]}.")
            if chunk.dtype not in (np.dtype("float32"), np.dtype("float64")):
                raise ValueError("score chunk must have dtype float32 or float64.")
            end = start + chunk.shape[0]
            if end > self.n_users:
                raise ValueError("score chunks supplied more rows than the evaluator's "
                                 f"n_users={self.n_users}: processed {end} rows.")
            if chunk.shape[0] == 0:
                continue
            rec, n_rec = select_topk(chunk, cmax, None if mask is None else mask[start:end],
                                     self._allowed_for(start, end))
            self._update(metrics, cutoffs, rec, n_rec, start, end)
            start = end
        if start != self.n_users:
            raise ValueError("score chunks did not cover the evaluator's "
                             f"n_users={self.n_users} rows: processed {start} rows.")
        return [self._metrics_as_dict(m) for m in metrics]


class EvaluatorWithColdUser(Evaluator):
    """Evaluation against users the model has not seen (evaluator.py:470-657): every block of
    ``input_interaction`` is folded in (``get_score_cold_user``), its own entries (or
    ``masked_interactions``) are excluded, the rest is ranked against ``ground_truth``."""

    def __init__(self, input_interaction: Any, ground_truth: Any, cutoff: int = 10,
                 target_metric: str = "ndcg", recommendable_items: Optional[List[int]] = None,
                 per_user_recommendable_items: Any = None, masked_interactions: Any = None,
                 n_threads: Optional[int] = None, recall_with_cutoff: bool = False,
                 mb_size: int = 1024, cold_item_features: Any = None) -> None:
        if cold_item_features is not None:
            raise NotImplementedError(
                "cold_item_features needs the feature-aware model, outside the B200 hot path")
        if input_interaction.shape[0] != ground_truth.shape[0]:
            raise ValueError("input_interaction and ground_truth must have the same number of rows.")
        super().__init__(ground_truth, offset=0, cutoff=cutoff, target_metric=target_metric,
                         recommendable_items=recommendable_items,
                         per_user_recommendable_items=per_user_recommendable_items,
                         masked_interactions=masked_interactions, n_threads=n_threads,
                         recall_with_cutoff=recall_with_cutoff, mb_size=mb_size)
        self.input_interaction = input_interaction
        self.n_warm_items = input_interaction.shape[1]
        self.cold_item_features = None
        self._input_interaction_mask = sps.csr_matrix(input_interaction)

    def _get_score_matrix_mask(self) -> Optional[sps.csr_matrix]:  # evaluator.py:574-577
        if self.masked_interactions is None:
            return self._input_interaction_mask
        return self.masked_interactions

    def _get_scores_as_list(self, model: Any, cutoffs: List[int]) -> List[Dict[str, float]]:
        if model.n_items != self.n_warm_items:  # evaluator.py:585-589
            raise ValueError("The model and input_interaction assume different numbers of "
                             "training items.")
        cmax = self._check_cutoffs(cutoffs)
        metrics = [Metrics(self.n_items) for _ in cutoffs]
        mask_all = self._get_score_matrix_mask()
        fused = hasattr(model, "recommend_cold_block")
        for b in range(0, self.n_users, self.mb_size):
            e = min(b + self.mb_size, self.n_users)
            chunk = self.input_interaction[b:e]
            mask = mask_all[b:e]
            rec = None
            if fused:  # device-resident path
                try:
                    if self._n_lists == 0:
                        rec, n_rec = model.recommend_cold_block(chunk, cmax, mask=mask)
                    else:
                        rec, n_rec = model.recommend_cold_block(
                            chunk, cmax, mask=mask, allowed=self._allowed_for(b, e, canonical=True))
                except NotImplementedError:
                    if not self._n_lists:
                        raise
                    fused = False
            if rec is None:
                rec, n_rec = select_topk(np.asarray(model.get_score_cold_user(chunk)), cmax, mask,
                                         self._allowed_for(b, e))
            self._update(metrics, cutoffs, rec, n_rec, b, e)
        return [self._metrics_as_dict(m) for m in metrics]
