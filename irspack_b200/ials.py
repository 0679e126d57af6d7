"""``IALSRecommender`` on the B200 backend.

Host-side mirror of /root/reference/src/irspack/recommenders/ials.py
(``IALSTrainer`` adapter :68-203, ``IALSConfig`` :211-229, ``compute_reg_scale``
:232-242, ``IALSRecommender`` :245-791) and of the pieces of ``base.py`` /
``base_earlystop.py`` that path goes through (CSR canonicalisation base.py:94-105,
``learn`` :119-126, ``get_score_remove_seen*`` :308-337, the epoch loop
base_earlystop.py:106-149).  Same constructor arguments, defaults and error
behaviour; the compute is ``irspack_b200._ials_core`` (sm_100a CUDA).

Outside the hot path, raising ``NotImplementedError``: the Optuna
tuning entry points.  ``solver_type="IALSPP"`` (iALS++ block solver, SURVEY.md 8 f4) runs on
the GPU for ``ialspp_subspace_dimension <= 256``.
"""
from __future__ import annotations

import enum
import pickle
from dataclasses import asdict, dataclass
from io import BytesIO
from typing import IO, Any, Dict, Optional

import numpy as np
import scipy.sparse as sps

from ._ials_core import IALSModelConfigBuilder, IALSSolverConfigBuilder
from ._ials_core import IALSTrainer as CoreTrainer
from ._ials_core import LossType, SolverType
from ._threading import get_n_threads


def str_to_solver_type(t: str) -> SolverType:  # ials.py:46-49
    result: SolverType = getattr(SolverType, t.upper())
    assert result in {SolverType.CG, SolverType.CHOLESKY, SolverType.IALSPP}
    return result


def str_to_loss_type(t: str) -> LossType:  # ials.py:52-55
    result: LossType = getattr(LossType, t.upper())
    assert result in {LossType.ORIGINAL, LossType.IALSPP}
    return result


def _feature_matrix_as_float32(X: Any) -> Any:  # ials.py:58-61
    if sps.issparse(X):
        return sps.csr_matrix(X).astype(np.float32)
    return np.asarray(X, dtype=np.float32)


class IALSTrainer:
    """Adapter between the recommender and the core trainer (ials.py:68-203)."""

    def __init__(self, X: sps.csr_matrix, n_components: int, alpha0: float, reg: float, nu: float,
                 init_std: float, solver_type: SolverType, max_cg_steps: int,
                 ialspp_subspace_dimension: int, loss_type: LossType, random_seed: int,
                 n_threads: int, prediction_time_max_cg_steps: int,
                 prediction_time_ialspp_iteration: int, user_features: Any = None,
                 item_features: Any = None, lambda_user_feature: float = 0.0,
                 lambda_item_feature: float = 0.0, feature_warmup_epochs: int = 0) -> None:
        X_train_all_f32 = X.astype(np.float32)  # ials.py:91
        config = (IALSModelConfigBuilder().set_K(n_components).set_init_stdev(init_std)
                  .set_alpha0(alpha0).set_reg(reg).set_nu(nu).set_loss_type(loss_type)
                  .set_random_seed(random_seed).set_lambda_user_feature(lambda_user_feature)
                  .set_lambda_item_feature(lambda_item_feature)
                  .set_feature_warmup_epochs(feature_warmup_epochs).build())
        self.solver_config = (IALSSolverConfigBuilder().set_n_threads(n_threads)
                              .set_solver_type(solver_type).set_max_cg_steps(max_cg_steps)
                              .set_ialspp_iteration(1)
                              .set_ialspp_subspace_dimension(ialspp_subspace_dimension).build())
        if user_features is None and item_features is None:  # ials.py:115-128
            self.core_trainer = CoreTrainer(config, X_train_all_f32)
        else:  # a side without features gets an empty (n x 0) sparse feature matrix
            uf = (sps.csr_matrix((X.shape[0], 0), dtype=np.float32) if user_features is None
                  else _feature_matrix_as_float32(user_features))
            itf = (sps.csr_matrix((X.shape[1], 0), dtype=np.float32) if item_features is None
                   else _feature_matrix_as_float32(item_features))
            self.core_trainer = CoreTrainer(config, X_train_all_f32, uf, itf)
        self.prediction_time_solver_config = (
            IALSSolverConfigBuilder().set_n_threads(n_threads).set_solver_type(solver_type)
            .set_max_cg_steps(prediction_time_max_cg_steps)
            .set_ialspp_subspace_dimension(ialspp_subspace_dimension)
            .set_ialspp_iteration(prediction_time_ialspp_iteration).build())

    def load_state(self, ifs: IO) -> None:  # ials.py:140-146
        params = pickle.load(ifs)
        self.core_trainer.user = params["user"]
        self.core_trainer.item = params["item"]
        if "user_feature_weight" in params:  # ials.py:144-146
            self.core_trainer.user_feature_weight = params["user_feature_weight"]
            self.core_trainer.item_feature_weight = params["item_feature_weight"]

    def save_state(self, ofs: IO) -> None:  # ials.py:151-161
        pickle.dump(dict(user=self.core_trainer.user, item=self.core_trainer.item,
                         user_feature_weight=self.core_trainer.user_feature_weight,
                         item_feature_weight=self.core_trainer.item_feature_weight),
                    ofs, protocol=pickle.HIGHEST_PROTOCOL)

    def compute_loss(self) -> float:
        return self.core_trainer.compute_loss(self.solver_config)

    def run_epoch(self) -> None:  # ials.py:163-164
        self.core_trainer.step(self.solver_config)

    def user_scores(self, begin: int, end: int) -> np.ndarray:  # ials.py:166-167
        return self.core_trainer.user_scores(begin, end, self.solver_config)

    def transform_user(self, X: sps.csr_matrix, user_features: Any = None) -> np.ndarray:  # ials.py:169-180
        if user_features is None:
            return self.core_trainer.transform_user(X, self.prediction_time_solver_config)
        return self.core_trainer.transform_user_with_feature(
            X, _feature_matrix_as_float32(user_features), self.prediction_time_solver_config)

    def transform_item(self, X: sps.csr_matrix, item_features: Any = None) -> np.ndarray:  # ials.py:182-193
        if item_features is None:
            return self.core_trainer.transform_item(X, self.prediction_time_solver_config)
        return self.core_trainer.transform_item_with_feature(
            X, _feature_matrix_as_float32(item_features), self.prediction_time_solver_config)

    def transform_user_feature(self, user_features: Any) -> np.ndarray:  # ials.py:195-198
        return self.core_trainer.transform_user_feature(_feature_matrix_as_float32(user_features))

    def transform_item_feature(self, item_features: Any) -> np.ndarray:  # ials.py:200-203
        return self.core_trainer.transform_item_feature(_feature_matrix_as_float32(item_features))


class IALSConfigScaling(enum.Enum):  # ials.py:206-208
    none = enum.auto()
    log = enum.auto()


@dataclass
class IALSConfig:  # ials.py:211-229
    n_components: int = 20
    alpha0: float = 1.0
    reg: float = 1e-3
    nu: float = 1.0
    confidence_scaling: str = "none"
    epsilon: float = 1.0
    init_std: float = 0.1
    solver_type: str = "CG"
    max_cg_steps: int = 3
    loss_type: str = "IALSPP"
    nu_star: Optional[float] = None
    random_seed: int = 42
    n_threads: Optional[int] = None
    train_epochs: int = 16
    prediction_time_max_cg_steps: int = 5

    def dict(self) -> Dict[str, Any]:
        return asdict(self)


def compute_reg_scale(X: sps.csr_matrix, alpha0: float, nu: float) -> float:  # ials.py:232-242
    X_csr = sps.csr_matrix(X)
    U, I = X_csr.shape
    nnz_row = np.diff(X_csr.indptr)
    nnz_col = np.bincount(X_csr.indices, minlength=I)
    return float(((nnz_row + alpha0 * I) ** nu).sum()) + float(((nnz_col + alpha0 * U) ** nu).sum())


class IALSRecommender:
    """Implicit ALS / weighted matrix factorisation (ials.py:245-791) on one B200.

    ``IALSRecommender(X, n_components, alpha0, reg, epsilon, solver_type,
    max_cg_steps).learn()`` then ``get_score`` / ``get_score_block`` /
    ``get_score_remove_seen`` behave as in the reference."""

    config_class = IALSConfig

    def __init__(self, X_train_all: Any, n_components: int = 20, alpha0: float = 0.0,
                 reg: float = 1e-3, nu: float = 1.0, confidence_scaling: str = "none",
                 epsilon: float = 1.0, init_std: float = 0.1, solver_type: str = "CG",
                 max_cg_steps: int = 3, ialspp_subspace_dimension: int = 64,
                 loss_type: str = "IALSPP", nu_star: Optional[float] = None,
                 random_seed: int = 42, n_threads: Optional[int] = None, train_epochs: int = 16,
                 prediction_time_max_cg_steps: int = 5, prediction_time_ialspp_iteration: int = 7,
                 user_features: Any = None, item_features: Any = None,
                 lambda_user_feature: float = 0.0, lambda_item_feature: float = 0.0,
                 feature_warmup_epochs: int = 0) -> None:
        # BaseRecommender.__init__, base.py:94-101
        self.X_train_all: sps.csr_matrix = sps.csr_matrix(X_train_all).astype(np.float64)
        self.n_users, self.n_items = self.X_train_all.shape
        self.X_train_all.sort_indices()
        self.learnt_config: Dict[str, Any] = dict()
        self.train_epochs = train_epochs
        self.trainer: Optional[IALSTrainer] = None
        self.best_state: Optional[bytes] = None

        self.n_components = n_components
        self.alpha0 = alpha0
        self.reg = reg
        self.nu = nu
        self.confidence_scaling = IALSConfigScaling[confidence_scaling]
        self.epsilon = epsilon
        self.init_std = init_std
        self.solver_type = str_to_solver_type(solver_type)
        self.max_cg_steps = max_cg_steps
        self.ialspp_subspace_dimension = ialspp_subspace_dimension
        self.random_seed = random_seed
        self.n_threads = get_n_threads(n_threads)
        self.loss_type = str_to_loss_type(loss_type)
        self.nu_star = nu_star
        self.scaled_reg = self.reg
        if self.nu_star is not None:  # ials.py:412-418
            self.scaled_reg = (self.reg * compute_reg_scale(self.X_train_all, alpha0, self.nu_star)
                               / compute_reg_scale(self.X_train_all, alpha0, nu))
        self.prediction_time_max_cg_steps = prediction_time_max_cg_steps
        self.prediction_time_ialspp_iteration = prediction_time_ialspp_iteration
        # feature-aware model, ials.py:421-436
        self.user_features = None if user_features is None else _feature_matrix_as_float32(user_features)
        self.item_features = None if item_features is None else _feature_matrix_as_float32(item_features)
        self.lambda_user_feature = lambda_user_feature
        self.lambda_item_feature = lambda_item_feature
        self.feature_warmup_epochs = feature_warmup_epochs
        if ((self.user_features is not None or self.item_features is not None)
                and self.solver_type == SolverType.IALSPP):
            raise ValueError("Feature-aware iALS does not support IALSPP.")

    @classmethod
    def from_config(cls, X_train_all: Any, config: IALSConfig) -> "IALSRecommender":
        if not isinstance(config, cls.config_class):
            raise ValueError(f"Different config has been given. config must be {cls.config_class}")
        return cls(X_train_all, **config.dict())

    @classmethod
    def _scale_X(cls, X: sps.csr_matrix, scheme: IALSConfigScaling, epsilon: float) -> sps.csr_matrix:
        if scheme is IALSConfigScaling.none:  # ials.py:437-446
            return X
        X_ret: sps.csr_matrix = X.copy()
        X_ret.data = np.log(1 + X_ret.data / epsilon)
        return X_ret

    def _create_trainer(self) -> IALSTrainer:  # ials.py:448-469
        return IALSTrainer(
            X=self._scale_X(self.X_train_all, self.confidence_scaling, self.epsilon),
            n_components=self.n_components, alpha0=self.alpha0, reg=self.scaled_reg, nu=self.nu,
            init_std=self.init_std, solver_type=self.solver_type, max_cg_steps=self.max_cg_steps,
            ialspp_subspace_dimension=self.ialspp_subspace_dimension, loss_type=self.loss_type,
            random_seed=self.random_seed, n_threads=self.n_threads,
            prediction_time_max_cg_steps=self.prediction_time_max_cg_steps,
            prediction_time_ialspp_iteration=self.prediction_time_ialspp_iteration,
            user_features=self.user_features, item_features=self.item_features,
            lambda_user_feature=self.lambda_user_feature, lambda_item_feature=self.lambda_item_feature,
            feature_warmup_epochs=self.feature_warmup_epochs)

    # -- BaseRecommenderWithEarlyStopping, base_earlystop.py:80-149 --
    def start_learning(self) -> None:
        self.trainer = self._create_trainer()

    def run_epoch(self) -> None:
        if self.trainer is None:
            raise RuntimeError("'run_epoch' called before initializing the trainer.")
        self.trainer.run_epoch()

    def save_state(self) -> None:
        if self.trainer is None:
            raise RuntimeError("'save_state' called before initializing the trainer.")
        with BytesIO() as ofs:
            self.trainer.save_state(ofs)
            self.best_state = ofs.getvalue()

    def load_state(self) -> None:
        if self.trainer is None:
            raise RuntimeError("'load_state' called before initializing the trainer.")
        if self.best_state is None:
            raise RuntimeError("'load_state' called before achieving any results.")
        with BytesIO(self.best_state) as ifs:
            self.trainer.load_state(ifs)

    def learn(self) -> "IALSRecommender":  # base.py:119-126
        self.learn_with_optimizer(None, None, max_epoch=self.train_epochs)
        return self

    def learn_with_optimizer(self, evaluator: Any, trial: Any = None, max_epoch: int = 128,
                             validate_epoch: int = 5, score_degradation_max: int = 5) -> None:
        """Epoch loop with validation-based early stopping (base_earlystop.py:106-149).
        ``trial`` (Optuna pruning) is accepted only as ``None``."""
        if trial is not None:
            raise NotImplementedError("Optuna pruning is outside the B200 hot path")
        self.start_learning()
        best_score = -float("inf")
        n_score_degradation = 0
        for epoch in range(max_epoch):
            self.run_epoch()
            if (epoch + 1) % validate_epoch or evaluator is None:
                continue
            target_score = evaluator.get_target_score(self)
            if target_score > best_score:
                best_score = target_score
                self.save_state()
                self.learnt_config["train_epochs"] = epoch + 1
                n_score_degradation = 0
            else:
                n_score_degradation += 1
                if n_score_degradation >= score_degradation_max:
                    break
        if evaluator is not None:
            self.load_state()

    @property
    def trainer_as_ials(self) -> IALSTrainer:
        if self.trainer is None:
            raise RuntimeError("tried to fetch trainer before the training.")
        return self.trainer

    # -- scoring --
    def get_score(self, user_indices: np.ndarray) -> np.ndarray:  # ials.py:477-481
        """Scores of arbitrary users.  (The reference does this one in numpy on the
        host; here a contiguous range goes through the GEMM kernel and a general
        index set is gathered block by block.)"""
        user_indices = np.asarray(user_indices)
        if user_indices.dtype == bool:
            user_indices = np.flatnonzero(user_indices)
        user_indices = user_indices.astype(np.int64)
        if user_indices.size == 0:
            return np.empty((0, self.n_items), dtype=np.float32)
        user_indices = np.where(user_indices < 0, user_indices + self.n_users, user_indices)
        if user_indices.min() < 0 or user_indices.max() >= self.n_users:
            raise IndexError("user index out of range")
        if np.all(np.diff(user_indices) == 1):
            return self.get_score_block(int(user_indices[0]), int(user_indices[-1]) + 1)
        if user_indices.size >= self._GATHER_MIN_ROWS:
            # a large arbitrary index set (e.g. IDMapper.recommend_for_known_user_batch): gather
            # the embeddings once and score them with ONE device GEMM instead of a launch, a
            # read-back and a synchronisation per user
            return self._score_embeddings(self.get_user_embedding()[user_indices])
        out = np.empty((user_indices.size, self.n_items), dtype=np.float32)
        for pos, u in enumerate(user_indices):
            out[pos] = self.get_score_block(int(u), int(u) + 1)[0]
        return out

    _GATHER_MIN_ROWS = 64

    def _score_embeddings(self, user_embedding: np.ndarray) -> np.ndarray:
        """``user_embedding @ item.T`` on the device (tcgen05 3xTF32 GEMM of ``user_scores``):
        a factors-only trainer over the given rows and this model's item factors."""
        core = self.trainer_as_ials.core_trainer
        emb = np.ascontiguousarray(user_embedding, dtype=np.float32)
        if emb.ndim != 2 or emb.shape[1] != core.K:
            raise ValueError("embedding must be (n, n_components)")
        if emb.shape[0] == 0:
            return np.empty((0, self.n_items), dtype=np.float32)
        tmp = type(core)._from_factors(core._config, emb, core.item)
        return tmp.user_scores(0, emb.shape[0], self.trainer_as_ials.solver_config)

    def get_score_block(self, begin: int, end: int) -> np.ndarray:  # ials.py:483-484
        return self.trainer_as_ials.user_scores(begin, end)

    def get_score_remove_seen(self, user_indices: np.ndarray) -> np.ndarray:  # base.py:308-322
        scores = self.get_score(user_indices)
        m = self.X_train_all[user_indices].tocsr()
        scores[m.nonzero()] = -np.inf
        return scores

    def get_score_remove_seen_block(self, begin: int, end: int) -> np.ndarray:  # base.py:324-337
        scores = self.get_score_block(begin, end)
        m = self.X_train_all[begin:end]
        scores[m.nonzero()] = -np.inf
        return scores

    def recommend_block(self, begin: int, end: int, cutoff: int, mask: Any = "train",
                        allowed: Any = None):
        """B200 extension: fused score GEMM + seen mask + top-``cutoff`` for users
        ``[begin, end)``; only indices come back (what ``Evaluator`` consumes).
        With ``mask="train"`` the mask is ``X_train_all[begin:end].nonzero()``.
        ``allowed``: ``(n_lists, indptr, indices)``, the recommendable items as one shared
        or one per-user strictly ascending list (``IALSTrainer.recommend``)."""
        return self.trainer_as_ials.core_trainer.recommend(begin, end, cutoff, mask=mask,
                                                           allowed=allowed)

    def recommend_users(self, user_indices: Any, cutoff: int, mask: Any = "train",
                        allowed: Any = None, return_scores: bool = True):
        """B200 extension, ``recommend_block`` for users picked by index (serving:
        ``IDMapper.recommend_for_known_user_batch``): (indices, counts, scores)."""
        u = np.asarray(user_indices, dtype=np.int64).reshape(-1)
        u = np.where(u < 0, u + self.n_users, u)
        return self.trainer_as_ials.core_trainer.recommend_users(
            u, cutoff, mask=mask, return_scores=return_scores, allowed=allowed)

    def _similar(self, side: int, indices: Any, cutoff: int, **kw: Any):
        n = self.n_users if side == 0 else self.n_items
        if indices is not None:  # negative and boolean indices as get_score takes them
            indices = np.asarray(indices)
            if indices.dtype == bool:
                indices = np.flatnonzero(indices)
            indices = indices.astype(np.int64).reshape(-1)
            indices = np.where(indices < 0, indices + n, indices)
        return self.trainer_as_ials.core_trainer.similar(side, indices, cutoff, **kw)

    def get_similar_items(self, item_indices: Any, cutoff: int = 10, metric: str = "cosine",
                          exclude_self: bool = True, forbidden: Any = None, allowed: Any = None,
                          return_scores: bool = True):
        """B200 extension: the ``cutoff`` items most similar to each of ``item_indices`` (None: every
        item) in the item factor space, on the device (``IALSTrainer.similar``, side 1):
        (indices, counts, scores)."""
        return self._similar(1, item_indices, cutoff, metric=metric, exclude_self=exclude_self,
                             forbidden=forbidden, allowed=allowed, return_scores=return_scores)

    def get_similar_users(self, user_indices: Any, cutoff: int = 10, metric: str = "cosine",
                          exclude_self: bool = True, forbidden: Any = None, allowed: Any = None,
                          return_scores: bool = True):
        """B200 extension: the ``cutoff`` users most similar to each of ``user_indices`` (None: every
        user) in the user factor space (``IALSTrainer.similar``, side 0): (indices, counts, scores)."""
        return self._similar(0, user_indices, cutoff, metric=metric, exclude_self=exclude_self,
                             forbidden=forbidden, allowed=allowed, return_scores=return_scores)

    def _user_index_array(self, user_indices: Any) -> np.ndarray:
        """Negative and boolean user indices as ``get_score`` takes them."""
        u = np.asarray(user_indices)
        if u.dtype == bool:
            u = np.flatnonzero(u)
        u = u.astype(np.int64).reshape(-1)
        return np.where(u < 0, u + self.n_users, u)

    def rank_candidates(self, user_indices: Any, candidates: Any, cutoff: int = 10, mask: Any = "train",
                        return_scores: bool = True):
        """B200 extension: the best ``cutoff`` of each user's own candidate items, on the device at a cost
        that follows the number of (user, candidate) pairs (``IALSTrainer.rank_candidates``).
        ``candidates``: ``(n_lists, indptr, indices)`` or a sequence of index lists, one shared list or
        one per user.  Returns (indices, counts[, scores])."""
        return self.trainer_as_ials.core_trainer.rank_candidates(
            self._user_index_array(user_indices), candidates, cutoff, mask=mask, return_scores=return_scores)

    def rank_candidates_cold_user(self, X: Any, candidates: Any, cutoff: int = 10, mask: Any = "input",
                                  return_scores: bool = True):
        """B200 extension, the cold-user twin of ``rank_candidates``: fold the rows of ``X`` in
        (``compute_user_embedding``), then rank each row's candidates.  ``mask``: "input" (the entries of
        ``X`` itself), None, or a sparse matrix with one row per row of ``X``."""
        if isinstance(mask, str) and mask != "input":
            raise ValueError("mask must be 'input', None or a sparse matrix")
        X = sps.csr_matrix(X)
        core = self.trainer_as_ials.core_trainer
        emb = (self.compute_user_embedding(X) if X.shape[0] else np.empty((0, core.K), dtype=np.float32))
        return core.rank_candidates_embeddings(emb, candidates, cutoff, mask=X if isinstance(mask, str) else mask,
                                               return_scores=return_scores)

    def get_score_pairs(self, user_indices: Any, item_indices: Any) -> np.ndarray:
        """B200 extension: ``score[u, i]`` for each pair (``user_indices[j]``, ``item_indices[j]``),
        float32[n], computed on the device for those pairs only."""
        u = self._user_index_array(user_indices)
        i = np.asarray(item_indices, dtype=np.int64).reshape(-1)
        if u.shape != i.shape:
            raise ValueError("user_indices and item_indices must have the same length")
        i = np.where(i < 0, i + self.n_items, i)
        n = u.size
        return self.trainer_as_ials.core_trainer.candidate_scores(u, (n, np.arange(n + 1, dtype=np.int64), i))

    def explain(self, user_indices: Any, item_lists: Any, n_top: int = 10) -> Any:
        """B200 extension: why each user scores the items of their list, as the contributions of the
        user's training items to each score (``IALSTrainer.explain``; indices as ``get_score`` takes
        them).  ``item_lists``: one list of item indices per user.  Returns an ``Explanation``."""
        return self.trainer_as_ials.core_trainer.explain(0, self._user_index_array(user_indices), item_lists,
                                                         n_top)

    def explain_cold_user(self, X: Any, item_lists: Any, n_top: int = 10) -> Any:
        """B200 extension, the cold-user twin of ``explain``: the rows of ``X`` are histories of users
        who are not in the model, scaled as ``compute_user_embedding`` scales them."""
        X = self._scale_X(sps.csr_matrix(X).astype(np.float32), self.confidence_scaling, self.epsilon)
        return self.trainer_as_ials.core_trainer.explain_history(0, X, item_lists, n_top)

    def recommend_cold_block(self, X: Any, cutoff: int, mask: Any = "input", allowed: Any = None,
                             return_scores: bool = False):
        """B200 extension, the cold-user twin of ``recommend_block``: fold the rows of ``X``
        in (``compute_user_embedding``, ials.py:538-562), then score them against the item
        factors, drop ``mask`` ("input": the entries of ``X`` itself, base.py:391-403; None;
        or a sparse matrix with one row per row of ``X``) and keep the best ``cutoff`` with
        the fused kernel; ``allowed`` as in ``recommend_block``.  Returns (indices int32
        [rows, cutoff] -1 padded, counts)."""
        X = sps.csr_matrix(X)
        if X.shape[0] == 0:
            empty = (np.empty((0, cutoff), dtype=np.int32), np.empty((0,), dtype=np.int32))
            return empty + (np.empty((0, cutoff), dtype=np.float32),) if return_scores else empty
        core = self.trainer_as_ials.core_trainer  # the item factors stay where they are
        return core.recommend_embeddings(self.compute_user_embedding(X), cutoff,
                                         mask=X if isinstance(mask, str) else mask,
                                         allowed=allowed, return_scores=return_scores)

    def get_score_cold_user(self, X: Any) -> np.ndarray:  # ials.py:486-490
        return self.get_score_from_user_embedding(self.compute_user_embedding(X))

    def get_score_cold_user_remove_seen(self, X: Any) -> np.ndarray:
        scores = self.get_score_cold_user(X)
        scores[sps.csr_matrix(X).nonzero()] = -np.inf
        return scores

    def get_user_embedding(self) -> np.ndarray:  # ials.py:526-527
        return self.trainer_as_ials.core_trainer.user

    def get_item_embedding(self) -> np.ndarray:  # ials.py:535-536
        return self.trainer_as_ials.core_trainer.item

    def get_score_from_user_embedding(self, user_embedding: np.ndarray) -> np.ndarray:
        """ials.py:529-533 (numpy ``user_embedding.dot(item.T)`` there): the device GEMM here."""
        return self._score_embeddings(user_embedding)

    def get_score_from_item_embedding(self, user_indices: np.ndarray,
                                      item_embedding: np.ndarray) -> np.ndarray:
        """ials.py:629-636: scores of known users against arbitrary item embeddings."""
        core = self.trainer_as_ials.core_trainer
        users = np.ascontiguousarray(self.get_user_embedding()[user_indices], dtype=np.float32)
        items = np.ascontiguousarray(item_embedding, dtype=np.float32)
        if items.ndim != 2 or items.shape[1] != core.K:
            raise ValueError("item_embedding must be (n, n_components)")
        if users.shape[0] == 0 or items.shape[0] == 0:
            return np.empty((users.shape[0], items.shape[0]), dtype=np.float32)
        tmp = type(core)._from_factors(core._config, users, items)
        return tmp.user_scores(0, users.shape[0], self.trainer_as_ials.solver_config)

    def compute_user_embedding(self, X: Any, user_features: Any = None) -> np.ndarray:  # ials.py:538-562
        return self.trainer_as_ials.transform_user(
            self._scale_X(sps.csr_matrix(X).astype(np.float32), self.confidence_scaling,
                          self.epsilon), user_features=user_features)

    def compute_user_embedding_from_features(self, user_features: Any) -> np.ndarray:  # ials.py:564-575
        X = sps.csr_matrix((user_features.shape[0], self.n_items), dtype=np.float32)
        return self.compute_user_embedding(X, user_features=user_features)

    def compute_item_embedding(self, X: Any, item_features: Any = None) -> np.ndarray:  # ials.py:583-608
        return self.trainer_as_ials.transform_item(
            self._scale_X(sps.csr_matrix(X).astype(np.float32), self.confidence_scaling,
                          self.epsilon), item_features=item_features)

    def compute_item_embedding_from_features(self, item_features: Any) -> np.ndarray:  # ials.py:610-621
        X = sps.csr_matrix((self.n_users, item_features.shape[0]), dtype=np.float32)
        return self.compute_item_embedding(X, item_features=item_features)
