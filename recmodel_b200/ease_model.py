"""B200-native EASE with the reference's Python surface (SURVEY.md 8f, N4).

Mirror of /root/reference/RecModel/ease_model.py:45-114: ``Ease(num_items, num_users)``, ``train(X, alpha, verbose,
cores)``, ``predict(users, items)``, ``rank(items, users, topn)``, ``save_mat`` / ``load_mat`` and the inherited
``eval_topn``, plus ``recommend`` (top-N over each user's unseen items for many users in one device call) and
``eval_ranking`` (full-ranking Recall / Precision / NDCG / MAP / hit rate at N), as the WMF model has them. The Gram X^T X + alpha I, its dense inverse and the prediction loop of
RecModel/fast_utils/ease_utils.pyx:15-30 run in the kernels of csrc/ease.cu behind the C ABI; there is no CPU
fallback. ``cores`` is accepted and ignored (the reference only sets MKL's thread count with it).
"""
import time

import numpy as np
import torch

from . import _lib, engine, ranking
from .base_model import RecModel
from .engine import DeviceCSR

_EVAL_CHUNK_IDS = ranking.EVAL_CHUNK_IDS


class Ease(RecModel):

    def __init__(self, num_items, num_users, device=None):
        self.num_items = num_items
        self.num_users = num_users
        self._device = device
        self._W_d = None
        self._W_h = None
        self._X = None

    @property
    def device(self):
        if self._device is None:
            self._device = engine.default_device()
        return torch.device(self._device)

    # W is a plain ndarray attribute in the reference (ease_model.py:49,109): host copy on demand
    @property
    def W(self):
        if self._W_h is None and self._W_d is not None:
            self._W_h = engine.d2h(self._W_d)
        return self._W_h

    @W.setter
    def W(self, value):
        self._W_h = None if value is None else np.asarray(value, dtype=np.float32)
        self._W_d = None

    @property
    def W_device(self):
        if self._W_d is None and self._W_h is not None:
            self._W_d = torch.from_numpy(np.ascontiguousarray(self._W_h)).to(self.device)
        return self._W_d

    def _set_X(self, X):
        X_csr = X.copy().tocsr()          # ease_model.py:86: prediction needs the training interactions
        self.X_indptr = X_csr.indptr.astype(np.int32)
        self.X_idx = X_csr.indices.astype(np.int32)
        self.X_data = X_csr.data.astype(np.float32)
        self._X = DeviceCSR.from_scipy(X_csr, self.device)

    def train(self, X, alpha, verbose, cores):
        """W = P / (-diag(P) + 1e-9) with zero diagonal, P = inv(X^T X + alpha I) (ease_model.py:81-114)."""
        self._set_X(X)
        if verbose > 0:
            print("Compute the dot product")
            start = time.time()
        self._W_d = engine.ease_train(self._X, alpha)
        self._W_h = None
        if verbose > 0:
            torch.cuda.synchronize(self.device)
            print(f"Computing the inverse took {time.time() - start} seconds!")
            print("Training finished!")

    def predict(self, users, items):
        """sum_j X[user, j] W[j, item] per (user, item) pair, float64 like the reference's loop (ease_utils.pyx:15-30)."""
        users = np.atleast_1d(np.asarray(users))
        items = np.atleast_1d(np.asarray(items))
        if len(users) == 0 or len(items) == 0:
            return np.full(1, 0.0, dtype=np.float32)   # ease_utils.pyx:19-20
        u = torch.from_numpy(users.astype(np.int64)).to(self.device)
        i = torch.from_numpy(items.astype(np.int64)).to(self.device)
        return engine.ease_predict(self._X, self.W_device, u, i).cpu().numpy()

    def rank(self, items, users, topn=None):
        """Top-``topn`` of the candidate ``items`` for one user, best first (ease_model.py:51-53)."""
        items = np.asarray(items)
        predictions = self.predict(np.full(items.shape[0], users, dtype=np.int32), items.astype(np.int32))
        return items[np.argpartition(predictions, list(range(-topn, 0, 1)))[-topn:]][::-1]

    def _X_and_W(self):
        """(X, W) on the device; ValueError when the model has no interaction matrix or W does not fit it."""
        if self._X is None:
            raise ValueError("ranking needs the interaction matrix X: call train(X, ...) or load_mat(path, X=X)")
        W = self.W_device
        if W is None:
            raise ValueError("the model has no weight matrix W: call train(X, ...) or load_mat(path, X=X)")
        if W.shape[0] != self._X.shape[1]:
            raise ValueError(f"W is {W.shape[0]} x {W.shape[1]} but X has {self._X.shape[1]} items")
        return self._X, W

    def recommend(self, users, topn, exclude=None):
        """int64 [len(users) x topn]: the top-``topn`` of all items for each user, best first, leaving out the stored
        entries of row ``users[k]`` of ``exclude`` (users x items like X, any SciPy format or a DeviceCSR; every stored
        entry excludes its item whatever its value). Row k is ``rank(np.delete(np.arange(num_items), seen), users[k],
        topn)`` followed by -1 where the user has fewer than ``topn`` unseen items; ties go to the lower item id. The
        scores are those of ``predict`` (float64, bitwise), ranked on the device without rounding to float32."""
        X, W = self._X_and_W()
        n = W.shape[0]
        users = np.ascontiguousarray(users, dtype=np.int64).reshape(-1)
        if len(users) and (users.min() < 0 or users.max() >= X.shape[0]):
            raise ValueError(f"user ids must lie in [0, {X.shape[0]}) (the rows of X)")
        if exclude is not None and tuple(exclude.shape) != tuple(X.shape):
            raise ValueError(f"exclude has shape {tuple(exclude.shape)}, X {tuple(X.shape)}")
        topn = int(topn)
        k = min(topn, n)
        out = np.full((len(users), topn), -1, dtype=np.int64)
        if k <= 0 or len(users) == 0:
            return out
        ex = None
        if exclude is not None:
            ex = exclude if isinstance(exclude, DeviceCSR) else DeviceCSR.from_scipy(exclude, self.device)
        out[:, :k] = self._recommend_ids(torch.from_numpy(users).to(self.device), k, ex).cpu().numpy()
        return out

    def _recommend_ids(self, users_d, k, ex):
        """Device int64 [len(users_d) x k], k <= num_items: the device part of ``recommend`` (``ex``: a DeviceCSR with
        rows in any order, or None to exclude nothing)."""
        X, W = self._X_and_W()
        if k <= _lib.TOPK_MAX:
            return engine.ease_score_topk(X, W, users_d, k, exclude=ex)
        # very long lists: exact device scores (ease_predict, the same bits), then stable device sorts
        n = W.shape[0]
        return ranking.sort_path_ids(users_d, n, k, ex, lambda chunk, items_d: engine.ease_predict(
            X, W, chunk.repeat_interleave(n), items_d.repeat(chunk.numel())).view(chunk.numel(), n))

    def eval_ranking(self, test_mat, topn=np.array([10]), exclude=None, users=None):
        """Full-ranking quality of ``recommend``: for each cutoff k of ``topn`` (an int or at most 16 distinct positive
        ints) a dict with "Recall@k", "Precision@k", "NDCG@k", "MAP@k" and "HitRate@k" (Python floats, means over the
        evaluated users) and "users" (their number). Unlike ``eval_topn``, which ranks each held-out item against
        ``rand_sampled`` random items and divides the hits by nnz(test), this ranks ALL items and averages per user.

        The list of user u is ``recommend(users, K, exclude)`` with K = max(topn) (ties to the lower item id, -1
        padding never a hit). T_u is the set of distinct columns of row u of ``test_mat`` with a stored non-zero value
        (duplicates count once; unsorted rows and explicit zeros are fine), h_i the hits among the first i items:
        Precision@k = h_k / k (k also when the list is padded), Recall@k = h_k / |T_u|, NDCG@k = the sum of
        1/log2(i+1) over the hits at i <= k over the same sum over i <= min(k, |T_u|) (binary gains), MAP@k = the sum
        of h_i / i over the hits at i <= k over min(k, |T_u|), HitRate@k = [h_k > 0]. Users with T_u empty are ranked
        but not counted; an item both in ``exclude`` and in T_u counts in |T_u| and can never be hit.

        ``test_mat`` and ``exclude`` (None: nothing excluded) are users x items SciPy matrices or DeviceCSRs of the
        shape of X, uploaded once. ``users`` defaults to the rows of ``test_mat`` with stored entries; repeated entries
        count each time. Lists, metrics and their sums stay on the device (the per-user rows are reduced once, in a
        fixed order: the result is bitwise reproducible)."""
        def dims():
            X, W = self._X_and_W()
            if tuple(test_mat.shape) != tuple(X.shape):
                raise ValueError(f"test_mat has shape {tuple(test_mat.shape)}, X {tuple(X.shape)}")
            return W.shape[0], X.shape[0]
        return ranking.eval_ranking(lambda users_d, k, ex: self._recommend_ids(users_d, k, ex), dims, "the rows of X",
                                    self.device, test_mat, topn, exclude, users, _EVAL_CHUNK_IDS)

    def load_mat(self, path="W_mat.npy", X=None):
        try:
            self.W = np.load(path).astype(np.float32)
            print("The weight matrix was loaded succesfully!")
            if X is not None:
                self._set_X(X)
        except FileNotFoundError:
            print("The weight matrix could not be loaded!")

    def save_mat(self, path="W_mat.npy"):
        if self.W is not None:
            np.save(path, self.W)
        else:
            print("Matrix could not be saved, please fit model first!")

    def eval_topn(self, test_mat, topn, rand_sampled=1000, cores=1, random_state=1993):
        """Sampled Recall@N with the protocol of RecModel.eval_topn (base_model.py:100-148); the reference's Pool
        variant (cores > 1, ease_model.py:119-131) draws from per-process RNG states and is not reproducible, so
        every ``cores`` takes the serial protocol."""
        np.random.seed(random_state)
        return super().eval_topn(test_mat=test_mat, topn=topn, rand_sampled=rand_sampled, cores=1, random_state=random_state,
                                 dtype="float32")
