"""B200-native EASE with the reference's Python surface (SURVEY.md 8f, N4).

Mirror of /root/reference/RecModel/ease_model.py:45-114: ``Ease(num_items, num_users)``, ``train(X, alpha, verbose,
cores)``, ``predict(users, items)``, ``rank(items, users, topn)``, ``save_mat`` / ``load_mat`` and the inherited
``eval_topn``, plus ``recommend`` (top-N over each user's unseen items for many users in one device call),
``eval_ranking`` (full-ranking Recall / Precision / NDCG / MAP / hit rate at N) and their forms for users outside X,
``recommend_for`` and ``eval_ranking_for``, from ``ranking.XWRanking``, which the item-item models share. The Gram X^T X + alpha I, its dense inverse and the prediction loop of
RecModel/fast_utils/ease_utils.pyx:15-30 run in the kernels of csrc/ease.cu behind the C ABI; there is no CPU
fallback. ``cores`` is accepted and ignored (the reference only sets MKL's thread count with it).
"""
import time

import numpy as np
import torch

from . import engine
from .base_model import RecModel
from .engine import DeviceCSR
from .ranking import XWRanking


class Ease(XWRanking, RecModel):

    _score_topk = staticmethod(engine.ease_score_topk)
    _predict_pairs = staticmethod(engine.ease_predict)

    def __init__(self, num_items, num_users, device=None):
        self.num_items = num_items
        self.num_users = num_users
        self._device = device
        self._W_d = None
        self._W_h = None
        self._X = None

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

    @staticmethod
    def _rows(X):
        """The CSR the scores read for the users x items matrix X: a copy, stored order and duplicates kept
        (ease_model.py:86); ``train`` keeps it for X, ``recommend_for`` scores the new histories from it."""
        return X.copy().tocsr()

    def _set_X(self, X):
        X_csr = self._rows(X)             # ease_model.py:86: prediction needs the training interactions
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
