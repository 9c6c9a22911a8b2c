"""ItemKNN: an item-item neighbourhood model trained, scored and ranked on the device (DESIGN.md 4.6), UserKNN, its
user-user counterpart (DESIGN.md 4.8), and ``ItemItemModel``, the scoring half both share with ``SLIM``
(slim_model.py).

``ItemKNN(num_items, num_users)``, ``train(X, k, similarity, shrink, verbose, cores)``, ``predict(users, items)``,
``rank(items, users, topn)``, ``recommend`` (top-N over each user's unseen items for many users in one device call),
``eval_ranking`` (full-ranking Recall / Precision / NDCG / MAP / hit rate at N), ``recommend_for`` and
``eval_ranking_for`` (the same for users that are not rows of X, DESIGN.md 4.10) and the inherited ``eval_topn``. The
co-occurrence counts, similarities, neighbour selection and scores run in the kernels of csrc/knn.cu behind the C ABI;
there is no CPU fallback. The similarities and scores are defined exactly (``train`` and ``predict``), so a NumPy
restatement reproduces every value bitwise. ``cores`` is accepted and ignored.
"""
import math
import time

import numpy as np
import scipy.sparse
import torch

from . import _lib, engine
from .base_model import RecModel
from .engine import DeviceCSR
from .ranking import XWRanking


def _canonical(M):
    """A CSR copy with duplicates summed, explicit zeros removed and sorted column indices (M is not modified)."""
    M = scipy.sparse.csr_matrix(M, copy=True)
    M.sum_duplicates()
    M.eliminate_zeros()
    M.sort_indices()
    return M


def _check_knn_args(k, similarity, shrink):
    """shrink as a float; ValueError for an unknown similarity, a k outside 1..1024 or a shrink not finite and >= 0."""
    if similarity not in _lib.KNN_SIMILARITIES:
        raise ValueError(f"similarity must be one of {sorted(_lib.KNN_SIMILARITIES)}, got {similarity!r}")
    if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k <= _lib.TOPK_MAX:
        raise ValueError(f"k must be an int in 1..{_lib.TOPK_MAX}, got {k!r}")
    shrink = float(shrink)
    if not (math.isfinite(shrink) and shrink >= 0.0):
        raise ValueError(f"shrink must be finite and >= 0, got {shrink}")
    return shrink


class ItemItemModel(XWRanking, RecModel):
    """The scoring half shared by the item-item models (``ItemKNN``, ``SLIM``, ``RP3beta``): the canonical X and an
    n x n item weight CSR W on the device, and ``predict`` and ``rank`` over s(u, i) = sum over the entries j of row u
    of X, ascending, of x_uj * W[j, i]; ``recommend`` and ``eval_ranking`` rank these scores (``ranking.XWRanking``). A
    subclass trains W and names it (``_W_NAME``, the attribute a user sets). ``UserKNN`` scores from a users x users W
    instead: it names the axis of X whose size W must have (``_W_AXIS``) and its own engine functions."""

    _W_NAME = "W"
    _W_AXIS = 1   # W is square over the columns of X (the items)
    _score_topk = staticmethod(engine.knn_score_topk)
    _predict_pairs = staticmethod(engine.knn_predict)
    _rows = staticmethod(_canonical)   # X as train keeps it, and the new histories of recommend_for

    def __init__(self, num_items, num_users, device=None):
        self.num_items = num_items
        self.num_users = num_users
        self._device = device
        self._X = None
        self._W_d = None      # (indptr int64, indices int32, data float64) on the device
        self._W_h = None

    def _W_host(self):
        """W as an n x n SciPy CSR (float64, sorted indices), a host copy made on first access."""
        if self._W_h is None and self._W_d is not None:
            indptr, indices, data = (engine.d2h(t) for t in self._W_d)
            n = indptr.shape[0] - 1
            self._W_h = scipy.sparse.csr_matrix((data.copy(), indices.copy(), indptr.copy()), shape=(n, n))
        return self._W_h

    def _set_W(self, value):
        """Replace W by any n x n SciPy matrix (canonicalised: duplicates summed, explicit zeros removed, indices
        sorted), or drop it with None."""
        if value is None:
            self._W_h = self._W_d = None
            return
        W = _canonical(value).astype(np.float64)
        if W.shape[0] != W.shape[1]:
            raise ValueError(f"{self._W_NAME} must be square, got {W.shape}")
        self._W_h = W
        self._W_d = None

    def _W_device(self):
        if self._W_d is None and self._W_h is not None:
            W = self._W_h
            self._W_d = (torch.from_numpy(W.indptr.astype(np.int64)).to(self.device),
                         torch.from_numpy(W.indices.astype(np.int32)).to(self.device),
                         torch.from_numpy(W.data.astype(np.float64)).to(self.device))
        return self._W_d

    def _X_and_W(self):
        """(X, W) on the device; ValueError when the model is untrained or W does not fit X."""
        if self._X is None:
            raise ValueError("the model has no interaction matrix X: call train(X, ...) first")
        W = self._W_device()
        if W is None:
            raise ValueError(f"the model has no {self._W_NAME}: call train(X, ...) first")
        if W[0].numel() - 1 != self._X.shape[self._W_AXIS]:
            raise ValueError(f"{self._W_NAME} is {W[0].numel() - 1} x {W[0].numel() - 1} but X has "
                             f"{self._X.shape[self._W_AXIS]} {('users', 'items')[self._W_AXIS]}")
        return self._X, W

    def predict(self, users, items):
        """float64 s(u, i) per (user, item) pair (one user broadcasts): the sum over the entries j of row u of the
        canonical X, in ascending j, from +0.0, of (double)x_uj * W[j, i] with x_uj as float32, each product and
        each addition rounded to nearest; +0.0 when no neighbour list of u's items holds i."""
        X, W = self._X_and_W()
        users = np.atleast_1d(np.asarray(users)).astype(np.int64).reshape(-1)
        items = np.atleast_1d(np.asarray(items)).astype(np.int64).reshape(-1)
        if len(users) and (users.min() < 0 or users.max() >= X.shape[0]):
            raise ValueError(f"user ids must lie in [0, {X.shape[0]}) (the rows of X)")
        if len(items) and (items.min() < 0 or items.max() >= X.shape[1]):
            raise ValueError(f"item ids must lie in [0, {X.shape[1]})")
        if len(items) == 0:
            return np.empty(0, dtype=np.float64)
        u = torch.from_numpy(users).to(self.device)
        i = torch.from_numpy(items).to(self.device)
        return self._predict_pairs(X, W, u, i).cpu().numpy()

    def rank(self, items, users, topn=None):
        """The candidate ``items`` for one user in descending ``predict`` order, ties by candidate position; the
        first ``topn`` (all when None)."""
        items = np.asarray(items)
        scores = self.predict(np.full(1, users, dtype=np.int64), items)
        return items[np.argsort(-scores, kind="stable")][:topn]


class ItemKNN(ItemItemModel):

    _W_NAME = "neighbors"

    @property
    def neighbors(self):
        """W as an n x n SciPy CSR (float64, sorted indices): row a holds sim(a, b) for the neighbours b of a.
        A host copy, made on first access. Assigning any n x n SciPy matrix (canonicalised: duplicates summed,
        explicit zeros removed, indices sorted) replaces the model."""
        return self._W_host()

    @neighbors.setter
    def neighbors(self, value):
        self._set_W(value)

    def train(self, X, k=100, similarity="cosine", shrink=0.0, verbose=0, cores=1):
        """Neighbours of every item from the users x items matrix X (any SciPy format, not modified).

        X is canonicalised on the host (CSR, duplicates summed, explicit zeros removed, sorted rows); that copy is
        kept for scoring. With P its binary pattern, c_ab = sum_u P[u, a] P[u, b] (exact integers; c_aa is the
        popularity of a), and in double with every operation rounded to nearest:
        "cosine" c_ab / (sqrt(c_aa) sqrt(c_bb) + shrink), "jaccard" c_ab / ((c_aa + c_bb - c_ab) + shrink),
        "conditional" c_ab / (c_aa + shrink) = P(b | a) (not symmetric). The neighbours of a are the top-k items
        b != a with c_ab > 0 by sim(a, b), ties to the lower id (fewer when a has fewer such items); W[a, b] =
        sim(a, b) (``neighbors``). k in 1..1024 (k >= num_items keeps every candidate), shrink finite and >= 0."""
        shrink = _check_knn_args(k, similarity, shrink)
        Xc = self._rows(X)
        if verbose > 0:
            print("Compute the item neighbourhoods")
            start = time.time()
        self._X = DeviceCSR.from_scipy(Xc, self.device)
        self._W_d = engine.knn_train(self._X, self._X.transpose(), int(k), similarity, shrink)
        self._W_h = None
        if verbose > 0:
            torch.cuda.synchronize(self.device)
            print(f"Training took {time.time() - start} seconds!")


class UserKNN(ItemItemModel):
    """A user-user neighbourhood model (DESIGN.md 4.8): each user's top-k most similar users vote for their items."""

    _W_NAME = "neighbors"
    _W_AXIS = 0   # the neighbours are users x users
    _score_topk = staticmethod(engine.userknn_score_topk)
    _predict_pairs = staticmethod(engine.userknn_predict)

    @property
    def neighbors(self):
        """The neighbours as a num_users x num_users SciPy CSR (float64, sorted indices): row u holds sim(u, v) for
        the neighbours v of u. A host copy, made on first access. Assigning any square SciPy matrix (canonicalised:
        duplicates summed, explicit zeros removed, indices sorted) replaces the model; it must have one row per row
        of X."""
        return self._W_host()

    @neighbors.setter
    def neighbors(self, value):
        self._set_W(value)

    _fold_in_args = None   # (similarity, shrink, k) of the last train

    def _fold_in(self, user_items):
        """(X, N'): the training X and the neighbours N' among the training users of the rows of ``user_items``
        (canonicalised like X), by the similarity, shrink and k of ``train`` (DESIGN.md 4.10)."""
        X, _ = self._X_and_W()
        similarity, shrink, k = self._fold_in_args
        Q = DeviceCSR.from_scipy(self._rows(user_items), self.device)
        return X, engine.userknn_fold_in(Q, X.transpose(), X, k, similarity, shrink)

    def predict(self, users, items):
        """float64 s(u, i) per (user, item) pair (one user broadcasts): the sum over the neighbours v of u, in
        ascending v, from +0.0, of sim(u, v) * (double)x_vi with x_vi the float32 entry of the canonical X, each
        product and each addition rounded to nearest; +0.0 when no neighbour of u has i."""
        return super().predict(users, items)

    def train(self, X, k=100, similarity="cosine", shrink=0.0, verbose=0, cores=1):
        """Neighbours of every user from the users x items matrix X (any SciPy format, not modified).

        X is canonicalised on the host (CSR, duplicates summed, explicit zeros removed, sorted rows); that copy is
        kept for scoring. With P its binary pattern, c_ab = sum_i P[a, i] P[b, i] is the number of items users a and
        b share (exact integers; c_aa is the number of items of a), and the similarities are ItemKNN's, applied to
        users: in double with every operation rounded to nearest, "cosine" c_ab / (sqrt(c_aa) sqrt(c_bb) + shrink),
        "jaccard" c_ab / ((c_aa + c_bb - c_ab) + shrink), "conditional" c_ab / (c_aa + shrink) (not symmetric). The
        neighbours of u are the top-k users v != u with c_uv > 0 by sim(u, v), ties to the lower id (fewer when u has
        fewer such users); ``neighbors[u, v]`` = sim(u, v), which equals ``ItemKNN`` trained on X^T bit for bit.
        k in 1..1024 (k >= num_users keeps every candidate), shrink finite and >= 0. ``cores`` is accepted and
        ignored. ``recommend_for`` and ``eval_ranking_for`` find the neighbours of a new history among the training
        users with the same similarity, shrink and k (DESIGN.md 4.10)."""
        shrink = _check_knn_args(k, similarity, shrink)
        Xc = self._rows(X)
        if verbose > 0:
            print("Compute the user neighbourhoods")
            start = time.time()
        self._X = DeviceCSR.from_scipy(Xc, self.device)
        self._W_d = engine.knn_train(self._X.transpose(), self._X, int(k), similarity, shrink)
        self._W_h = None
        self._fold_in_args = (similarity, shrink, int(k))
        if verbose > 0:
            torch.cuda.synchronize(self.device)
            print(f"Training took {time.time() - start} seconds!")
