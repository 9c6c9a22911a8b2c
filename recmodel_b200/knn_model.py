"""ItemKNN: an item-item neighbourhood model trained, scored and ranked on the device (DESIGN.md 4.6), and
``ItemItemModel``, the scoring half it shares with ``SLIM`` (slim_model.py).

``ItemKNN(num_items, num_users)``, ``train(X, k, similarity, shrink, verbose, cores)``, ``predict(users, items)``,
``rank(items, users, topn)``, ``recommend`` (top-N over each user's unseen items for many users in one device call),
``eval_ranking`` (full-ranking Recall / Precision / NDCG / MAP / hit rate at N) and the inherited ``eval_topn``. The
co-occurrence counts, similarities, neighbour selection and scores run in the kernels of csrc/knn.cu behind the C ABI;
there is no CPU fallback. The similarities and scores are defined exactly (``train`` and ``predict``), so a NumPy
restatement reproduces every value bitwise. ``cores`` is accepted and ignored.
"""
import math
import time

import numpy as np
import scipy.sparse
import torch

from . import _lib, engine, ranking
from .base_model import RecModel
from .engine import DeviceCSR

_EVAL_CHUNK_IDS = ranking.EVAL_CHUNK_IDS


def _canonical(M):
    """A CSR copy with duplicates summed, explicit zeros removed and sorted column indices (M is not modified)."""
    M = scipy.sparse.csr_matrix(M, copy=True)
    M.sum_duplicates()
    M.eliminate_zeros()
    M.sort_indices()
    return M


class ItemItemModel(RecModel):
    """The scoring half shared by the item-item models (``ItemKNN``, ``SLIM``): the canonical X and an n x n item
    weight CSR W on the device, and ``predict``, ``rank``, ``recommend`` and ``eval_ranking`` over
    s(u, i) = sum over the entries j of row u of X, ascending, of x_uj * W[j, i]. A subclass trains W and names it
    (``_W_NAME``, the attribute a user sets)."""

    _W_NAME = "W"

    def __init__(self, num_items, num_users, device=None):
        self.num_items = num_items
        self.num_users = num_users
        self._device = device
        self._X = None
        self._W_d = None      # (indptr int64, indices int32, data float64) on the device
        self._W_h = None

    @property
    def device(self):
        if self._device is None:
            self._device = engine.default_device()
        return torch.device(self._device)

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
        if W[0].numel() - 1 != self._X.shape[1]:
            raise ValueError(f"{self._W_NAME} is {W[0].numel() - 1} x {W[0].numel() - 1} but X has "
                             f"{self._X.shape[1]} items")
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
        return engine.knn_predict(X, W, u, i).cpu().numpy()

    def rank(self, items, users, topn=None):
        """The candidate ``items`` for one user in descending ``predict`` order, ties by candidate position; the
        first ``topn`` (all when None)."""
        items = np.asarray(items)
        scores = self.predict(np.full(1, users, dtype=np.int64), items)
        return items[np.argsort(-scores, kind="stable")][:topn]

    def recommend(self, users, topn, exclude=None):
        """int64 [len(users) x topn]: the top-``topn`` of all items for each user, best first, leaving out the stored
        entries of row ``users[k]`` of ``exclude`` (users x items like X, any SciPy format or a DeviceCSR; every stored
        entry excludes its item whatever its value). Ties go to the lower item id, and a user with fewer than ``topn``
        unseen items gets -1 in the rest of its row. The scores are those of ``predict`` (float64, bitwise)."""
        X, W = self._X_and_W()
        n = X.shape[1]
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
        """Device int64 [len(users_d) x k], k <= num_items: the device part of ``recommend``."""
        X, W = self._X_and_W()
        if k <= _lib.TOPK_MAX:
            return engine.knn_score_topk(X, W, users_d, k, exclude=ex)
        n = X.shape[1]   # very long lists: the scores of predict, then stable device sorts
        return ranking.sort_path_ids(users_d, n, k, ex, lambda chunk, items_d: engine.knn_predict(
            X, W, chunk.repeat_interleave(n), items_d.repeat(chunk.numel())).view(chunk.numel(), n))

    def eval_ranking(self, test_mat, topn=np.array([10]), exclude=None, users=None):
        """Full-ranking quality of ``recommend`` with the definitions of ``Ease.eval_ranking``: for each cutoff k of
        ``topn`` (an int or at most 16 distinct positive ints) "Recall@k", "Precision@k", "NDCG@k", "MAP@k" and
        "HitRate@k" averaged over the evaluated users with a stored non-zero test entry, and "users", their number.
        ``test_mat`` and ``exclude`` are users x items matrices of the shape of X (SciPy or DeviceCSR); ``users``
        defaults to the rows of ``test_mat`` with stored entries. The sums are bitwise reproducible."""
        def dims():
            X, W = self._X_and_W()
            if tuple(test_mat.shape) != tuple(X.shape):
                raise ValueError(f"test_mat has shape {tuple(test_mat.shape)}, X {tuple(X.shape)}")
            return X.shape[1], X.shape[0]
        return ranking.eval_ranking(lambda users_d, k, ex: self._recommend_ids(users_d, k, ex), dims, "the rows of X",
                                    self.device, test_mat, topn, exclude, users, _EVAL_CHUNK_IDS)


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
        if similarity not in _lib.KNN_SIMILARITIES:
            raise ValueError(f"similarity must be one of {sorted(_lib.KNN_SIMILARITIES)}, got {similarity!r}")
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k <= _lib.TOPK_MAX:
            raise ValueError(f"k must be an int in 1..{_lib.TOPK_MAX}, got {k!r}")
        shrink = float(shrink)
        if not (math.isfinite(shrink) and shrink >= 0.0):
            raise ValueError(f"shrink must be finite and >= 0, got {shrink}")
        Xc = _canonical(X)
        if verbose > 0:
            print("Compute the item neighbourhoods")
            start = time.time()
        self._X = DeviceCSR.from_scipy(Xc, self.device)
        self._W_d = engine.knn_train(self._X, self._X.transpose(), int(k), similarity, shrink)
        self._W_h = None
        if verbose > 0:
            torch.cuda.synchronize(self.device)
            print(f"Training took {time.time() - start} seconds!")
