"""SLIM: sparse non-negative item-item regression trained, scored and ranked on the device (DESIGN.md 4.7).

``SLIM(num_items, num_users)``, ``train(X, l1, l2, k, max_iter, tol, verbose, cores)``, a settable ``W`` and
``sweeps``, and from ``ItemItemModel`` ``predict``, ``rank``, ``recommend``, ``eval_ranking``, ``recommend_for`` and
``eval_ranking_for``. The Gram, the
candidates, the coordinate descent and the scores run in the kernels of csrc/knn.cu behind the C ABI; there is no CPU
fallback. The model is this project's own definition (the reference's SLIM sources are not in this repository); its
optimum is the one scikit-learn's ``ElasticNet(positive=True)`` finds on the same problem.
"""
import math
import time

import numpy as np
import torch

from . import _lib, engine
from .engine import DeviceCSR
from .knn_model import ItemItemModel, _canonical


def _int_in(name, v, lo, hi=None):
    if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)) or v < lo or (hi is not None and v > hi):
        raise ValueError(f"{name} must be an int in {lo}..{'' if hi is None else hi}, got {v!r}")
    return int(v)


def _pattern(M):
    """The binary pattern P of the canonical M (float32 ones): what SLIM and RP3beta train on and score."""
    P = _canonical(M)
    P.data = np.ones_like(P.data, dtype=np.float32)
    return P


def _finite_nonneg(name, v):
    v = float(v)
    if not (math.isfinite(v) and v >= 0.0):
        raise ValueError(f"{name} must be finite and >= 0, got {v}")
    return v


class SLIM(ItemItemModel):

    _rows = staticmethod(_pattern)   # P: training and scores see the pattern only

    def __init__(self, num_items, num_users, device=None):
        super().__init__(num_items, num_users, device)
        self._sweeps = None

    @property
    def W(self):
        """The weights as an n x n SciPy CSR (float64, sorted indices): W[a, j] is the weight of feature item a in
        the regression of item j. A host copy, made on first access. Assigning any n x n SciPy matrix (canonicalised:
        duplicates summed, explicit zeros removed, indices sorted) replaces the model."""
        return self._W_host()

    @W.setter
    def W(self, value):
        self._set_W(value)
        self._sweeps = None

    @property
    def sweeps(self):
        """int32 [n]: the coordinate-descent sweeps each column of the last ``train`` ran (None before it, or after
        ``W`` was set)."""
        if self._sweeps is not None and not isinstance(self._sweeps, np.ndarray):
            self._sweeps = engine.d2h(self._sweeps).copy()
        return self._sweeps

    def train(self, X, l1=1.0, l2=10.0, k=128, max_iter=100, tol=1e-4, verbose=0, cores=1):
        """The SLIM weights of the users x items matrix X (any SciPy format, not modified).

        X is canonicalised on the host (CSR, duplicates summed, explicit zeros removed, sorted rows); that copy is
        kept for scoring. P is its binary pattern and G = P^T P (G[a, b] = c_ab, exact integers). The candidates S_j of
        item j are its ``ItemKNN`` cosine neighbours (shrink 0, ``k`` of them, fewer when j co-occurs with fewer
        items). Column j of W solves

            min_w 1/2 ||P[:, j] - P[:, S_j] w||^2 + l1 sum(w) + l2/2 ||w||^2   subject to w >= 0,

        which is scikit-learn's ``ElasticNet(alpha=(l1 + l2) / m, l1_ratio=l1 / (l1 + l2), positive=True,
        fit_intercept=False)`` on P with column j zeroed (m users). Items that never co-occur with j are 0 at the
        optimum, so when S_j holds every item that co-occurs with j this is full SLIM; the cap k makes it the
        feature-selected variant. The solver is cyclic coordinate descent in double on G[S_j, S_j] and G[S_j, j],
        every operation rounded to nearest, from w = 0, stopping after a sweep whose largest change is at most
        ``tol`` times the largest weight (or whose weights are all 0), or after ``max_iter`` sweeps (``sweeps``).
        W[a, j] = w_a for the candidates with w_a > 0. The scores of ``predict``, ``recommend`` and ``eval_ranking``
        are s(u, i) = sum over the entries j of row u of P, ascending, of W[j, i]. l1, l2 finite and >= 0, k in
        1..128, max_iter >= 1, tol finite and >= 0. The defaults are a starting point, not tuned values. ``cores``
        is accepted and ignored."""
        l1 = _finite_nonneg("l1", l1)
        l2 = _finite_nonneg("l2", l2)
        k = _int_in("k", k, 1, _lib.SLIM_K_MAX)
        max_iter = _int_in("max_iter", max_iter, 1, 2 ** 31 - 1)
        tol = _finite_nonneg("tol", tol)
        Xc = self._rows(X)
        if verbose > 0:
            print("Compute the SLIM weights")
            start = time.time()
        self._X = DeviceCSR.from_scipy(Xc, self.device)
        self._W_d, self._sweeps = engine.slim_train(self._X, self._X.transpose(), k, l1, l2, max_iter, tol)
        self._W_h = None
        if verbose > 0:
            torch.cuda.synchronize(self.device)
            print(f"Training took {time.time() - start} seconds!")
