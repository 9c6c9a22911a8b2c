"""RP3beta: a three-step random-walk item model trained, scored and ranked on the device (DESIGN.md 4.9).

``RP3beta(num_items, num_users)``, ``train(X, alpha, beta, k, verbose, cores)``, a settable ``W``, and from
``ItemItemModel`` ``predict``, ``rank``, ``recommend``, ``eval_ranking``, ``recommend_for`` and
``eval_ranking_for``. The walk sums, the weights, the neighbour
selection and the scores run in the kernels of csrc/knn.cu behind the C ABI; there is no CPU fallback. The powers
are per-user and per-item scalars computed on the host with NumPy, so the device only adds and multiplies and a NumPy
restatement reproduces every weight and every score bitwise (Paudel et al. 2016; Dacrema et al., RecSys 2019).
"""
import math
import time

import numpy as np
import torch

from . import _lib, engine
from .engine import DeviceCSR
from .knn_model import ItemItemModel
from .slim_model import _int_in, _pattern


def _exponent(name, v):
    v = float(v)
    if not (math.isfinite(v) and 0.0 <= v <= 2.0):
        raise ValueError(f"{name} must be finite and in [0, 2], got {v}")
    return v


def _scale(counts, exponent):
    """float64 counts^-exponent (np.power) where counts > 0, 0 elsewhere."""
    out = np.zeros(len(counts), np.float64)
    nz = counts > 0
    out[nz] = np.power(counts[nz].astype(np.float64), -exponent)
    return out


class RP3beta(ItemItemModel):

    _rows = staticmethod(_pattern)   # P: training and scores see the pattern only

    @property
    def W(self):
        """The weights as an n x n SciPy CSR (float64, sorted indices): row a holds W'_ab for the kept items b of a.
        A host copy, made on first access. Assigning any n x n SciPy matrix (canonicalised: duplicates summed,
        explicit zeros removed, indices sorted) replaces the model."""
        return self._W_host()

    @W.setter
    def W(self, value):
        self._set_W(value)

    def train(self, X, alpha=1.0, beta=0.5, k=100, verbose=0, cores=1):
        """The RP3beta weights of the users x items matrix X (any SciPy format, not modified).

        X is canonicalised on the host (CSR, duplicates summed, explicit zeros removed, sorted rows); that copy is
        kept for scoring. P is its binary pattern, deg_u the number of items of user u and pop_a the number of users
        of item a. The scales du[u] = deg_u^-alpha, ra[a] = pop_a^-alpha and cb[b] = pop_b^-beta are NumPy float64
        ``np.power`` on the host. In double, every operation rounded to nearest: S_ab = the sum over the users u of
        both a and b, ascending, from +0.0, of du[u], and W'_ab = (ra[a] S_ab) cb[b], the probability of the walk
        a -> u -> b with item popularity damped by beta (with alpha = 1 and beta = 0, P3alpha). Row a of ``W`` keeps
        the top-k items b != a with S_ab > 0 by W'_ab, ties to the lower id (fewer when a has fewer such items). The
        scores of ``predict``, ``recommend`` and ``eval_ranking`` are s(u, i) = sum over the entries j of row u of
        P, ascending, of W[j, i]. alpha and beta finite and in [0, 2], k in 1..1024. The defaults are a starting
        point, not tuned values. ``cores`` is accepted and ignored."""
        alpha = _exponent("alpha", alpha)
        beta = _exponent("beta", beta)
        k = _int_in("k", k, 1, _lib.TOPK_MAX)
        Xc = self._rows(X)
        deg = np.diff(Xc.indptr)
        pop = np.bincount(Xc.indices, minlength=Xc.shape[1])
        if verbose > 0:
            print("Compute the RP3beta weights")
            start = time.time()
        self._X = DeviceCSR.from_scipy(Xc, self.device)
        du, ra, cb = (torch.from_numpy(_scale(c, e)).to(self.device)
                      for c, e in ((deg, alpha), (pop, alpha), (pop, beta)))
        self._W_d = engine.rp3beta_train(self._X, self._X.transpose(), du, ra, cb, k)
        self._W_h = None
        if verbose > 0:
            torch.cuda.synchronize(self.device)
            print(f"Training took {time.time() - start} seconds!")
