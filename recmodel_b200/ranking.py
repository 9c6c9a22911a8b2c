"""Model-independent parts of ``recommend`` and ``eval_ranking``, shared by every model: the exact-score sort path for
lists longer than the selection kernels take, the full-ranking evaluation around a model's device ranking, and the
bodies of ``recommend_for`` / ``eval_ranking_for``, which rank users that are not rows of the training matrix from a
representation folded in from their histories (DESIGN.md 4.10). ``XWRanking`` builds these methods on them for the
models scored from a device X and a weight W (``Ease``, ``ItemKNN``, ``UserKNN``, ``SLIM``, ``RP3beta``)."""
import numpy as np
import scipy.sparse
import torch

from . import _lib, engine
from .engine import DeviceCSR

EVAL_CHUNK_IDS = 1 << 25  # eval_ranking ranks users in chunks of at most this many list entries (32 M ids, 256 MB)


def sort_path_ids(users_d, ni, k, ex, scores, cand=None):
    """Device int64 [len(users_d) x k]: each user's ni items ``items_d`` (the device int64 candidate ids ``cand``, or
    None for the items 0..ni-1) in descending order of ``scores(chunk, items_d)`` (a device [len(chunk) x ni] tensor of
    exact scores), ties to the lower position, reported as ``items_d[position]``. Only with ``cand`` None, the stored
    entries of row ``users_d[r]`` of ``ex`` (a DeviceCSR indexed by user id, or None) are moved behind every unseen
    item and reported as -1. The users are scored in chunks of at most ~16 M (user, item) pairs."""
    assert ex is None or cand is None, "exclusion is by item id: it needs the candidates 0..ni-1"
    dev = users_d.device
    rows = []
    per = max(1, (1 << 24) // ni)
    items_d = torch.arange(ni, dtype=torch.int64, device=dev) if cand is None else cand
    for u0 in range(0, users_d.numel(), per):
        chunk = users_d[u0:u0 + per]
        n = chunk.numel()
        order = torch.sort(scores(chunk, items_d), dim=1, descending=True, stable=True).indices
        if ex is None:
            rows.append(order[:, :k] if cand is None else cand[order[:, :k]])
            continue
        lo, cnt = ex.indptr[chunk], ex.indptr[chunk + 1] - ex.indptr[chunk]
        total = int(cnt.sum())
        row = torch.repeat_interleave(torch.arange(n, device=dev), cnt, output_size=total)
        entry = torch.arange(total, device=dev) + torch.repeat_interleave(lo - (torch.cumsum(cnt, 0) - cnt),
                                                                         cnt, output_size=total)
        seen = torch.zeros((n, ni), dtype=torch.bool, device=dev)
        seen[row, ex.indices[entry].long()] = True
        # unseen first, each group in score order (a seen item never displaces an unseen one, whatever the scores)
        seen_sorted = seen.gather(1, order)
        regroup = torch.sort(seen_sorted.to(torch.uint8), dim=1, stable=True).indices[:, :k]
        rows.append(torch.where(seen_sorted.gather(1, regroup), -1, order.gather(1, regroup)))
    return torch.cat(rows) if rows else torch.empty((0, k), dtype=torch.int64, device=dev)


def eval_ranking(rank_ids, dims, users_what, device, test_mat, topn, exclude, users):
    """The full-ranking evaluation of ``WMF.eval_ranking`` / ``XWRanking.eval_ranking`` (see their docstrings) for a
    model whose ``rank_ids(users_d, k, ex)`` returns the device int64 [len(users_d) x k] lists of ``recommend`` (k <= the
    number of items; ex: the exclusion DeviceCSR, or None). ``dims()`` returns (items, users) of the model, read once
    ``topn`` is valid: user ids must lie below that number of users and the rows of ``test_mat``; ``users_what`` names
    what bounds them in the error message. The users are ranked in chunks of at most ``EVAL_CHUNK_IDS`` list entries
    (``eval_ranking_sums``)."""
    ks = np.asarray(topn)
    if ks.ndim == 0:
        ks = ks.reshape(1)
    if (ks.ndim != 1 or not 1 <= len(ks) <= 16 or not np.issubdtype(ks.dtype, np.integer) or ks.min() < 1
            or len(np.unique(ks)) != len(ks)):
        raise ValueError("topn must be an int or a 1-D sequence of at most 16 distinct positive ints")
    ks = ks.astype(np.int64)
    ni, n_users = dims()
    if test_mat.shape[1] != ni:
        raise ValueError(f"test_mat has {test_mat.shape[1]} columns but the model has {ni} items")
    if exclude is not None and tuple(exclude.shape) != tuple(test_mat.shape):
        raise ValueError(f"exclude has shape {tuple(exclude.shape)}, test_mat {tuple(test_mat.shape)}")
    n_ok = min(test_mat.shape[0], n_users)
    bad_users = ValueError(f"user ids must lie in [0, {n_ok}) ({users_what})")
    if users is not None:
        users = np.ascontiguousarray(users, dtype=np.int64).reshape(-1)
        if len(users) and (users.min() < 0 or users.max() >= n_ok):
            raise bad_users
    T = (test_mat if isinstance(test_mat, DeviceCSR) else DeviceCSR.from_scipy(test_mat, device)).sorted()
    ex = None
    if exclude is not None:
        ex = exclude if isinstance(exclude, DeviceCSR) else DeviceCSR.from_scipy(exclude, device)
    if users is None:
        users_d = torch.nonzero(T.indptr[1:] > T.indptr[:-1]).squeeze(1)
        if users_d.numel() and int(users_d[-1]) >= n_ok:
            raise bad_users
    else:
        users_d = torch.from_numpy(users).to(device)
    sums = eval_ranking_sums(rank_ids, ni, T, ex, users_d, ks).cpu().numpy()
    count = int(sums[-1])
    out = {}
    for j, kk in enumerate(ks.tolist()):
        for m, name in enumerate(engine.TOPN_METRICS):
            out[f"{name}@{kk}"] = float(sums[j * 5 + m] / count) if count else float("nan")
    out["users"] = count
    return out


def eval_ranking_sums(rank_ids, ni, T, ex, users_d, ks, chunk_ids=None):
    """The device part of ``eval_ranking`` (T: the test DeviceCSR with sorted rows; ex: the exclusion DeviceCSR or
    None; ks: int64 cutoffs): the users are ranked in chunks of at most ``chunk_ids`` list entries (None:
    ``EVAL_CHUNK_IDS`` as it is at the call), each chunk's
    per-user metrics land in one buffer, and one reduce returns the device float64 [len(ks)*5 + 1] sums and the
    evaluated-user count, summed in a fixed order (bitwise reproducible). No ids leave the device."""
    device = users_d.device
    K = int(max(ks))
    k = min(K, ni)
    n = users_d.numel()
    per_user = torch.empty((n, len(ks), 5), dtype=torch.float64, device=device)
    chunk = max(1, (EVAL_CHUNK_IDS if chunk_ids is None else chunk_ids) // K)
    for u0 in range(0, n, chunk):
        part = users_d[u0:u0 + chunk]
        ids = rank_ids(part, k, ex)
        if k < K:  # cutoffs past the number of items: -1 padding, as recommend returns it
            ids = torch.cat((ids, torch.full((part.numel(), K - k), -1, dtype=torch.int64, device=device)), dim=1)
        engine.topn_metrics(ids, part, T, ks, out=per_user[u0:u0 + chunk])
    return engine.topn_metrics_reduce(per_user, len(ks))


def check_fold_in(user_items, ni, exclude, test_mat=None):
    """ValueError unless ``user_items`` is a 2-D SciPy matrix with ``ni`` columns, ``exclude`` is True, None or a matrix
    of its shape, and ``test_mat`` (when given) has its shape."""
    if not scipy.sparse.issparse(user_items) or len(user_items.shape) != 2:
        raise ValueError(f"user_items must be a 2-D SciPy sparse matrix, got {type(user_items).__name__}")
    if user_items.shape[1] != ni:
        raise ValueError(f"user_items has {user_items.shape[1]} columns but the model has {ni} items")
    shape = tuple(user_items.shape)
    if not (exclude is True or exclude is None) and tuple(getattr(exclude, "shape", ())) != shape:
        raise ValueError(f"exclude must be True, None or a matrix of the shape of user_items {shape}")
    if test_mat is not None and tuple(test_mat.shape) != shape:
        raise ValueError(f"test_mat has shape {tuple(test_mat.shape)}, user_items {shape}")


def recommend_for(fold_in, rank_ids, ni, device, user_items, topn, exclude):
    """The body of every model's ``recommend_for`` for a model of ``ni`` items: ``fold_in(user_items)`` computes the
    representation of the new rows once, and ``rank_ids(rep, users_d, k, ex)`` returns the device int64 lists of the
    rows ``users_d`` (ids into ``user_items``), k <= ni, leaving out the stored entries of row ``users_d[r]`` of ``ex``
    (a DeviceCSR, or None). ``exclude`` True excludes each row's own stored entries."""
    check_fold_in(user_items, ni, exclude)
    topn = int(topn)
    k = min(topn, ni)
    nq = user_items.shape[0]
    out = np.full((nq, topn), -1, dtype=np.int64)
    if k <= 0 or nq == 0:
        return out
    rep = fold_in(user_items)
    ex = None
    if exclude is not None:
        ex = exclude if isinstance(exclude, DeviceCSR) else DeviceCSR.from_scipy(
            user_items if exclude is True else exclude, device)
    out[:, :k] = rank_ids(rep, torch.arange(nq, dtype=torch.int64, device=device), k, ex).cpu().numpy()
    return out


def eval_ranking_for(fold_in, rank_ids, ni, device, user_items, test_mat, topn, exclude, users):
    """The body of every model's ``eval_ranking_for``: ``eval_ranking`` over the lists of ``recommend_for`` (``fold_in``
    and ``rank_ids`` as there). The representation is folded in once, when the first chunk is ranked, after every
    argument check."""
    check_fold_in(user_items, ni, exclude, test_mat)
    rep = []

    def ranked(users_d, k, ex):
        if not rep:
            rep.append(fold_in(user_items))
        return rank_ids(rep[0], users_d, k, ex)
    return eval_ranking(ranked, lambda: (ni, user_items.shape[0]), "the rows of user_items", device, test_mat, topn,
                        user_items if exclude is True else exclude, users)


class XWRanking:
    """``recommend``, ``eval_ranking``, ``recommend_for`` and ``eval_ranking_for`` of a model whose score s(u, i) is
    computed on the device from the users x items interaction matrix X and a weight W (``Ease``, ``ItemItemModel``). A
    subclass provides ``_X_and_W()`` (X as a DeviceCSR and W in the layout of its engine functions, or ValueError when
    the model cannot score), ``_score_topk(X, W, users_d, k, exclude=ex)``, the device top-k of at most
    ``_lib.TOPK_MAX`` items, ``_predict_pairs(X, W, users_d, items_d)``, the float64 scores of (user, item) pairs,
    which it ranks bitwise, and ``_fold_in(user_items)``, the (X', W') that score the rows of ``user_items`` as users
    0..len-1. The default ``_fold_in`` is (``_rows(user_items)`` on the device, W): the row preparation ``train``
    applies to X, then the trained W."""

    @property
    def device(self):
        if self._device is None:
            self._device = engine.default_device()
        return torch.device(self._device)

    def recommend(self, users, topn, exclude=None):
        """int64 [len(users) x topn]: the top-``topn`` of all items for each user, best first, leaving out the stored
        entries of row ``users[k]`` of ``exclude`` (users x items like X, any SciPy format or a DeviceCSR; every stored
        entry excludes its item whatever its value). Ties go to the lower item id, and a user with fewer than ``topn``
        unseen items gets -1 in the rest of its row. The scores are those of ``predict`` (float64, bitwise), ranked on
        the device without rounding to float32."""
        X, W = self._X_and_W()
        users = np.ascontiguousarray(users, dtype=np.int64).reshape(-1)
        if len(users) and (users.min() < 0 or users.max() >= X.shape[0]):
            raise ValueError(f"user ids must lie in [0, {X.shape[0]}) (the rows of X)")
        if exclude is not None and tuple(exclude.shape) != tuple(X.shape):
            raise ValueError(f"exclude has shape {tuple(exclude.shape)}, X {tuple(X.shape)}")
        topn = int(topn)
        k = min(topn, X.shape[1])
        out = np.full((len(users), topn), -1, dtype=np.int64)
        if k <= 0 or len(users) == 0:
            return out
        ex = None
        if exclude is not None:
            ex = exclude if isinstance(exclude, DeviceCSR) else DeviceCSR.from_scipy(exclude, self.device)
        out[:, :k] = self._recommend_ids(X, W, torch.from_numpy(users).to(self.device), k, ex).cpu().numpy()
        return out

    def _recommend_ids(self, X, W, users_d, k, ex):
        """Device int64 [len(users_d) x k], k <= num_items: the device part of ``recommend`` and ``recommend_for`` for
        the rows ``users_d`` of the device X scored with W (``ex``: a DeviceCSR with rows in any order, or None to
        exclude nothing)."""
        if k <= _lib.TOPK_MAX:
            return self._score_topk(X, W, users_d, k, exclude=ex)
        n = X.shape[1]   # very long lists: the scores of predict, then stable device sorts
        return sort_path_ids(users_d, n, k, ex, lambda chunk, items_d: self._predict_pairs(
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
            X, _ = self._X_and_W()
            if tuple(test_mat.shape) != tuple(X.shape):
                raise ValueError(f"test_mat has shape {tuple(test_mat.shape)}, X {tuple(X.shape)}")
            return X.shape[1], X.shape[0]
        return eval_ranking(lambda users_d, k, ex: self._recommend_ids(*self._X_and_W(), users_d, k, ex), dims,
                            "the rows of X", self.device, test_mat, topn, exclude, users)

    def _fold_in(self, user_items):
        _, W = self._X_and_W()
        return DeviceCSR.from_scipy(self._rows(user_items), self.device), W

    def recommend_for(self, user_items, topn, exclude=True):
        """int64 [user_items.shape[0] x topn]: ``recommend`` for users that are not rows of X. Row r is the top-``topn``
        of all items for the history in row r of ``user_items`` (new users x items, any SciPy format, in the form
        ``train`` takes X; not modified), best first, ties to the lower item id, -1 padding. The history is prepared
        as ``train`` prepares X and scored with the trained model, so a copy of row u of X gets the list and the scores
        of ``recommend([u], topn, exclude=X)``. ``exclude``: True leaves out each row's own stored entries (whatever
        their value), None nothing, a SciPy matrix or DeviceCSR of the shape of ``user_items`` its stored entries."""
        X, _ = self._X_and_W()
        return recommend_for(self._fold_in, lambda XW, users_d, k, ex: self._recommend_ids(*XW, users_d, k, ex),
                             X.shape[1], self.device, user_items, topn, exclude)

    def eval_ranking_for(self, user_items, test_mat, topn=np.array([10]), exclude=True, users=None):
        """``eval_ranking`` (the same metrics and definitions) over the lists of ``recommend_for(user_items, K,
        exclude)``, K = max(topn): the strong-generalisation protocol, where the evaluated users are not rows of X.
        ``test_mat`` has the shape of ``user_items``; ``users`` (ids into its rows) defaults to the rows of ``test_mat``
        with stored entries. The histories are folded in once per call; no list leaves the device and the result is
        bitwise reproducible."""
        X, _ = self._X_and_W()
        return eval_ranking_for(self._fold_in, lambda XW, users_d, k, ex: self._recommend_ids(*XW, users_d, k, ex),
                                X.shape[1], self.device, user_items, test_mat, topn, exclude, users)
