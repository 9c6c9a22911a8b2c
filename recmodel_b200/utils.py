"""The callers on either side of the WMF path (SURVEY.md 8f N3): mirrors of
/root/reference/RecModel/utils.py with the reference's names and argument meaning.

* ``train_test_split_sparse_mat`` (utils.py:20-37): the 80/20 split with the reference's RNG semantics.
* ``test_coverage`` (utils.py:3-18): how often each item appears in the users' top-N over the items they
  have not interacted with; the ranking runs on the device in one ``recommend`` call instead of one ``rank``
  call per user.
* ``split_users``: the strong-generalisation split of Liang et al. 2018 and Steck 2019 (held-out users, part of
  each one's history folded in), the protocol of ``recommend_for`` / ``eval_ranking_for``.
"""
import numpy as np

from .synthetic import split_train_test


def train_test_split_sparse_mat(matrix, train=0.8, seed=1993):
    """[train, test] CSR halves: ``np.random.seed(seed)``, entry k (CSR data order) goes to train iff
    ``np.random.rand(nnz)[k] < train`` (utils.py:21-27). Under SciPy >= 1.15 the reference's two ``tocoo()``
    views alias the input and both halves come out empty (SURVEY.md 4, item 3); this keeps the draw and
    returns the halves the code was written to return, without touching the input."""
    return split_train_test(matrix, train=train, seed=seed)


def test_coverage(cls, Train, topN):
    """``item_counts[i]`` = number of users whose top-``topN`` over their unseen items contains item i
    (utils.py:3-18). Like the reference the result has ``Train.shape[0]`` entries (it sizes the array by the
    row count, utils.py:7). ``cls`` is any model with the RecModel ``rank``; models with ``recommend`` (WMF,
    Ease, ItemKNN, UserKNN, SLIM, RP3beta) rank every user's unseen items on the device in one call, with the stored entries of ``Train`` excluded
    there (ties are ordered by item id, as ``rank`` orders them over the ascending candidate list)."""
    Train = Train.tocsr()
    n_users, n_items = Train.shape
    item_counts = np.zeros(n_users, dtype=np.int32)
    if hasattr(cls, "recommend"):
        ranked = cls.recommend(np.arange(n_users), topN, exclude=Train)
        np.add.at(item_counts, ranked[ranked >= 0], 1)  # each row holds distinct ids: one count per (user, item)
        return item_counts
    all_items = np.arange(n_items, dtype=np.int32)
    for user in range(n_users):  # the reference's loop
        lo, hi = Train.indptr[user], Train.indptr[user + 1]
        items_to_rank = np.delete(all_items, Train.indices[lo:hi])
        ranked = np.asarray(cls.rank(users=user, items=items_to_rank, topn=topN)).reshape(-1)
        item_counts[ranked[:topN]] += 1
    return item_counts


test_coverage.__test__ = False  # a library function, not a pytest test


def split_users(matrix, held_out, fold_in=0.8, seed=1993):
    """(Train, FoldIn, Test, held): the strong-generalisation split. ``held`` is the sorted int64 ids
    ``np.random.default_rng(seed).choice(n_users, held_out, replace=False)``; ``Train`` is the CSR of the other users'
    rows, in row order; ``FoldIn`` and ``Test`` (``held_out`` rows each, row r for user ``held[r]``) are
    ``split_train_test(matrix[held], train=fold_in, seed=seed)``: the histories to fold in and the entries to predict.
    ``matrix`` is not modified."""
    matrix = matrix.tocsr()
    n_users = matrix.shape[0]
    if isinstance(held_out, (bool, np.bool_)) or not isinstance(held_out, (int, np.integer)) or not 0 <= held_out <= n_users:
        raise ValueError(f"held_out must be an int in 0..{n_users}, got {held_out!r}")
    held = np.sort(np.random.default_rng(seed).choice(n_users, int(held_out), replace=False)).astype(np.int64)
    keep = np.ones(n_users, dtype=bool)
    keep[held] = False
    fold, test = split_train_test(matrix[held], train=fold_in, seed=seed)
    return matrix[np.flatnonzero(keep)], fold, test, held
