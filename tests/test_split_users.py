"""utils.split_users: the strong-generalisation split (held-out users, part of each history folded in). Host only."""
import numpy as np
import pytest
import scipy.sparse

from recmodel_b200 import split_users
from recmodel_b200.synthetic import make_counts, split_train_test


def test_split_users_is_the_definition():
    M = make_counts(500, 300, 12_000, seed=4)
    orig = M.copy()
    Train, FoldIn, Test, held = split_users(M.tocoo(), 60, fold_in=0.7, seed=11)
    want = np.sort(np.random.default_rng(11).choice(500, 60, replace=False))
    assert held.dtype == np.int64
    np.testing.assert_array_equal(held, want)
    rest = np.setdiff1d(np.arange(500), held)
    assert (Train != M[rest]).nnz == 0 and Train.shape == (440, 300)
    f, t = split_train_test(M[held], train=0.7, seed=11)
    assert (FoldIn != f).nnz == 0 and (Test != t).nnz == 0 and FoldIn.shape == Test.shape == (60, 300)
    assert ((FoldIn + Test) != M[held]).nnz == 0   # every held-out entry lands in exactly one half
    assert (M != orig).nnz == 0


def test_split_users_edges_and_errors():
    M = scipy.sparse.random(20, 8, density=0.3, format="csr", dtype=np.float32, random_state=0)
    Train, FoldIn, Test, held = split_users(M, 0)
    assert Train.shape == (20, 8) and FoldIn.shape == Test.shape == (0, 8) and len(held) == 0
    Train, FoldIn, Test, held = split_users(M, 20)
    assert Train.shape == (0, 8) and len(held) == 20
    for bad in (-1, 21, 2.5, True):
        with pytest.raises(ValueError):
            split_users(M, bad)
