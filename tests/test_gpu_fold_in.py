"""recommend_for, eval_ranking_for and WMF.fold_in (DESIGN.md 4.10): ranking users that are not rows of the training
matrix. A history folded into an item model or WMF must rank exactly like the same history as a training row; UserKNN's
neighbours of a new history (include/wmf_b200.h: wmf_userknn_fold_in) and its lists must equal a NumPy restatement of
the definitions bit for bit; WMF's fold-in must be train's user half-step, row by row, whatever rows share the call."""
import numpy as np
import pytest
import scipy.sparse
import torch

from conftest import row_rel_err
from oracle import wmf_oracle as orc
from test_gpu_ease_recommend import oracle_scores as ease_oracle_scores
from test_gpu_eval_ranking import oracle_means, oracle_per_user
from test_gpu_itemknn import EMPTY_ITEM, EMPTY_USER, N_ITEMS, canonical, make_X, messy_csr, oracle_lists
from test_gpu_itemknn import oracle_scores as item_oracle_scores
from test_gpu_userknn import oracle_scores as user_oracle_scores
from recmodel_b200 import RP3beta, SLIM, WMF, Ease, ItemKNN, UserKNN, _lib, build
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts

gpu = pytest.mark.gpu
FULL_USER = 9               # a training row holding every item
TOPNS = [1, 10, 100, 1024, 1500]   # 1500: the sort path


def rows_of(M):
    return [M.indices[M.indptr[u]:M.indptr[u + 1]] for u in range(M.shape[0])]


def messy_train():
    """make_X with FULL_USER holding every item and users 0..99 unsorted, duplicated and a third explicit zeros."""
    X = make_X()
    rows = rows_of(X)
    rows[FULL_USER] = np.arange(N_ITEMS)
    head = messy_csr(rows[:100], (100, N_ITEMS), seed=1)
    tail = scipy.sparse.csr_matrix((np.ones(sum(len(r) for r in rows[100:]), np.float32) * 2.0,
                                    np.concatenate(rows[100:]).astype(np.int32),
                                    np.concatenate([[0], np.cumsum([len(r) for r in rows[100:]])])),
                                   shape=(X.shape[0] - 100, N_ITEMS))
    Xm = scipy.sparse.vstack([head, tail], format="csr")
    Xm.has_sorted_indices = False
    return Xm


def new_histories(n, seed):
    """n histories that are not training rows: random, plus an empty row (0), every item (1) and one messy row (2)."""
    rng = np.random.default_rng(seed)
    rows = [rng.choice(N_ITEMS, size=int(rng.integers(1, 120)), replace=False) for _ in range(n)]
    rows[0] = np.empty(0, np.int64)
    rows[1] = np.arange(N_ITEMS)
    return messy_csr(rows, (n, N_ITEMS), seed=seed)


@pytest.fixture(scope="module")
def item_models():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    X = messy_train()
    out = {}
    for name, m, kw in (("Ease", Ease(N_ITEMS, X.shape[0]), {"alpha": 100.0, "verbose": 0, "cores": 1}),
                        ("ItemKNN", ItemKNN(N_ITEMS, X.shape[0]), {"k": 100, "shrink": 5.0}),
                        ("SLIM", SLIM(N_ITEMS, X.shape[0]), {"k": 32}),
                        ("RP3beta", RP3beta(N_ITEMS, X.shape[0]), {})):
        m.train(X, **kw)
        out[name] = m
    return X, out


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape
    np.testing.assert_array_equal(a.view(np.uint64 if a.dtype == np.float64 else np.uint32),
                                  b.view(np.uint64 if b.dtype == np.float64 else np.uint32))


@gpu
@pytest.mark.parametrize("topn", TOPNS)
@pytest.mark.parametrize("name", ["Ease", "ItemKNN", "SLIM", "RP3beta"])
def test_item_model_fold_in_of_a_training_row_is_recommend(cuda_device, item_models, name, topn):
    X, models = item_models
    m = models[name]
    rows = np.concatenate([[EMPTY_USER, FULL_USER], np.arange(0, 100, 3), np.arange(100, X.shape[0], 29)])
    Q = X[rows]
    np.testing.assert_array_equal(m.recommend_for(Q, topn), m.recommend(rows, topn, exclude=X))
    np.testing.assert_array_equal(m.recommend_for(Q, topn, exclude=None), m.recommend(rows, topn))
    if topn <= _lib.TOPK_MAX:   # the scores inside the two lists, bit for bit
        Xq, Wq = m._fold_in(Q)
        got = m._score_topk(Xq, Wq, torch.arange(len(rows), device=cuda_device), topn,
                            exclude=DeviceCSR.from_scipy(Q, cuda_device), want_scores=True)
        want = m._score_topk(*m._X_and_W(), torch.from_numpy(rows).to(cuda_device), topn,
                             exclude=DeviceCSR.from_scipy(X, cuda_device), want_scores=True)
        np.testing.assert_array_equal(got[0].cpu().numpy(), want[0].cpu().numpy())
        same_bits(got[1].cpu().numpy(), want[1].cpu().numpy())


@gpu
@pytest.mark.parametrize("topn", [10, 1500])
@pytest.mark.parametrize("name", ["Ease", "ItemKNN", "SLIM", "RP3beta"])
def test_item_model_new_rows_equal_the_definitions(cuda_device, item_models, name, topn):
    X, models = item_models
    m = models[name]
    Q = new_histories(40, seed=11)
    if name == "Ease":
        Qp, W = Q.copy().tocsr(), m.W
        S = np.stack([ease_oracle_scores(Qp, W, r) for r in range(Q.shape[0])])
    else:
        Qp = canonical(Q)
        if name != "ItemKNN":
            Qp.data[:] = 1.0
        W = m.neighbors if name == "ItemKNN" else m.W
        S = np.stack([item_oracle_scores(Qp, W, r) for r in range(Q.shape[0])])
    seen = rows_of(Q)
    np.testing.assert_array_equal(m.recommend_for(Q, topn), oracle_lists(S, range(Q.shape[0]), seen, topn))
    none = [np.empty(0, np.int64)] * Q.shape[0]
    np.testing.assert_array_equal(m.recommend_for(Q, topn, exclude=None),
                                  oracle_lists(S, range(Q.shape[0]), none, topn))
    other = scipy.sparse.csr_matrix((np.ones(Q.shape[0]), (np.arange(Q.shape[0]), np.arange(Q.shape[0]) % 7)),
                                    shape=Q.shape)
    np.testing.assert_array_equal(m.recommend_for(Q, topn, exclude=other),
                                  oracle_lists(S, range(Q.shape[0]), rows_of(other), topn))


@gpu
@pytest.mark.parametrize("name", ["Ease", "ItemKNN", "SLIM", "RP3beta"])
def test_item_model_eval_ranking_for_is_eval_ranking(cuda_device, item_models, name):
    X, models = item_models
    m = models[name]
    T = make_counts(X.shape[0], N_ITEMS, 20_000, seed=5)
    ks = [100, 10, 1]
    assert m.eval_ranking_for(X, T, topn=ks) == m.eval_ranking(T, topn=ks, exclude=X)
    users = np.array([3, 3, 17, 400])
    assert m.eval_ranking_for(X, T, topn=ks, users=users) == m.eval_ranking(T, topn=ks, exclude=X, users=users)


# ---- UserKNN

U_USERS, U_ITEMS = 1200, N_ITEMS


def oracle_fold_in(Q, X, k, similarity, shrink):
    """N' of the definitions: SciPy int64 counts Q P^T, float64 similarities, neighbours by lexsort((v, -sim))."""
    def pattern(M):
        P = canonical(M)
        P.data = np.ones_like(P.data)
        return P.astype(np.int64)
    Pq, P = pattern(Q), pattern(X)
    C = (Pq @ P.T).tocsr()
    C.sort_indices()
    crr, cvv = np.diff(Pq.indptr).astype(np.float64), np.diff(P.indptr).astype(np.float64)
    rows, cols, vals = [], [], []
    for r in range(Q.shape[0]):
        v = C.indices[C.indptr[r]:C.indptr[r + 1]].astype(np.int64)
        c = C.data[C.indptr[r]:C.indptr[r + 1]].astype(np.float64)
        keep = c > 0
        v, c = v[keep], c[keep]
        if similarity == "cosine":
            s = c / (np.sqrt(crr[r]) * np.sqrt(cvv[v]) + shrink)
        elif similarity == "jaccard":
            s = c / ((crr[r] + cvv[v] - c) + shrink)
        else:
            s = c / (crr[r] + shrink)
        top = np.lexsort((v, -s))[:k]
        top = top[np.argsort(v[top])]
        rows.append(np.full(len(top), r))
        cols.append(v[top])
        vals.append(s[top])
    N = scipy.sparse.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                                shape=(Q.shape[0], X.shape[0]))
    N.sort_indices()
    return N


def device_csr_to_scipy(N, shape):
    indptr, indices, data = (t.cpu().numpy() for t in N)
    return scipy.sparse.csr_matrix((data, indices, indptr), shape=shape)


def assert_same_csr(got, want):
    np.testing.assert_array_equal(got.indptr, want.indptr)
    np.testing.assert_array_equal(got.indices, want.indices)
    same_bits(got.data, want.data)


@pytest.fixture(scope="module")
def user_data():
    X = make_X(n_users=U_USERS, n_items=U_ITEMS, nnz=50_000, seed=4)
    Q = new_histories(300, seed=12)
    return X, Q


@gpu
@pytest.mark.parametrize("k", [1, 100, 1024])
@pytest.mark.parametrize("shrink", [0.0, 10.0])
@pytest.mark.parametrize("similarity", ["cosine", "jaccard", "conditional"])
def test_userknn_fold_in_neighbours_equal_the_oracle(cuda_device, user_data, similarity, shrink, k):
    X, Q = user_data
    m = UserKNN(num_items=U_ITEMS, num_users=U_USERS)
    m.train(X, k=k, similarity=similarity, shrink=shrink)
    Xd, N = m._fold_in(Q)
    assert Xd is m._X
    assert_same_csr(device_csr_to_scipy(N, (Q.shape[0], U_USERS)), oracle_fold_in(Q, X, k, similarity, shrink))


@gpu
@pytest.mark.parametrize("similarity", ["cosine", "jaccard", "conditional"])
def test_userknn_fold_in_of_a_training_row_is_its_neighbours(cuda_device, similarity):
    X = make_X(n_users=700, n_items=900, nnz=25_000, seed=6)
    m = UserKNN(num_items=900, num_users=700)
    m.train(X, k=1024, similarity=similarity, shrink=3.0)   # k >= num_users: every candidate is kept
    rows = np.arange(0, 700, 3)
    _, N = m._fold_in(X[rows])
    got = device_csr_to_scipy(N, (len(rows), 700)).tolil()
    for r, u in enumerate(rows):
        if X.indptr[u + 1] > X.indptr[u]:
            assert got[r, u] > 0   # the row itself is its own best match under every similarity
        got[r, u] = 0
    got = got.tocsr()
    got.eliminate_zeros()
    assert_same_csr(got, m.neighbors[rows])


@gpu
@pytest.mark.parametrize("topn", [1, 10, 100, 1500])
def test_userknn_lists_equal_the_oracle(cuda_device, user_data, topn):
    X, Q = user_data
    alone = scipy.sparse.csr_matrix(([1.0], ([0], [EMPTY_ITEM])), shape=(1, U_ITEMS))   # shares no item with anyone
    Q = scipy.sparse.vstack([Q, alone], format="csr")
    m = UserKNN(num_items=U_ITEMS, num_users=U_USERS)
    m.train(X, k=50, similarity="jaccard", shrink=2.0)
    N = oracle_fold_in(Q, X, 50, "jaccard", 2.0)
    assert N.indptr[-1] == N.indptr[-2] and N.indptr[1] == N.indptr[0]   # the lone and the empty history
    Xc = canonical(X)
    S = np.stack([user_oracle_scores(Xc, N, r) for r in range(Q.shape[0])])
    np.testing.assert_array_equal(m.recommend_for(Q, topn), oracle_lists(S, range(Q.shape[0]), rows_of(Q), topn))
    got = m.recommend_for(Q, topn, exclude=None)
    np.testing.assert_array_equal(got, oracle_lists(S, range(Q.shape[0]), [np.empty(0, np.int64)] * Q.shape[0], topn))
    lowest = np.full(topn, -1)
    lowest[:min(topn, U_ITEMS)] = np.arange(min(topn, U_ITEMS))
    np.testing.assert_array_equal(got[-1], lowest)   # all scores +0.0: the lowest ids


@gpu
def test_userknn_eval_ranking_for_equals_the_oracle(cuda_device, user_data):
    X, Q = user_data
    T = make_counts(Q.shape[0], U_ITEMS, 6_000, seed=8)
    m = UserKNN(num_items=U_ITEMS, num_users=U_USERS)
    m.train(X, k=100)
    N = oracle_fold_in(Q, X, 100, "cosine", 0.0)
    Xc = canonical(X)
    S = np.stack([user_oracle_scores(Xc, N, r) for r in range(Q.shape[0])])
    ks = [20, 5]
    users = np.flatnonzero(np.diff(T.indptr) > 0)
    ids = oracle_lists(S, users, rows_of(Q), max(ks))
    want = oracle_means(oracle_per_user(ids, users, T, ks), ks)
    got = m.eval_ranking_for(Q, T, topn=ks)
    assert got["users"] == want["users"]
    for key, v in want.items():
        assert got[key] == pytest.approx(v, rel=1e-12, abs=1e-15), key
    assert m.eval_ranking_for(Q, T, topn=ks) == got   # bitwise reproducible


# ---- WMF

WMF_CASES = [  # weighted, bias, pre_process_count, preprocess_mat, f
    (True, False, "log", False, 32),
    (True, True, "log", False, 16),
    (True, False, "linear", False, 64),
    (True, True, "linear", False, 128),
    (False, False, "log", False, 16),
    (False, False, "log", True, 16),
]


def wmf_data(seed=2):
    C = make_counts(900, 700, 30_000, seed=seed, planted_rank=5)
    return C


def trained_wmf(C, weighted, bias, mode, pre, f, seed=7):
    m = WMF(num_items=C.shape[1], num_users=C.shape[0], dim=f, gamma=0.1, weighted=weighted, bias=bias, seed=seed)
    m.train(C, 1, eval_mat=C, count_mat=C, pre_process_count=mode, preprocess_mat=pre, alpha=4, beta=0.5, cores=1)
    return m


@gpu
@pytest.mark.parametrize("weighted,bias,mode,pre,f", WMF_CASES)
def test_wmf_fold_in_is_the_user_half_step_of_train(cuda_device, weighted, bias, mode, pre, f):
    C = wmf_data()
    items0 = WMF(C.shape[1], C.shape[0], f, 0.1, weighted=weighted, bias=bias, seed=7).items.copy()
    m = trained_wmf(C, weighted, bias, mode, pre, f)
    U1 = m.users.copy()
    m.items = items0                     # the factors train solved the users against
    U = m.fold_in(C)
    same_bits(U, U1)
    # one call, two calls, permuted: the same bits per row
    perm = np.random.default_rng(0).permutation(C.shape[0])
    same_bits(m.fold_in(C[perm]), U[perm])
    same_bits(np.concatenate([m.fold_in(C[:333]), m.fold_in(C[333:])]), U)
    # within the project's bar of an fp64 solve of each row's normal equations
    if weighted:
        Cp = C.astype(np.float32).tocsr(copy=True)
        Cp.data = orc.preprocess_counts(Cp.data, mode, np.float32(4), np.float32(0.5)).astype(np.float32)
        ref = (orc.half_step_bias if bias else orc.half_step)(items0.astype(np.float64), Cp, 0.1, dtype=np.float64)
    else:
        R = C.astype(np.float32).tocsr(copy=True)
        if pre:
            R.data = orc.preprocess_counts(R.data, mode, np.float32(4), np.float32(0.5)).astype(np.float32)
        ref = orc.unweighted_half_step(items0.astype(np.float64), R, 0.1, f, dtype=np.float64)
    assert row_rel_err(U, ref) < 1e-4


@gpu
def test_wmf_fold_in_on_a_fresh_model_uses_the_train_defaults(cuda_device):
    C = wmf_data(seed=3)
    fresh = WMF(C.shape[1], C.shape[0], 32, 0.1, weighted=True, seed=9)
    U = fresh.fold_in(C)
    m = WMF(C.shape[1], C.shape[0], 32, 0.1, weighted=True, seed=9)
    m.train(C, 1, eval_mat=C, count_mat=C, cores=1)
    same_bits(U, m.users)
    assert fresh.fold_in(C[:0]).shape == (0, 32)


@gpu
@pytest.mark.parametrize("topn", [1, 10, 100, 1500])
@pytest.mark.parametrize("bias", [False, True])
def test_wmf_recommend_for_is_recommend_with_the_folded_in_factors(cuda_device, bias, topn):
    C = wmf_data(seed=4)
    m = trained_wmf(C, True, bias, "log", False, 32)
    Q = C[::2]
    Q = scipy.sparse.vstack([Q, scipy.sparse.csr_matrix((1, C.shape[1]), dtype=np.float32)], format="csr")
    U = m.fold_in(Q)
    ref = WMF(C.shape[1], Q.shape[0], 32, 0.1, weighted=True, bias=bias)
    ref.items, ref.users = m.items.copy(), U
    np.testing.assert_array_equal(m.recommend_for(Q, topn), ref.recommend(np.arange(Q.shape[0]), topn, exclude=Q))
    unexcluded = np.full((Q.shape[0], topn), -1)   # recommend without exclusion is rank_batch: no -1 padding
    unexcluded[:, :min(topn, C.shape[1])] = ref.recommend(np.arange(Q.shape[0]), topn)
    np.testing.assert_array_equal(m.recommend_for(Q, topn, exclude=None), unexcluded)
    T = make_counts(Q.shape[0], C.shape[1], 5_000, seed=6)
    ks = [topn, 3] if topn != 3 else [topn]
    assert m.eval_ranking_for(Q, T, topn=ks) == ref.eval_ranking(T, topn=ks, exclude=Q)
    assert m.eval_ranking_for(Q, T, topn=ks, exclude=None) == ref.eval_ranking(T, topn=ks)


# ---- errors


@gpu
def test_input_errors(cuda_device, item_models):
    X, models = item_models
    C = wmf_data()
    w = WMF(C.shape[1], C.shape[0], 16, 0.1, weighted=True)
    uk = UserKNN(N_ITEMS, X.shape[0])
    uk.train(X, k=10)
    good = X[:20]
    T = X[:20]
    for m in list(models.values()) + [uk, w]:
        ni = N_ITEMS if m is not w else C.shape[1]
        Q = good if m is not w else C[:20]
        TT = T if m is not w else C[:20]
        bad_cols = scipy.sparse.csr_matrix((20, ni + 1), dtype=np.float32)
        bad_shape = scipy.sparse.csr_matrix((19, ni), dtype=np.float32)
        for call in (lambda: m.recommend_for(bad_cols, 10), lambda: m.recommend_for(Q.toarray(), 10),
                     lambda: m.recommend_for(Q, 10, exclude=bad_shape), lambda: m.recommend_for(Q, 10, exclude=False),
                     lambda: m.eval_ranking_for(bad_cols, TT), lambda: m.eval_ranking_for(Q, bad_shape),
                     lambda: m.eval_ranking_for(Q, TT, exclude=bad_shape), lambda: m.eval_ranking_for(Q, TT, topn=[0]),
                     lambda: m.eval_ranking_for(Q, TT, users=np.array([20]))):
            with pytest.raises(ValueError):
                call()
        assert m.recommend_for(Q, 0).shape == (20, 0)
        assert m.recommend_for(Q[:0], 10).shape == (0, 10)
    with pytest.raises(ValueError):
        w.fold_in(C[:, :-1])
    for cls in (Ease, ItemKNN, UserKNN, SLIM, RP3beta):
        fresh = cls(N_ITEMS, X.shape[0])
        for call in (lambda: fresh.recommend_for(good, 10), lambda: fresh.eval_ranking_for(good, T)):
            with pytest.raises(ValueError):
                call()


def test_userknn_fold_in_entry_rejects_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    need = lib.wmf_userknn_fold_in_workspace_bytes(100, 1000, 10)
    assert need >= 100 * 1000 * 12
    for nq, m, k in ((0, 1000, 10), (100, 0, 10), (100, 1 << 31, 10), (1 << 31, 1000, 10), (100, 1000, 0),
                     (100, 1000, 1025)):
        assert lib.wmf_userknn_fold_in_workspace_bytes(nq, m, k) == 0
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call

    def fold(qp=p, qi=p, nq=100, xtp=p, xti=p, ni=500, xp=p, m=1000, k=10, sim=0, shrink=0.0, op=p, oi=p, od=p,
             ws=p, ws_bytes=need):
        return lib.wmf_userknn_fold_in(qp, qi, nq, xtp, xti, ni, xp, m, k, sim, shrink, op, oi, od, ws, ws_bytes, None)
    for m in (0, -1, 1 << 31):
        assert fold(m=m) == 1 and "n=" in _lib.last_error()
    for k in (0, 1025):
        assert fold(k=k) == 1 and "k=" in _lib.last_error()
    assert fold(sim=3) == 1 and "similarity" in _lib.last_error()
    for shrink in (-1.0, float("inf"), float("nan")):
        assert fold(shrink=shrink) == 1 and "shrink" in _lib.last_error()
    for nq in (0, -1, 1 << 31):
        assert fold(nq=nq) == 1 and "nq=" in _lib.last_error()
    assert fold(ni=-1) == 1 and "n_items" in _lib.last_error()
    for name in ("qp", "xtp", "xp", "op", "oi", "od"):
        assert fold(**{name: None}) == 1 and "null" in _lib.last_error()
    assert fold(ws=None) == 2 and "workspace" in _lib.last_error()
    assert fold(ws_bytes=need - 1) == 2
    assert "wmf_userknn_fold_in" in (fold(ws=None) and _lib.last_error())
