"""SLIM (include/wmf_b200.h: wmf_slim_train): sparse non-negative item-item regression trained, scored and ranked on
the device. W and the sweep counts must equal, bit for bit, a NumPy restatement of the coordinate descent; W must be
scikit-learn's ElasticNet(positive=True) optimum where every co-occurring item is a candidate; and the scores are
ItemKNN's over the binary pattern of X."""
import numpy as np
import pytest
import scipy.sparse
import torch

from test_gpu_eval_ranking import oracle_means, oracle_per_user
from test_gpu_itemknn import (EMPTY_ITEM, EMPTY_USER, N_ITEMS, canonical, make_X, messy_csr, oracle_lists,
                              oracle_neighbors, oracle_scores, seen_lists)
from recmodel_b200 import SLIM, _lib, build, engine, ranking, utils
from recmodel_b200.synthetic import make_counts, split_train_test

gpu = pytest.mark.gpu


def pattern(X):
    P = canonical(X)
    P.data = np.ones_like(P.data)
    return P


def gram(X):
    """G = P^T P as exact int64 (SciPy)."""
    P = pattern(X).astype(np.int64)
    return (P.T @ P).tocsr()


def oracle_cd(Gs, b, l1, l2, max_iter, tol):
    """The defined loop: cyclic coordinate descent with scalar float64 steps (the q update is the same rounded
    product and difference per element)."""
    G = Gs.astype(np.float64)
    q = b.astype(np.float64).copy()
    w = np.zeros(len(b))
    for sweep in range(1, max_iter + 1):
        d = wm = 0.0
        for p in range(len(b)):
            old, gpp = float(w[p]), float(G[p, p])
            z = float(q[p]) + gpp * old
            new = (z - l1) / (gpp + l2) if z > l1 else 0.0
            if new != old:
                q -= G[:, p] * (new - old)
                w[p] = new
            d = max(d, abs(new - old))
            wm = max(wm, abs(new))
        if wm == 0.0 or d <= tol * wm:
            break
    return w, sweep


def oracle_columns(X, cols, k, l1, l2, max_iter, tol, cand=None):
    """{j: (ids, weights, sweeps)} of the definition for the columns ``cols``."""
    cand = oracle_neighbors(X, k, "cosine", 0.0) if cand is None else cand
    G = gram(X)
    out = {}
    for j in cols:
        S = cand.indices[cand.indptr[j]:cand.indptr[j + 1]].astype(np.int64)
        Gs = G[S][:, S].toarray()
        b = G[S][:, [j]].toarray().reshape(-1)
        w, sweeps = oracle_cd(Gs, b, l1, l2, max_iter, tol)
        out[j] = (S[w > 0], w[w > 0], sweeps)
    return out


def assert_columns_equal(m, want):
    Wc = m.W.tocsc()
    Wc.sort_indices()
    for j, (ids, vals, sweeps) in want.items():
        lo, hi = Wc.indptr[j], Wc.indptr[j + 1]
        np.testing.assert_array_equal(Wc.indices[lo:hi], ids, err_msg=f"column {j}")
        np.testing.assert_array_equal(Wc.data[lo:hi].view(np.uint64), vals.view(np.uint64), err_msg=f"column {j}")
        assert m.sweeps[j] == sweeps, (j, m.sweeps[j], sweeps)


def assert_same_model(a, b):
    np.testing.assert_array_equal(a.W.indptr, b.W.indptr)
    np.testing.assert_array_equal(a.W.indices, b.W.indices)
    np.testing.assert_array_equal(a.W.data.view(np.uint64), b.W.data.view(np.uint64))
    np.testing.assert_array_equal(a.sweeps, b.sweeps)


RARE_ITEMS = (1098, 1099)


@pytest.fixture(scope="module")
def data():
    """The ItemKNN tests' data (an empty user, an empty item) with two items kept to one user each: they co-occur
    with fewer than 128 items."""
    X = make_X().tocoo()
    first = {j: X.row[X.col == j].min() for j in RARE_ITEMS}
    keep = np.array([c not in first or r == first[c] for r, c in zip(X.row, X.col)])
    return scipy.sparse.csr_matrix((X.data[keep], (X.row[keep], X.col[keep])), shape=X.shape)


@pytest.fixture(scope="module")
def cands(data):
    """The candidates of the definition per k (ItemKNN cosine, shrink 0), computed once."""
    return {k: oracle_neighbors(data, k, "cosine", 0.0) for k in (1, 16, 128)}


def sample_columns(data, cand, seed):
    """A seeded sample plus the edges: item 0, the last item, the empty item, the most popular item and the items
    with the fewest candidates."""
    lens = np.diff(cand.indptr)
    pop = np.diff(canonical(data).tocsc().indptr)
    short = np.argsort(np.where(lens == 0, 10 ** 9, lens), kind="stable")[:4]
    rng = np.random.default_rng(seed)
    return sorted(set(rng.choice(N_ITEMS, 20, replace=False).tolist())
                  | {0, N_ITEMS - 1, EMPTY_ITEM, int(np.argmax(pop))} | set(short.tolist()))


CASES = [  # (l1, l2, k, max_iter, tol)
    (1.0, 10.0, 128, 100, 1e-4),
    (0.0, 5.0, 128, 100, 1e-4),
    (5.0, 0.0, 128, 100, 1e-4),
    (1e9, 1.0, 128, 100, 1e-4),   # every column is 0
    (1.0, 10.0, 1, 100, 1e-4),
    (1.0, 10.0, 16, 100, 1e-4),
    (1.0, 10.0, 128, 1, 1e-4),    # one sweep
    (1.0, 10.0, 128, 12, 0.0),    # tol 0: runs to max_iter
]


@gpu
@pytest.mark.parametrize("l1,l2,k,max_iter,tol", CASES)
def test_W_equals_the_coordinate_descent_oracle(cuda_device, data, cands, l1, l2, k, max_iter, tol):
    m = SLIM(num_items=N_ITEMS, num_users=data.shape[0])
    m.train(data, l1=l1, l2=l2, k=k, max_iter=max_iter, tol=tol)
    W = m.W
    assert isinstance(W, scipy.sparse.csr_matrix) and W.dtype == np.float64 and W.shape == (N_ITEMS, N_ITEMS)
    assert W.has_sorted_indices and np.all(W.data > 0)
    sweeps = m.sweeps
    assert sweeps.dtype == np.int32 and sweeps.shape == (N_ITEMS,) and sweeps.min() >= 1 and sweeps.max() <= max_iter
    cand = cands[k]
    # W[a, j] > 0 only for candidates a of j
    cw = scipy.sparse.csr_matrix((np.ones(cand.nnz), cand.indices, cand.indptr), shape=W.shape).T.tocsr()
    Wb = W.copy()
    Wb.data[:] = 1.0
    outside = Wb - Wb.multiply(cw)
    outside.eliminate_zeros()
    assert outside.nnz == 0
    cols = sample_columns(data, cand, seed=k + max_iter)
    assert_columns_equal(m, oracle_columns(data, cols, k, l1, l2, max_iter, tol, cand))
    assert sweeps[EMPTY_ITEM] == 1 and W[:, EMPTY_ITEM].nnz == 0 and W[EMPTY_ITEM].nnz == 0
    if l1 >= 1e9:
        assert W.nnz == 0 and np.all(sweeps == 1)
    else:
        assert W.nnz > 0
    if tol == 0.0:   # only a sweep that changes nothing (d = 0) or finds nothing to do (wm = 0) stops early
        assert np.count_nonzero(sweeps == max_iter) > N_ITEMS // 2
    if k == 128:
        lens = np.diff(cand.indptr)
        assert np.any((lens > 0) & (lens < k))   # items with fewer candidates than k


@gpu
def test_messy_input_trains_the_canonical_model(cuda_device, data, cands):
    head = messy_csr([data.indices[data.indptr[u]:data.indptr[u + 1]] for u in range(200)], (200, N_ITEMS), seed=1)
    X = scipy.sparse.vstack([head, data[200:]], format="csr")
    X.has_sorted_indices = False
    before = (X.indptr.copy(), X.indices.copy(), X.data.copy())
    a = SLIM(num_items=N_ITEMS, num_users=X.shape[0])
    a.train(X, l1=0.5, l2=4.0, k=64)
    for arr, old in zip((X.indptr, X.indices, X.data), before):   # the caller's matrix is untouched
        np.testing.assert_array_equal(arr, old)
    b = SLIM(num_items=N_ITEMS, num_users=X.shape[0])
    b.train(canonical(X), l1=0.5, l2=4.0, k=64)
    assert_same_model(a, b)
    cols = sample_columns(X, oracle_neighbors(X, 64, "cosine", 0.0), seed=5)
    assert_columns_equal(a, oracle_columns(X, cols, 64, 0.5, 4.0, 100, 1e-4))


@gpu
def test_determinism(cuda_device, data):
    runs = []
    for _ in range(2):
        m = SLIM(num_items=N_ITEMS, num_users=data.shape[0])
        m.train(data, l1=0.2, l2=3.0, tol=1e-8)
        runs.append(m)
    assert_same_model(runs[0], runs[1])


@gpu
@pytest.mark.parametrize("l1,l2", [(1.0, 10.0), (5.0, 2.0)])
def test_same_optimum_as_scikit_learn(cuda_device, l1, l2):
    """100 items, k = 128: every item that co-occurs with j is a candidate, so W is full SLIM and each column is the
    ElasticNet(positive=True) solution on P with column j zeroed."""
    from sklearn.linear_model import ElasticNet
    X = make_counts(400, 100, 4000, seed=21, planted_rank=4)
    P = pattern(X).toarray().astype(np.float64)
    users = P.shape[0]
    m = SLIM(num_items=100, num_users=users)
    m.train(X, l1=l1, l2=l2, k=128, max_iter=100_000, tol=1e-13)
    W = m.W.toarray()
    assert np.count_nonzero(W) > 0
    for j in range(100):
        A = P.copy()
        A[:, j] = 0.0
        en = ElasticNet(alpha=(l1 + l2) / users, l1_ratio=l1 / (l1 + l2), positive=True, fit_intercept=False,
                        tol=1e-14, max_iter=1_000_000)
        en.fit(A, P[:, j])
        want, got = en.coef_, W[:, j]
        assert np.linalg.norm(got - want) <= 1e-8 * max(np.linalg.norm(want), 1e-300) or \
            (not want.any() and not got.any()), (j, np.linalg.norm(got - want), np.linalg.norm(want))


@gpu
def test_kkt_conditions(cuda_device, data, cands):
    """Each column's restricted problem: with g = G_S w - b, g_p + l1 + l2 w_p = 0 where w_p > 0 and g_p + l1 >= 0
    where w_p = 0, to the accuracy the stopping rule allows."""
    l1, l2 = 2.0, 8.0
    m = SLIM(num_items=N_ITEMS, num_users=data.shape[0])
    m.train(data, l1=l1, l2=l2, k=128, max_iter=10_000, tol=1e-12)
    G = gram(data)
    Wc = m.W.tocsc()
    cand = cands[128]
    for j in range(N_ITEMS):
        S = cand.indices[cand.indptr[j]:cand.indptr[j + 1]]
        if len(S) == 0:
            continue
        Gs = G[S][:, S].toarray().astype(np.float64)
        b = G[S][:, [j]].toarray().reshape(-1).astype(np.float64)
        w = np.asarray(Wc[:, j].toarray()).reshape(-1)[S]
        g = Gs @ w - b
        scale = 1e-7 * (np.abs(b).max() + l1)
        on = w > 0
        assert np.all(np.abs(g[on] + l1 + l2 * w[on]) <= scale), j
        assert np.all(g[~on] + l1 >= -scale), j


@gpu
def test_scale_past_2_31_gram_entries(cuda_device):
    """50 000 items: G has 2.5e9 entries, so every row a >= 42 950 starts past 2^31 (64-bit offsets)."""
    n = 50_000
    X = make_counts(20_000, n, 400_000, seed=5, planted_rank=6)
    m = SLIM(num_items=n, num_users=X.shape[0])
    m.train(X, l1=0.5, l2=5.0, k=32)
    assert m.W.shape == (n, n) and m.W.nnz > 0
    cand = oracle_neighbors(X, 32, "cosine", 0.0)
    rng = np.random.default_rng(7)
    lens = np.diff(cand.indptr)
    high = np.flatnonzero(lens[45_000:] > 3) + 45_000
    cols = sorted(set(rng.choice(high, 12, replace=False).tolist()) | {int(high[-1])}
                  | set(rng.choice(n, 4, replace=False).tolist()))
    assert_columns_equal(m, oracle_columns(X, cols, 32, 0.5, 5.0, 100, 1e-4, cand))


@pytest.fixture(scope="module")
def trained(data):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    m = SLIM(num_items=N_ITEMS, num_users=data.shape[0])
    m.train(data, l1=0.5, l2=5.0)
    W = m.W
    P = pattern(data)
    S = np.stack([oracle_scores(P, W, u) for u in range(data.shape[0])])
    return m, data, W, S


@gpu
def test_predict_is_the_oracle_score(cuda_device, trained):
    m, X, W, S = trained
    rng = np.random.default_rng(0)
    users = np.concatenate([rng.integers(0, X.shape[0], 4000), [EMPTY_USER] * 10])
    items = rng.integers(0, N_ITEMS, len(users))
    got = m.predict(users, items)
    assert got.dtype == np.float64
    np.testing.assert_array_equal(got.view(np.uint64), S[users, items].view(np.uint64))
    assert np.any(got > 0) and np.all(m.predict(EMPTY_USER, np.arange(N_ITEMS)) == 0)
    np.testing.assert_array_equal(m.predict(3, np.arange(N_ITEMS)).view(np.uint64), S[3].view(np.uint64))


@gpu
@pytest.mark.parametrize("topn", [1, 100, N_ITEMS])
def test_recommend_equals_the_oracle(cuda_device, trained, topn):
    m, X, W, S = trained
    n_users = X.shape[0]
    seen = seen_lists(n_users, seed=topn)
    Ex = messy_csr(seen, (n_users, N_ITEMS), seed=topn)
    users = np.concatenate([np.random.default_rng(topn).permutation(n_users), [EMPTY_USER, 3, 0]])
    got = m.recommend(users, topn, exclude=Ex)
    assert got.dtype == np.int64 and got.shape == (len(users), topn)
    np.testing.assert_array_equal(got, oracle_lists(S, users, seen, topn))
    assert np.all(got[users == 3] == -1)
    if topn >= 100:
        assert np.any(got[users % 5 == 2] == -1)


@gpu
def test_eval_ranking_equals_the_definitions_in_any_chunking(cuda_device, monkeypatch):
    ks = [10, 50, 5]
    full = make_counts(2000, N_ITEMS, 60_000, seed=8, planted_rank=6)
    Train, Test = split_train_test(full)
    m = SLIM(num_items=N_ITEMS, num_users=2000)
    m.train(Train, k=64)
    users = np.flatnonzero(np.diff(Test.indptr) > 0)
    ids = m.recommend(users, max(ks), exclude=Train)
    want = oracle_per_user(ids, users, Test, ks)
    res = m.eval_ranking(Test, topn=ks, exclude=Train)
    means = oracle_means(want, ks)
    assert res["users"] == means["users"] == len(users) and set(res) == set(means)
    for key in means:
        np.testing.assert_allclose(res[key], means[key], rtol=1e-12, atol=1e-15)
    assert res["Recall@50"] > 0
    real, calls = engine.topn_metrics, []
    monkeypatch.setattr(engine, "topn_metrics", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    monkeypatch.setattr(ranking, "EVAL_CHUNK_IDS", 1)
    assert m.eval_ranking(Test, topn=ks, exclude=Train) == res
    assert len(calls) == len(users)   # chunks of 1 user


@gpu
def test_coverage_equals_the_per_user_loop(cuda_device):
    full = make_counts(1500, N_ITEMS, 40_000, seed=12, planted_rank=6)
    m = SLIM(num_items=N_ITEMS, num_users=1500)
    m.train(full, k=32)

    class LoopOnly:
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    got = utils.test_coverage(m, full, 10)
    np.testing.assert_array_equal(got, utils.test_coverage(LoopOnly(), full, 10))
    assert got.sum() > 0


@gpu
def test_W_setter_round_trips(cuda_device, trained, data):
    m, X, W, S = trained
    other = SLIM(num_items=N_ITEMS, num_users=X.shape[0])
    other.train(data, k=8)
    assert other.sweeps is not None
    other.W = W.tocoo()
    assert other.sweeps is None
    got = other.W
    np.testing.assert_array_equal(got.indptr, W.indptr)
    np.testing.assert_array_equal(got.indices, W.indices)
    np.testing.assert_array_equal(got.data.view(np.uint64), W.data.view(np.uint64))
    np.testing.assert_array_equal(other.recommend(np.arange(50), 20), m.recommend(np.arange(50), 20))
    with pytest.raises(ValueError):
        other.W = scipy.sparse.csr_matrix((N_ITEMS, N_ITEMS + 1))
    other.W = scipy.sparse.identity(N_ITEMS - 1, format="csr")
    with pytest.raises(ValueError):
        other.recommend(np.arange(3), 10)


@gpu
def test_input_errors(cuda_device, data):
    fresh = SLIM(num_items=N_ITEMS, num_users=data.shape[0])
    for call in (lambda: fresh.recommend(np.arange(3), 10), lambda: fresh.eval_ranking(data),
                 lambda: fresh.predict([0], [0])):
        with pytest.raises(ValueError):
            call()
    assert fresh.sweeps is None
    bad = ({"l1": -1.0}, {"l1": float("nan")}, {"l1": float("inf")}, {"l2": -0.5}, {"l2": float("inf")},
           {"k": 0}, {"k": 129}, {"k": 2.5}, {"k": True}, {"max_iter": 0}, {"max_iter": 1.5},
           {"tol": -1e-9}, {"tol": float("nan")}, {"tol": float("inf")})
    for kwargs in bad:
        with pytest.raises(ValueError):
            fresh.train(data, **kwargs)
    assert fresh._X is None


def test_slim_entry_points_reject_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call
    need = lib.wmf_slim_train_workspace_bytes(1000, 100)
    assert need >= 1000 * 1000 * 4 + 1000 * 100 * 12
    for n, k in ((0, 100), (-1, 100), ((1 << 30) + 1, 100), (1000, 0), (1000, 129), (1000, -1)):
        assert lib.wmf_slim_train_workspace_bytes(n, k) == 0
    assert lib.wmf_slim_train_workspace_bytes(50, 128) >= 50 * 50 * 4 + 50 * 50 * 12

    def train(xp=p, xi=p, rows=50, xtp=p, xti=p, n=1000, cp=p, ci=p, k=100, l1=1.0, l2=10.0, max_iter=100, tol=1e-4,
              wp=p, wi=p, wd=p, sw=p, ws=p, ws_bytes=need):
        return lib.wmf_slim_train(xp, xi, rows, xtp, xti, n, cp, ci, k, l1, l2, max_iter, tol, wp, wi, wd, sw, ws,
                                  ws_bytes, None)
    for n in (0, -1, (1 << 30) + 1):
        assert train(n=n) == 1 and "n=" in _lib.last_error()
    for k in (0, -1, 129):
        assert train(k=k) == 1 and "k=" in _lib.last_error()
    for name in ("l1", "l2", "tol"):
        for v in (-1e-300, float("inf"), float("nan")):
            assert train(**{name: v}) == 1 and name + "=" in _lib.last_error()
    for max_iter in (0, -5):
        assert train(max_iter=max_iter) == 1 and "max_iter" in _lib.last_error()
    assert train(rows=-1) == 1
    for name in ("xp", "xtp", "cp", "wp", "wi", "wd", "sw"):
        assert train(**{name: None}) == 1 and "null" in _lib.last_error()
    assert train(ws=None) == 2 and "workspace" in _lib.last_error()
    assert train(ws_bytes=need - 1) == 2
