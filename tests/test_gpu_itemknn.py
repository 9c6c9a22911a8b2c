"""ItemKNN (include/wmf_b200.h: wmf_knn_*): item-item neighbourhoods trained, scored and ranked on the device. The
neighbours, their similarities, predict and the scores inside recommend must equal, bit for bit, a NumPy oracle that
restates the definitions with the same double operations in the same order."""
import numpy as np
import pytest
import scipy.sparse
import torch

from test_gpu_eval_ranking import oracle_means, oracle_per_user
from recmodel_b200 import ItemKNN, _lib, build, engine, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts, split_train_test

gpu = pytest.mark.gpu
N_ITEMS = 1100
EMPTY_ITEM, EMPTY_USER = 17, 5


def canonical(X):
    X = scipy.sparse.csr_matrix(X, copy=True)
    X.sum_duplicates()
    X.eliminate_zeros()
    X.sort_indices()
    return X


def oracle_neighbors(X, k, similarity, shrink):
    """W of the definitions: SciPy int64 counts, float64 similarities, neighbours by lexsort((b, -sim))."""
    X = canonical(X)
    P = X.copy()
    P.data = np.ones_like(P.data, dtype=np.int64)
    P = P.astype(np.int64)
    C = (P.T @ P).tocsr()
    C.sort_indices()
    pop = np.diff(X.tocsc().indptr).astype(np.float64)
    n = X.shape[1]
    rows, cols, vals = [], [], []
    oracle_neighbors.tie_cuts = 0   # rows whose k-th and (k+1)-th candidates have the same similarity
    for a in range(n):
        b = C.indices[C.indptr[a]:C.indptr[a + 1]].astype(np.int64)
        c = C.data[C.indptr[a]:C.indptr[a + 1]].astype(np.float64)
        keep = (b != a) & (c > 0)
        b, c = b[keep], c[keep]
        caa, cbb = pop[a], pop[b]
        if similarity == "cosine":
            s = c / (np.sqrt(caa) * np.sqrt(cbb) + shrink)
        elif similarity == "jaccard":
            s = c / ((caa + cbb - c) + shrink)
        else:
            s = c / (caa + shrink)
        order = np.lexsort((b, -s))
        oracle_neighbors.tie_cuts += len(order) > k and s[order[k - 1]] == s[order[k]]
        top = order[:k]
        top = top[np.argsort(b[top])]
        rows.append(np.full(len(top), a))
        cols.append(b[top])
        vals.append(s[top])
    W = scipy.sparse.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    W.sort_indices()
    return W


def oracle_scores(X, W, u):
    """float64 [items]: acc[W_j.indices] += x_uj * W_j.data over the entries j of row u of the canonical X, ascending."""
    acc = np.zeros(W.shape[1], np.float64)
    for e in range(X.indptr[u], X.indptr[u + 1]):
        j = X.indices[e]
        lo, hi = W.indptr[j], W.indptr[j + 1]
        acc[W.indices[lo:hi]] += np.float64(np.float32(X.data[e])) * W.data[lo:hi]
    return acc


def oracle_lists(S, users, seen, topn):
    out = np.full((len(users), topn), -1, dtype=np.int64)
    for r, u in enumerate(users):
        s = S[u]
        cand = np.setdiff1d(np.arange(S.shape[1]), seen[u])
        best = cand[np.lexsort((cand, -s[cand]))][:topn]
        out[r, :len(best)] = best
    return out


def assert_same_W(got, want):
    np.testing.assert_array_equal(got.indptr, want.indptr)
    np.testing.assert_array_equal(got.indices, want.indices)
    np.testing.assert_array_equal(got.data.view(np.uint64), want.data.view(np.uint64))


def messy_csr(rows, shape, seed):
    """Unsorted rows, three duplicates per row, a third of the values explicit zeros: every stored entry counts."""
    rng = np.random.default_rng(seed)
    out = []
    for r in rows:
        r = rng.permutation(np.asarray(r, np.int64))
        out.append(np.concatenate([r, r[:3]]) if len(r) > 3 else r)
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in out])]).astype(np.int64)
    indices = np.concatenate(out).astype(np.int32) if out else np.empty(0, np.int32)
    data = rng.integers(0, 3, size=len(indices)).astype(np.float32)
    return scipy.sparse.csr_matrix((data, indices, indptr), shape=shape)


def make_X(n_users=3000, n_items=N_ITEMS, nnz=60_000, seed=3):
    """Counts with an empty user row and an item nobody interacted with."""
    C = make_counts(n_users, n_items, nnz, seed=seed, planted_rank=6).tocoo()
    keep = (C.row != EMPTY_USER) & (C.col != EMPTY_ITEM)
    return scipy.sparse.csr_matrix((C.data[keep], (C.row[keep], C.col[keep])), shape=C.shape)


@pytest.fixture(scope="module")
def data():
    X = make_X()
    assert X.indptr[EMPTY_USER + 1] == X.indptr[EMPTY_USER] and np.diff(X.tocsc().indptr)[EMPTY_ITEM] == 0
    return X


@pytest.fixture(scope="module")
def trained(data):
    """A cosine model (k = 100, shrink 5) whose neighbors were edited to give items 7 and 901 equal columns: an exact
    score tie for every user that votes for either."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    m = ItemKNN(num_items=N_ITEMS, num_users=data.shape[0])
    m.train(data, k=100, similarity="cosine", shrink=5.0)
    Wd = m.neighbors.toarray()
    Wd[:, 901] = Wd[:, 7]
    W = scipy.sparse.csr_matrix(Wd)
    m.neighbors = W
    S = np.stack([oracle_scores(data, W, u) for u in range(data.shape[0])])
    return m, data, W, S


@gpu
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
@pytest.mark.parametrize("shrink", [0.0, 10.0])
@pytest.mark.parametrize("similarity", ["cosine", "jaccard", "conditional"])
def test_neighbors_equal_the_oracle(cuda_device, data, similarity, shrink, k):
    m = ItemKNN(num_items=N_ITEMS, num_users=data.shape[0])
    m.train(data, k=k, similarity=similarity, shrink=shrink)
    W = m.neighbors
    assert isinstance(W, scipy.sparse.csr_matrix) and W.dtype == np.float64 and W.shape == (N_ITEMS, N_ITEMS)
    want = oracle_neighbors(data, k, similarity, shrink)
    assert_same_W(W, want)
    lengths = np.diff(W.indptr)
    assert lengths[EMPTY_ITEM] == 0 and lengths.max() <= k
    if k == 1024:
        assert 0 < lengths.min(where=np.arange(N_ITEMS) != EMPTY_ITEM, initial=k) < k   # items with fewer candidates
    if similarity == "conditional" and k <= 100:
        assert oracle_neighbors.tie_cuts > 0   # exact ties at the k-th place, kept by the lower id


@gpu
def test_training_spans_several_item_blocks(cuda_device):
    """16 500 items: the [B x n] tiles hold 508 item rows, so training runs 33 blocks."""
    X = make_X(n_users=4000, n_items=16_500, nnz=120_000, seed=4)
    for similarity, k in (("conditional", 20), ("cosine", 300)):
        m = ItemKNN(num_items=X.shape[1], num_users=X.shape[0])
        m.train(X, k=k, similarity=similarity, shrink=1.0)
        assert_same_W(m.neighbors, oracle_neighbors(X, k, similarity, 1.0))


@gpu
def test_messy_input_trains_the_canonical_model(cuda_device, data):
    head = messy_csr([data.indices[data.indptr[u]:data.indptr[u + 1]] for u in range(200)], (200, N_ITEMS), seed=1)
    X = scipy.sparse.vstack([head, data[200:]], format="csr")
    X.has_sorted_indices = False
    before = (X.indptr.copy(), X.indices.copy(), X.data.copy())
    a = ItemKNN(num_items=N_ITEMS, num_users=X.shape[0])
    a.train(X, k=50, similarity="jaccard", shrink=2.0)
    for arr, old in zip((X.indptr, X.indices, X.data), before):   # the caller's matrix is untouched
        np.testing.assert_array_equal(arr, old)
    b = ItemKNN(num_items=N_ITEMS, num_users=X.shape[0])
    b.train(canonical(X), k=50, similarity="jaccard", shrink=2.0)
    assert_same_W(a.neighbors, b.neighbors)
    assert_same_W(a.neighbors, oracle_neighbors(X, 50, "jaccard", 2.0))
    users = np.arange(300)
    for m in (a, b):
        got = m.predict(np.repeat(users, 40), np.tile(np.arange(40), len(users)))
        want = np.stack([oracle_scores(canonical(X), a.neighbors, u)[:40] for u in users]).reshape(-1)
        np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))


@gpu
def test_determinism_and_orientation(cuda_device, data):
    """Two trainings give the same bits; "conditional" is P(b | a) in row a, which differs from its transpose."""
    runs = []
    for _ in range(2):
        m = ItemKNN(num_items=N_ITEMS, num_users=data.shape[0])
        m.train(data, k=1024, similarity="conditional")
        runs.append(m.neighbors)
    assert_same_W(runs[0], runs[1])
    W = runs[0]
    assert_same_W(W, oracle_neighbors(data, 1024, "conditional", 0.0))
    X = canonical(data)
    pop = np.diff(X.tocsc().indptr)
    a = int(np.argmax(pop))
    row_a = W.indices[W.indptr[a]:W.indptr[a + 1]]
    b = next(int(b) for b in row_a if a in W.indices[W.indptr[b]:W.indptr[b + 1]] and pop[b] != pop[a])
    c = int(((X[:, a] > 0).multiply(X[:, b] > 0)).sum())
    assert c > 0 and W[a, b] == c / pop[a] and W[b, a] == c / pop[b] and W[a, b] != W[b, a]


@gpu
def test_predict_equals_the_oracle(cuda_device, trained):
    m, X, W, S = trained
    rng = np.random.default_rng(0)
    users = np.concatenate([rng.integers(0, X.shape[0], 4000), [EMPTY_USER] * 10])
    items = rng.integers(0, N_ITEMS, len(users))
    got = m.predict(users, items)
    assert got.dtype == np.float64
    want = S[users, items]
    np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))
    assert np.any(want == 0) and np.any(want > 0)       # pairs nobody votes for score +0.0
    assert np.all(got[np.signbit(got)] != 0)
    np.testing.assert_array_equal(m.predict(3, np.arange(N_ITEMS)).view(np.uint64), S[3].view(np.uint64))


def seen_lists(n_users, seed):
    """Per user: nothing, random subsets, all but 5 items (fewer unseen than topn), or everything (user 3)."""
    rng = np.random.default_rng(seed)
    seen = []
    for u in range(n_users):
        kind = u % 5
        if u == 3:
            s = np.arange(N_ITEMS)
        elif kind == 0:
            s = np.empty(0, np.int64)
        elif kind == 2:
            s = rng.choice(N_ITEMS, size=N_ITEMS - 5, replace=False)
        else:
            s = rng.choice(N_ITEMS, size=int(rng.integers(1, 200)), replace=False)
        seen.append(np.asarray(s, np.int64))
    return seen


@gpu
@pytest.mark.parametrize("topn", [1, 10, 100, 1024, N_ITEMS])
def test_recommend_equals_the_oracle(cuda_device, trained, topn):
    """8 000 listed users: more than the 7 626 of one [ub x n] score tile at 1 100 items."""
    m, X, W, S = trained
    n_users = X.shape[0]
    seen = seen_lists(n_users, seed=topn)
    Ex = messy_csr(seen, (n_users, N_ITEMS), seed=topn)
    rng = np.random.default_rng(topn)
    users = np.concatenate([rng.permutation(n_users), rng.integers(0, n_users, 5000 - 3), [EMPTY_USER, 3, 0]])
    got = m.recommend(users, topn, exclude=Ex)
    assert got.dtype == np.int64 and got.shape == (len(users), topn)
    np.testing.assert_array_equal(got, oracle_lists(S, users, seen, topn))
    assert np.all(got[users == 3] == -1)
    if topn >= 10:
        assert np.any(got[users % 5 == 2] == -1)                         # padded rows
        ties = 0
        for row in got:
            row = row.tolist()
            if 7 in row and 901 in row:
                assert row.index(7) < row.index(901)
                ties += 1
        assert topn < 100 or ties > 0
    if topn <= _lib.TOPK_MAX:
        users_d = torch.from_numpy(users).to(cuda_device)
        ex = DeviceCSR.from_scipy(Ex, cuda_device)
        ids, scores = engine.knn_score_topk(m._X, m._W_device(), users_d, topn, exclude=ex, want_scores=True)
        ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
        np.testing.assert_array_equal(ids, got)
        valid = ids >= 0
        assert np.all(np.isnan(scores[~valid]))
        pred = m.predict(np.repeat(users, topn)[valid.reshape(-1)], ids[valid])
        np.testing.assert_array_equal(scores[valid].view(np.uint64), pred.view(np.uint64))
        np.testing.assert_array_equal(scores[users == EMPTY_USER][valid[users == EMPTY_USER]].view(np.uint64), 0)


@gpu
def test_lists_independent_of_the_batch(cuda_device, trained):
    m, X, W, S = trained
    users_d = torch.arange(X.shape[0], device=cuda_device).flip(0).repeat(3)
    Ex = messy_csr(seen_lists(X.shape[0], seed=9), X.shape, seed=9)
    ex = DeviceCSR.from_scipy(Ex, cuda_device)
    for topn in (10, 300):
        ids, scores = engine.knn_score_topk(m._X, m._W_device(), users_d, topn, exclude=ex, want_scores=True)
        pieces, u0 = [], 0
        for size in (1, 7, 64, 999, 8000):
            part = users_d[u0:u0 + size]
            if part.numel():
                pieces.append(engine.knn_score_topk(m._X, m._W_device(), part, topn, exclude=ex, want_scores=True))
            u0 += size
        assert u0 >= users_d.numel()
        torch.testing.assert_close(ids, torch.cat([p[0] for p in pieces]), rtol=0, atol=0)
        np.testing.assert_array_equal(scores.cpu().numpy().view(np.uint64),
                                      torch.cat([p[1] for p in pieces]).cpu().numpy().view(np.uint64))
    np.testing.assert_array_equal(m.recommend(np.arange(X.shape[0]), 20, exclude=Ex),
                                  m.recommend(np.arange(X.shape[0]), 20, exclude=ex))


@gpu
@pytest.mark.parametrize("ks", [[10, 50, 5], [1200, 10]])    # the second: the sort path and padding past the items
def test_eval_ranking_equals_the_definitions_in_any_chunking(cuda_device, monkeypatch, ks):
    full = make_counts(2000, N_ITEMS, 60_000, seed=8, planted_rank=6)
    Train, Test = split_train_test(full)
    m = ItemKNN(num_items=N_ITEMS, num_users=2000)
    m.train(Train, k=50)
    K = max(ks)
    users = np.flatnonzero(np.diff(Test.indptr) > 0)
    ids = m.recommend(users, K, exclude=Train)
    sample = users[::97]
    Xc = canonical(Train)
    S = np.zeros((Train.shape[0], N_ITEMS))
    S[sample] = np.stack([oracle_scores(Xc, m.neighbors, u) for u in sample])
    seen = [Train.indices[Train.indptr[u]:Train.indptr[u + 1]] for u in range(Train.shape[0])]
    np.testing.assert_array_equal(ids[::97][:, :min(K, N_ITEMS)], oracle_lists(S, sample, seen, min(K, N_ITEMS)))
    want = oracle_per_user(ids, users, Test, ks)
    res = m.eval_ranking(Test, topn=ks, exclude=Train)
    means = oracle_means(want, ks)
    assert res["users"] == means["users"] == len(users) and set(res) == set(means)
    for key in means:
        np.testing.assert_allclose(res[key], means[key], rtol=1e-12, atol=1e-15)
    assert res[f"Recall@{K}"] > 0
    real, calls = engine.topn_metrics, []
    monkeypatch.setattr(engine, "topn_metrics", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    for chunk in (K * 13, 1):
        monkeypatch.setattr(ranking, "EVAL_CHUNK_IDS", chunk)
        calls.clear()
        assert m.eval_ranking(Test, topn=ks, exclude=Train) == res
        assert len(calls) == -(-len(users) // max(1, chunk // K))   # one metrics call per chunk


@gpu
def test_coverage_equals_the_per_user_loop(cuda_device):
    """utils.test_coverage takes recommend for ItemKNN and equals the reference's rank(np.delete(...)) loop: rank
    breaks ties by candidate position, which is the item id there."""
    full = make_counts(1500, N_ITEMS, 40_000, seed=12, planted_rank=6)
    m = ItemKNN(num_items=N_ITEMS, num_users=1500)
    m.train(full, k=30, similarity="jaccard")

    class LoopOnly:
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    got = utils.test_coverage(m, full, 10)
    np.testing.assert_array_equal(got, utils.test_coverage(LoopOnly(), full, 10))
    assert got.sum() > 0


@gpu
def test_rank_is_a_stable_sort_of_predict(cuda_device, trained):
    m, X, W, S = trained
    items = np.random.default_rng(1).permutation(N_ITEMS)[:500]
    got = m.rank(items, 11, 50)
    np.testing.assert_array_equal(got, items[np.argsort(-S[11, items], kind="stable")][:50])
    assert len(m.rank(items, 11)) == 500


@gpu
def test_input_errors(cuda_device, trained):
    m, X, W, S = trained
    fresh = ItemKNN(num_items=N_ITEMS, num_users=X.shape[0])
    for call in (lambda: fresh.recommend(np.arange(3), 10), lambda: fresh.eval_ranking(X),
                 lambda: fresh.predict([0], [0])):
        with pytest.raises(ValueError):
            call()
    for kwargs in ({"similarity": "pearson"}, {"k": 0}, {"k": 1025}, {"k": 2.5}, {"shrink": -1.0},
                   {"shrink": float("inf")}, {"shrink": float("nan")}):
        with pytest.raises(ValueError):
            fresh.train(X, **kwargs)
    assert fresh._X is None
    for users in ([-1], [0, X.shape[0]]):
        with pytest.raises(ValueError):
            m.recommend(np.array(users), 10)
        with pytest.raises(ValueError):
            m.eval_ranking(X, users=np.array(users))
        with pytest.raises(ValueError):
            m.predict(np.array(users), np.zeros(len(users), np.int64))
    with pytest.raises(ValueError):
        m.predict([0], [N_ITEMS])
    for shape in ((X.shape[0], N_ITEMS - 1), (X.shape[0] - 1, N_ITEMS)):
        with pytest.raises(ValueError):
            m.recommend(np.arange(3), 10, exclude=scipy.sparse.csr_matrix(shape, dtype=np.float32))
        with pytest.raises(ValueError):
            m.eval_ranking(X, exclude=scipy.sparse.csr_matrix(shape, dtype=np.float32))
    for shape in ((X.shape[0], N_ITEMS + 1), (X.shape[0] + 1, N_ITEMS)):
        with pytest.raises(ValueError):
            m.eval_ranking(scipy.sparse.csr_matrix(shape, dtype=np.float32))
    for topn in ([0], [5, 5], np.arange(1, 18), [[1, 2]], [1.5], []):
        with pytest.raises(ValueError):
            m.eval_ranking(X, topn=topn)
    with pytest.raises(ValueError):
        m.neighbors = scipy.sparse.csr_matrix((N_ITEMS, N_ITEMS + 1))
    other = ItemKNN(num_items=N_ITEMS, num_users=X.shape[0])
    other.train(X, k=5)
    other.neighbors = scipy.sparse.identity(N_ITEMS - 1, format="csr")
    with pytest.raises(ValueError):
        other.recommend(np.arange(3), 10)
    assert m.recommend(np.arange(4), 0).shape == (4, 0)
    assert m.recommend(np.array([], dtype=np.int64), 10).shape == (0, 10)
    users_d = torch.arange(4, device=cuda_device)
    for topn in (0, 1025):
        with pytest.raises(_lib.WMFLibraryError, match="UNSUPPORTED"):
            engine.knn_score_topk(m._X, m._W_device(), users_d, topn)


def test_knn_entry_points_reject_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call
    need = lib.wmf_knn_train_workspace_bytes(1000, 100)
    assert need >= 1000 * 100 * 12 and lib.wmf_knn_train_workspace_bytes(0, 100) == 0
    assert lib.wmf_knn_train_workspace_bytes(1000, 0) == 0 and lib.wmf_knn_train_workspace_bytes(1000, 1025) == 0

    def train(xp=p, xi=p, rows=50, xtp=p, xti=p, n=1000, k=100, sim=0, shrink=0.0, wp=p, wi=p, wd=p, ws=p,
              ws_bytes=need):
        return lib.wmf_knn_train(xp, xi, rows, xtp, xti, n, k, sim, shrink, wp, wi, wd, ws, ws_bytes, None)
    for n in (0, -1, 1 << 31):
        assert train(n=n) == 1 and "n=" in _lib.last_error()
    for k in (0, -1, 1025):
        assert train(k=k) == 1 and "k=" in _lib.last_error()
    for sim in (-1, 3):
        assert train(sim=sim) == 1 and "similarity" in _lib.last_error()
    for shrink in (-1e-300, float("inf"), float("nan")):
        assert train(shrink=shrink) == 1 and "shrink" in _lib.last_error()
    assert train(rows=-1) == 1
    for name in ("xp", "xtp", "wp", "wi", "wd"):
        assert train(**{name: None}) == 1 and "null" in _lib.last_error()
    assert train(ws=None) == 2 and "workspace" in _lib.last_error()
    assert train(ws_bytes=need - 1) == 2

    assert lib.wmf_knn_predict(p, p, p, p, p, p, p, 1, p, -1, p, None) == 1
    assert lib.wmf_knn_predict(p, p, p, None, p, p, p, 1, p, 10, p, None) == 1 and "null" in _lib.last_error()
    assert lib.wmf_knn_predict(None, None, None, None, None, None, None, 1, None, 0, None, None) == 0

    sneed = lib.wmf_knn_score_topk_workspace_bytes(100, 1000, 10)
    assert sneed >= 100 * 1000 * 8 and lib.wmf_knn_score_topk_workspace_bytes(100, 0, 10) == 0

    def score(xp=p, xi=p, xd=p, wp=p, wi=p, wd=p, n=1000, users=p, nu=100, ep=None, ei=None, topn=10, ids=p, sc=None,
              ws=p, ws_bytes=sneed):
        return lib.wmf_knn_score_topk(xp, xi, xd, wp, wi, wd, n, users, nu, ep, ei, topn, ids, sc, ws, ws_bytes, None)
    for n in (0, -1, 1 << 31):
        assert score(n=n) == 1 and "n=" in _lib.last_error()
    assert score(nu=-1) == 1
    for topn in (0, -3, 1025):
        assert score(topn=topn) == 5 and "topn" in _lib.last_error()
    assert score(n=20, topn=21) == 5
    for name in ("xp", "wp", "users", "ids"):
        assert score(**{name: None}) == 1 and "null" in _lib.last_error()
    assert score(ws=None) == 2 and "workspace" in _lib.last_error()
    assert score(ws_bytes=sneed - 1) == 2
    assert score(nu=0, xp=None, users=None, ids=None, ws=None, ws_bytes=0) == 0
