"""UserKNN (include/wmf_b200.h: wmf_knn_train on (X^T, X), wmf_userknn_*): user-user neighbourhoods trained, scored
and ranked on the device. The neighbours, their similarities, predict and the scores inside recommend must equal, bit
for bit, a NumPy oracle that restates the definitions with the same double operations in the same order."""
import numpy as np
import pytest
import scipy.sparse
import torch

from test_gpu_eval_ranking import oracle_means, oracle_per_user
from test_gpu_itemknn import assert_same_W, canonical, messy_csr, oracle_lists, oracle_neighbors
from recmodel_b200 import ItemKNN, UserKNN, _lib, build, engine, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts, split_train_test

gpu = pytest.mark.gpu
N_USERS, N_ITEMS = 1200, 2000
EMPTY_USER, EMPTY_ITEM = 5, 17
NO_NEIGHBOURS = 11          # a user with items whose neighbour row the `trained` fixture empties
SINGLE = range(1, N_USERS, 7)   # users whose only neighbour the fixture makes u + 1 at 0.5: exact score ties


def make_X(n_users=N_USERS, n_items=N_ITEMS, nnz=60_000, seed=3):
    """Counts with an empty user row and an item nobody interacted with."""
    C = make_counts(n_users, n_items, nnz, seed=seed, planted_rank=6).tocoo()
    keep = (C.row != EMPTY_USER) & (C.col != EMPTY_ITEM)
    return scipy.sparse.csr_matrix((C.data[keep], (C.row[keep], C.col[keep])), shape=C.shape)


def oracle_scores(X, N, u):
    """float64 [items]: acc[X_v.indices] += sim(u, v) * x_v over the neighbours v of row u of N, ascending."""
    acc = np.zeros(X.shape[1], np.float64)
    for e in range(N.indptr[u], N.indptr[u + 1]):
        v = N.indices[e]
        lo, hi = X.indptr[v], X.indptr[v + 1]
        acc[X.indices[lo:hi]] += N.data[e] * X.data[lo:hi].astype(np.float32).astype(np.float64)
    return acc


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
            s = rng.choice(N_ITEMS, size=int(rng.integers(1, 300)), replace=False)
        seen.append(np.asarray(s, np.int64))
    return seen


@pytest.fixture(scope="module")
def data():
    X = make_X()
    assert X.indptr[EMPTY_USER + 1] == X.indptr[EMPTY_USER] and np.diff(X.tocsc().indptr)[EMPTY_ITEM] == 0
    assert X.indptr[NO_NEIGHBOURS + 1] > X.indptr[NO_NEIGHBOURS]
    return X


@pytest.fixture(scope="module")
def trained(data):
    """A cosine model (k = 100, shrink 5) whose neighbors were edited: user NO_NEIGHBOURS has none, and each user of
    SINGLE has the single neighbour u + 1 at 0.5, so its scores are 0.5 x_{u+1, i}: exact ties between items."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    m = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
    m.train(data, k=100, similarity="cosine", shrink=5.0)
    Nd = m.neighbors.toarray()
    Nd[NO_NEIGHBOURS] = 0.0
    for u in SINGLE:
        Nd[u] = 0.0
        Nd[u, (u + 1) % N_USERS] = 0.5
    N = scipy.sparse.csr_matrix(Nd)
    m.neighbors = N
    Xc = canonical(data)
    S = np.stack([oracle_scores(Xc, N, u) for u in range(N_USERS)])
    return m, data, N, S


@gpu
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
@pytest.mark.parametrize("shrink", [0.0, 10.0])
@pytest.mark.parametrize("similarity", ["cosine", "jaccard", "conditional"])
def test_neighbors_equal_the_oracle_and_itemknn_on_the_transpose(cuda_device, data, similarity, shrink, k):
    m = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
    m.train(data, k=k, similarity=similarity, shrink=shrink)
    N = m.neighbors
    assert isinstance(N, scipy.sparse.csr_matrix) and N.dtype == np.float64 and N.shape == (N_USERS, N_USERS)
    assert_same_W(N, oracle_neighbors(data.T, k, similarity, shrink))
    lengths = np.diff(N.indptr)
    assert np.all(lengths[np.diff(data.indptr) == 0] == 0) and lengths[EMPTY_USER] == 0 and lengths.max() <= k
    if k == 1024:
        assert 0 < lengths[lengths > 0].min() < k   # users with fewer candidates
    if similarity == "conditional" and k <= 100:
        assert oracle_neighbors.tie_cuts > 0   # exact ties at the k-th place, kept by the lower id
    item = ItemKNN(num_items=N_USERS, num_users=N_ITEMS)
    item.train(data.T, k=k, similarity=similarity, shrink=shrink)
    assert_same_W(N, item.neighbors)


@gpu
def test_training_spans_several_user_blocks(cuda_device):
    """16 500 users: the [B x n] tiles hold 508 user rows, so training runs 33 blocks."""
    X = make_X(n_users=16_500, n_items=4000, nnz=120_000, seed=4)
    for similarity, k in (("conditional", 20), ("cosine", 300)):
        m = UserKNN(num_items=X.shape[1], num_users=X.shape[0])
        m.train(X, k=k, similarity=similarity, shrink=1.0)
        assert_same_W(m.neighbors, oracle_neighbors(X.T, k, similarity, 1.0))


@gpu
def test_messy_input_trains_the_canonical_model(cuda_device, data):
    head = messy_csr([data.indices[data.indptr[u]:data.indptr[u + 1]] for u in range(200)], (200, N_ITEMS), seed=1)
    X = scipy.sparse.vstack([head, data[200:]], format="csr")
    X.has_sorted_indices = False
    before = (X.indptr.copy(), X.indices.copy(), X.data.copy())
    a = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
    a.train(X, k=50, similarity="jaccard", shrink=2.0)
    for arr, old in zip((X.indptr, X.indices, X.data), before):   # the caller's matrix is untouched
        np.testing.assert_array_equal(arr, old)
    b = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
    b.train(canonical(X), k=50, similarity="jaccard", shrink=2.0)
    assert_same_W(a.neighbors, b.neighbors)
    assert_same_W(a.neighbors, oracle_neighbors(X.T, 50, "jaccard", 2.0))
    users = np.arange(300)
    want = np.stack([oracle_scores(canonical(X), a.neighbors, u)[:40] for u in users]).reshape(-1)
    assert np.any(want > 0)
    for m in (a, b):
        got = m.predict(np.repeat(users, 40), np.tile(np.arange(40), len(users)))
        np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))


@gpu
def test_determinism(cuda_device, data):
    runs = []
    for _ in range(2):
        m = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
        m.train(data, k=1024, similarity="conditional")
        runs.append(m.neighbors)
    assert_same_W(runs[0], runs[1])


@gpu
def test_predict_equals_the_oracle(cuda_device, trained):
    m, X, N, S = trained
    rng = np.random.default_rng(0)
    users = np.concatenate([rng.integers(0, N_USERS, 4000), [EMPTY_USER] * 10, [NO_NEIGHBOURS] * 10])
    items = rng.integers(0, N_ITEMS, len(users))
    got = m.predict(users, items)
    assert got.dtype == np.float64
    want = S[users, items]
    np.testing.assert_array_equal(got.view(np.uint64), want.view(np.uint64))
    assert np.any(want == 0) and np.any(want > 0)       # pairs no neighbour votes for score +0.0
    assert np.all(got[np.signbit(got)] != 0)
    for u in (3, NO_NEIGHBOURS, EMPTY_USER, SINGLE[2]):
        np.testing.assert_array_equal(m.predict(u, np.arange(N_ITEMS)).view(np.uint64), S[u].view(np.uint64))
    assert not S[NO_NEIGHBOURS].any() and not S[EMPTY_USER].any()


@gpu
@pytest.mark.parametrize("topn", [1, 10, 100, 1024, 1100])
def test_recommend_equals_the_oracle(cuda_device, trained, topn):
    """9 000 listed users: more than the 4 194 of one [ub x n] score tile at 2 000 items. topn 1100 takes the sort
    path."""
    m, X, N, S = trained
    seen = seen_lists(N_USERS, seed=topn)
    Ex = messy_csr(seen, (N_USERS, N_ITEMS), seed=topn)
    rng = np.random.default_rng(topn)
    users = np.concatenate([rng.permutation(N_USERS), rng.integers(0, N_USERS, 9000 - N_USERS - 4),
                            [EMPTY_USER, NO_NEIGHBOURS, 3, 0]])
    got = m.recommend(users, topn, exclude=Ex)
    assert got.dtype == np.int64 and got.shape == (len(users), topn)
    np.testing.assert_array_equal(got, oracle_lists(S, users, seen, topn))
    assert np.all(got[users == 3] == -1)                              # fully excluded
    if topn >= 10:
        assert np.any(got[users % 5 == 2] == -1)                     # padded rows
        single = np.isin(users, SINGLE) & (users % 5 != 2)
        g = got[single]
        s = S[users[single][:, None], np.maximum(g, 0)]
        tied = (s[:, 1:] == s[:, :-1]) & (s[:, 1:] > 0) & (g[:, 1:] >= 0)
        assert tied.any()                                             # exact ties, ordered by the lower id
        assert np.all(g[:, 1:][tied] > g[:, :-1][tied])
    if topn <= _lib.TOPK_MAX:
        users_d = torch.from_numpy(users).to(cuda_device)
        ex = DeviceCSR.from_scipy(Ex, cuda_device)
        ids, scores = engine.userknn_score_topk(m._X, m._W_device(), users_d, topn, exclude=ex, want_scores=True)
        ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
        np.testing.assert_array_equal(ids, got)
        valid = ids >= 0
        assert np.all(np.isnan(scores[~valid]))
        pred = m.predict(np.repeat(users, topn)[valid.reshape(-1)], ids[valid])
        np.testing.assert_array_equal(scores[valid].view(np.uint64), pred.view(np.uint64))
        for u in (EMPTY_USER, NO_NEIGHBOURS):
            np.testing.assert_array_equal(scores[users == u][valid[users == u]].view(np.uint64), 0)


@gpu
def test_lists_independent_of_the_batch(cuda_device, trained):
    m, X, N, S = trained
    users_d = torch.arange(N_USERS, device=cuda_device).flip(0).repeat(4)
    Ex = messy_csr(seen_lists(N_USERS, seed=9), X.shape, seed=9)
    ex = DeviceCSR.from_scipy(Ex, cuda_device)
    for topn in (10, 300):
        ids, scores = engine.userknn_score_topk(m._X, m._W_device(), users_d, topn, exclude=ex, want_scores=True)
        pieces, u0 = [], 0
        for size in (1, 7, 64, 999, 5000):
            part = users_d[u0:u0 + size]
            if part.numel():
                pieces.append(engine.userknn_score_topk(m._X, m._W_device(), part, topn, exclude=ex, want_scores=True))
            u0 += size
        assert u0 >= users_d.numel()
        torch.testing.assert_close(ids, torch.cat([p[0] for p in pieces]), rtol=0, atol=0)
        np.testing.assert_array_equal(scores.cpu().numpy().view(np.uint64),
                                      torch.cat([p[1] for p in pieces]).cpu().numpy().view(np.uint64))
    np.testing.assert_array_equal(m.recommend(np.arange(N_USERS), 20, exclude=Ex),
                                  m.recommend(np.arange(N_USERS), 20, exclude=ex))


@gpu
@pytest.mark.parametrize("ks", [[10, 50, 5], [2100, 10]])    # the second: the sort path and padding past the items
def test_eval_ranking_equals_the_definitions_in_any_chunking(cuda_device, monkeypatch, ks):
    full = make_counts(1500, N_ITEMS, 60_000, seed=8, planted_rank=6)
    Train, Test = split_train_test(full)
    m = UserKNN(num_items=N_ITEMS, num_users=1500)
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
    """utils.test_coverage takes recommend for UserKNN and equals the reference's rank(np.delete(...)) loop: rank
    breaks ties by candidate position, which is the item id there. Like the reference it counts into an array of one
    entry per user, so the matrix has more users than items."""
    full = make_counts(2500, N_ITEMS, 60_000, seed=12, planted_rank=6)
    m = UserKNN(num_items=N_ITEMS, num_users=2500)
    m.train(full, k=30, similarity="jaccard")

    class LoopOnly:
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    got = utils.test_coverage(m, full, 10)
    np.testing.assert_array_equal(got, utils.test_coverage(LoopOnly(), full, 10))
    assert got.sum() > 0


@gpu
def test_rank_is_a_stable_sort_of_predict(cuda_device, trained):
    m, X, N, S = trained
    items = np.random.default_rng(1).permutation(N_ITEMS)[:500]
    for u in (12, SINGLE[3]):    # the second has exact ties: kept in candidate order
        got = m.rank(items, u, 50)
        np.testing.assert_array_equal(got, items[np.argsort(-S[u, items], kind="stable")][:50])
    assert len(m.rank(items, 12)) == 500


@gpu
def test_input_errors(cuda_device, trained):
    m, X, N, S = trained
    fresh = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
    for call in (lambda: fresh.recommend(np.arange(3), 10), lambda: fresh.eval_ranking(X),
                 lambda: fresh.predict([0], [0])):
        with pytest.raises(ValueError):
            call()
    for kwargs in ({"similarity": "pearson"}, {"k": 0}, {"k": 1025}, {"k": 2.5}, {"k": True}, {"shrink": -1.0},
                   {"shrink": float("inf")}, {"shrink": float("nan")}):
        with pytest.raises(ValueError):
            fresh.train(X, **kwargs)
    assert fresh._X is None
    for users in ([-1], [0, N_USERS]):
        with pytest.raises(ValueError):
            m.recommend(np.array(users), 10)
        with pytest.raises(ValueError):
            m.eval_ranking(X, users=np.array(users))
        with pytest.raises(ValueError):
            m.predict(np.array(users), np.zeros(len(users), np.int64))
    with pytest.raises(ValueError):
        m.predict([0], [N_ITEMS])
    for shape in ((N_USERS, N_ITEMS - 1), (N_USERS - 1, N_ITEMS)):
        with pytest.raises(ValueError):
            m.recommend(np.arange(3), 10, exclude=scipy.sparse.csr_matrix(shape, dtype=np.float32))
        with pytest.raises(ValueError):
            m.eval_ranking(X, exclude=scipy.sparse.csr_matrix(shape, dtype=np.float32))
    for topn in ([0], [5, 5], np.arange(1, 18), [[1, 2]], [1.5], []):
        with pytest.raises(ValueError):
            m.eval_ranking(X, topn=topn)
    with pytest.raises(ValueError, match="square"):
        m.neighbors = scipy.sparse.csr_matrix((N_USERS, N_USERS + 1))
    other = UserKNN(num_items=N_ITEMS, num_users=N_USERS)
    other.train(X, k=5)
    for n in (N_USERS - 1, N_ITEMS):   # the neighbours must be num_users x num_users, not num_items x num_items
        other.neighbors = scipy.sparse.identity(n, format="csr")
        for call in (lambda: other.recommend(np.arange(3), 10), lambda: other.predict([0], [0]),
                     lambda: other.eval_ranking(X)):
            with pytest.raises(ValueError, match=f"neighbors is {n} x {n} but X has {N_USERS} users"):
                call()
    other.neighbors = scipy.sparse.identity(N_USERS, format="csr")   # each user its own neighbour: s(u, i) = x_ui
    np.testing.assert_array_equal(other.predict(7, np.arange(N_ITEMS)),
                                  canonical(X)[7].toarray().ravel().astype(np.float32).astype(np.float64))
    assert m.recommend(np.arange(4), 0).shape == (4, 0)
    assert m.recommend(np.array([], dtype=np.int64), 10).shape == (0, 10)
    users_d = torch.arange(4, device=cuda_device)
    for topn in (0, 1025):
        with pytest.raises(_lib.WMFLibraryError, match="UNSUPPORTED"):
            engine.userknn_score_topk(m._X, m._W_device(), users_d, topn)


def test_userknn_entry_points_reject_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call
    assert lib.wmf_userknn_predict(p, p, p, p, p, p, p, 1, p, -1, p, None) == 1
    assert lib.wmf_userknn_predict(p, p, p, p, p, p, p, -1, p, 10, p, None) == 1
    for pos in (0, 3, 6, 8, 10):   # x_indptr, nb_indptr, users, items, out
        args = [p, p, p, p, p, p, p, 1, p, 10, p, None]
        args[pos] = None
        assert lib.wmf_userknn_predict(*args) == 1 and "null" in _lib.last_error()
    assert lib.wmf_userknn_predict(None, None, None, None, None, None, None, 1, None, 0, None, None) == 0

    sneed = lib.wmf_userknn_score_topk_workspace_bytes(100, 1000, 10)
    assert sneed == lib.wmf_knn_score_topk_workspace_bytes(100, 1000, 10) >= 100 * 1000 * 8
    for nu, n in ((100, 0), (0, 1000), (-1, 1000), (100, 1 << 31)):
        assert lib.wmf_userknn_score_topk_workspace_bytes(nu, n, 10) == 0

    def score(xp=p, xi=p, xd=p, np_=p, ni=p, nd=p, n=1000, users=p, nu=100, ep=None, ei=None, topn=10, ids=p, sc=None,
              ws=p, ws_bytes=sneed):
        return lib.wmf_userknn_score_topk(xp, xi, xd, np_, ni, nd, n, users, nu, ep, ei, topn, ids, sc, ws, ws_bytes,
                                          None)
    for n in (0, -1, 1 << 31):
        assert score(n=n) == 1 and "n=" in _lib.last_error()
    assert score(nu=-1) == 1 and "nu=" in _lib.last_error()
    for topn in (0, -3, 1025):
        assert score(topn=topn) == 5 and "topn" in _lib.last_error()
    assert score(n=20, topn=21) == 5
    assert score(n=0, topn=0) == 1 and score(nu=-1, topn=0) == 1   # n, then nu, then topn
    for name in ("xp", "np_", "users", "ids"):
        assert score(**{name: None}) == 1 and "null" in _lib.last_error()
    assert score(ws=None) == 2 and "workspace" in _lib.last_error()
    assert score(ws_bytes=sneed - 1) == 2
    assert score(nu=0, xp=None, np_=None, users=None, ids=None, ws=None, ws_bytes=0) == 0
    assert "wmf_userknn_score_topk" in (score(ws=None) and _lib.last_error())
