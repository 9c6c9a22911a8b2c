"""RP3beta (include/wmf_b200.h: wmf_rp3beta_train): a three-step random-walk item model trained, scored and ranked on
the device. W must equal, bit for bit, a NumPy oracle that sums the walk weights per item row in ascending user order
and applies the two rounded products; the scores are ItemKNN's over the binary pattern of X."""
import numpy as np
import pytest
import scipy.sparse
import torch

from test_gpu_eval_ranking import oracle_means, oracle_per_user
from test_gpu_itemknn import (EMPTY_ITEM, EMPTY_USER, N_ITEMS, assert_same_W, canonical, make_X, messy_csr,
                              oracle_lists, oracle_neighbors, oracle_scores, seen_lists)
from recmodel_b200 import ItemKNN, RP3beta, _lib, build, engine, ranking, utils
from recmodel_b200.synthetic import make_counts, split_train_test

gpu = pytest.mark.gpu
TILE_BYTES = 64 << 20   # knn_batch: rows per [B x n] double tile


def pattern(X):
    P = canonical(X)
    P.data = np.ones_like(P.data)
    return P


def scales(P, alpha, beta):
    """du, ra, cb: NumPy float64 np.power of the degrees and popularities, 0 for empty rows and columns."""
    deg = np.diff(P.indptr)
    pop = np.bincount(P.indices, minlength=P.shape[1])

    def power(c, e):
        out = np.zeros(len(c), np.float64)
        out[c > 0] = np.power(c[c > 0].astype(np.float64), -e)
        return out
    return power(deg, alpha), power(pop, alpha), power(pop, beta)


def oracle_S(P, du):
    """Dense float64 [n x n]: row a is acc[P.indices[row u]] += du[u] over the users u of a, ascending, from +0.0."""
    PT = P.T.tocsr()
    PT.sort_indices()
    S = np.zeros((P.shape[1], P.shape[1]), np.float64)
    for a in range(P.shape[1]):
        acc = S[a]
        for u in PT.indices[PT.indptr[a]:PT.indptr[a + 1]]:
            acc[P.indices[P.indptr[u]:P.indptr[u + 1]]] += du[u]
    return S


def oracle_W(S, ra, cb, k):
    """W of the definition: W'_ab = (ra[a] S_ab) cb[b] for b != a with S_ab > 0, the top k by lexsort((b, -W'))."""
    n = S.shape[0]
    rows, cols, vals = [], [], []
    oracle_W.tie_cuts = 0   # rows whose k-th and (k+1)-th candidates have the same weight
    for a in range(n):
        b = np.flatnonzero(S[a] > 0)
        b = b[b != a]
        w = (ra[a] * S[a, b]) * cb[b]
        order = np.lexsort((b, -w))
        oracle_W.tie_cuts += len(order) > k and w[order[k - 1]] == w[order[k]]
        top = order[:k]
        top = top[np.argsort(b[top])]
        rows.append(np.full(len(top), a))
        cols.append(b[top])
        vals.append(w[top])
    W = scipy.sparse.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    W.sort_indices()
    return W


def oracle(X, alpha, beta, k):
    P = pattern(X)
    du, ra, cb = scales(P, alpha, beta)
    return oracle_W(oracle_S(P, du), ra, cb, k)


@pytest.fixture(scope="module")
def data():
    X = make_X()
    assert X.indptr[EMPTY_USER + 1] == X.indptr[EMPTY_USER] and np.diff(X.tocsc().indptr)[EMPTY_ITEM] == 0
    return X


@pytest.fixture(scope="module")
def sums(data):
    """The walk sums S of the oracle per alpha, computed once."""
    P = pattern(data)
    return {alpha: oracle_S(P, scales(P, alpha, 0.0)[0]) for alpha in (0.0, 0.5, 1.0, 2.0)}


@gpu
@pytest.mark.parametrize("beta", [0.0, 0.3, 1.0, 2.0])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0, 2.0])
def test_W_equals_the_oracle(cuda_device, data, sums, alpha, beta):
    _, ra, cb = scales(pattern(data), alpha, beta)
    for k in (1, 10, 100, 1024):
        m = RP3beta(num_items=N_ITEMS, num_users=data.shape[0])
        m.train(data, alpha=alpha, beta=beta, k=k)
        W = m.W
        assert isinstance(W, scipy.sparse.csr_matrix) and W.dtype == np.float64 and W.shape == (N_ITEMS, N_ITEMS)
        assert W.has_sorted_indices and np.all(W.data > 0)
        assert_same_W(W, oracle_W(sums[alpha], ra, cb, k))
        lengths = np.diff(W.indptr)
        assert lengths[EMPTY_ITEM] == 0 and W[:, EMPTY_ITEM].nnz == 0 and lengths.max() <= k
        if k == 1024:
            assert 0 < lengths[lengths > 0].min() < k   # items with fewer candidates than k
        if alpha == beta == 0.0 and k <= 100:
            assert oracle_W.tie_cuts > 0   # exact integer ties at the k-th place, kept by the lower id


@gpu
def test_training_spans_several_blocks_in_walk_length_order(cuda_device):
    """8 000 items: a [B x n] tile holds 1 048 item rows, so training runs 8 blocks, and the rows grouped by walk
    length put high ids into the first block and low ids into later ones."""
    n = 8000
    X = make_counts(6000, n, 150_000, seed=6, planted_rank=6)
    P = pattern(X)
    B = TILE_BYTES // (n * 8)
    deg = np.diff(P.indptr)
    PT = P.T.tocsr()
    chain = np.array([((deg[PT.indices[PT.indptr[a]:PT.indptr[a + 1]]] + 255) // 256).sum() for a in range(n)])
    grouped = np.lexsort((np.arange(n), -chain))
    assert -(-n // B) == 8 and grouped[:B].max() >= B and grouped[B:].min() < B
    for alpha, beta, k in ((0.8, 0.4, 50), (0.0, 0.0, 20)):
        m = RP3beta(num_items=n, num_users=X.shape[0])
        m.train(X, alpha=alpha, beta=beta, k=k)
        assert_same_W(m.W, oracle(X, alpha, beta, k))


@gpu
def test_p3alpha_rows_are_walk_probabilities(cuda_device):
    """alpha = 1, beta = 0, 900 items and k = 1024: every candidate is kept, and each row plus its self term
    ra[a] S_aa is the two-hop walk distribution from a, which sums to 1."""
    X = make_counts(700, 900, 20_000, seed=13, planted_rank=5)
    P = pattern(X)
    m = RP3beta(num_items=900, num_users=700)
    m.train(X, alpha=1.0, beta=0.0, k=1024)
    du, ra, _ = scales(P, 1.0, 0.0)
    S = oracle_S(P, du)
    W = m.W
    pop = np.bincount(P.indices, minlength=900)
    assert np.count_nonzero(pop) > 800
    total = np.asarray(W.sum(axis=1)).ravel() + ra * np.diag(S)
    np.testing.assert_allclose(total[pop > 0], 1.0, rtol=0, atol=1e-12)
    assert np.all(total[pop == 0] == 0)
    np.testing.assert_array_equal(np.diff(W.indptr), np.count_nonzero(S > 0, axis=1) - (pop > 0))


@gpu
def test_unscaled_walk_is_the_cooccurrence(cuda_device, data):
    """alpha = beta = 0: W'_ab = c_ab, so W is P^T P off the diagonal when every candidate is kept, and the kept ids
    are ItemKNN's conditional neighbours (c_ab / c_aa orders each row like c_ab)."""
    X = make_counts(700, 900, 20_000, seed=14, planted_rank=5)
    P = pattern(X).astype(np.int64)
    m = RP3beta(num_items=900, num_users=700)
    m.train(X, alpha=0.0, beta=0.0, k=1024)
    C = (P.T @ P).toarray().astype(np.float64)
    np.fill_diagonal(C, 0.0)
    np.testing.assert_array_equal(m.W.toarray(), C)
    m = RP3beta(num_items=N_ITEMS, num_users=data.shape[0])
    for k in (1, 10, 100):
        m.train(data, alpha=0.0, beta=0.0, k=k)
        want = oracle_neighbors(data, k, "conditional", 0.0)
        knn = ItemKNN(num_items=N_ITEMS, num_users=data.shape[0])
        knn.train(data, k=k, similarity="conditional", shrink=0.0)
        for W in (want, knn.neighbors):
            np.testing.assert_array_equal(m.W.indptr, W.indptr)
            np.testing.assert_array_equal(m.W.indices, W.indices)


@gpu
def test_messy_input_trains_the_canonical_model(cuda_device, data):
    head = messy_csr([data.indices[data.indptr[u]:data.indptr[u + 1]] for u in range(200)], (200, N_ITEMS), seed=1)
    X = scipy.sparse.vstack([head, data[200:]], format="csr")
    X.has_sorted_indices = False
    before = (X.indptr.copy(), X.indices.copy(), X.data.copy())
    a = RP3beta(num_items=N_ITEMS, num_users=X.shape[0])
    a.train(X, alpha=0.7, beta=0.2, k=64)
    for arr, old in zip((X.indptr, X.indices, X.data), before):   # the caller's matrix is untouched
        np.testing.assert_array_equal(arr, old)
    b = RP3beta(num_items=N_ITEMS, num_users=X.shape[0])
    b.train(canonical(X), alpha=0.7, beta=0.2, k=64)
    assert_same_W(a.W, b.W)
    assert_same_W(a.W, oracle(X, 0.7, 0.2, 64))


@gpu
def test_determinism(cuda_device, data):
    runs = []
    for _ in range(2):
        m = RP3beta(num_items=N_ITEMS, num_users=data.shape[0])
        m.train(data, alpha=0.9, beta=0.6, k=1024)
        runs.append(m.W)
    assert_same_W(runs[0], runs[1])


@pytest.fixture(scope="module")
def trained(data):
    """A default model (alpha 1, beta 0.5, k 100) whose W was edited to give items 7 and 901 equal columns: an exact
    score tie for every user that votes for either."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    m = RP3beta(num_items=N_ITEMS, num_users=data.shape[0])
    m.train(data)
    assert_same_W(m.W, oracle(data, 1.0, 0.5, 100))
    Wd = m.W.toarray()
    Wd[:, 901] = Wd[:, 7]
    W = scipy.sparse.csr_matrix(Wd)
    m.W = W
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
@pytest.mark.parametrize("topn", [1, 100, N_ITEMS])   # N_ITEMS: more than every user's unseen items, the sort path
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
        both = got[(got == 7).any(axis=1) & (got == 901).any(axis=1)]   # equal scores: the lower id first
        assert np.all(np.argmax(both == 7, axis=1) < np.argmax(both == 901, axis=1))
        assert len(both) or topn < N_ITEMS
    if topn <= _lib.TOPK_MAX:
        users_d = torch.from_numpy(users).to(cuda_device)
        ex = engine.DeviceCSR.from_scipy(Ex, cuda_device)
        ids, scores = engine.knn_score_topk(m._X, m._W_device(), users_d, topn, exclude=ex, want_scores=True)
        ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
        np.testing.assert_array_equal(ids, got)
        valid = ids >= 0
        assert np.all(np.isnan(scores[~valid]))
        want = S[np.repeat(users, topn).reshape(ids.shape)[valid], ids[valid]]
        np.testing.assert_array_equal(scores[valid].view(np.uint64), want.view(np.uint64))


@gpu
def test_eval_ranking_equals_the_definitions_in_any_chunking(cuda_device, monkeypatch):
    ks = [10, 50, 5]
    full = make_counts(2000, N_ITEMS, 60_000, seed=8, planted_rank=6)
    Train, Test = split_train_test(full)
    m = RP3beta(num_items=N_ITEMS, num_users=2000)
    m.train(Train, alpha=0.8, beta=0.3, k=64)
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
    m = RP3beta(num_items=N_ITEMS, num_users=1500)
    m.train(full, k=32)

    class LoopOnly:
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    got = utils.test_coverage(m, full, 10)
    np.testing.assert_array_equal(got, utils.test_coverage(LoopOnly(), full, 10))
    assert got.sum() > 0


@gpu
def test_rank_is_a_stable_sort_of_predict(cuda_device, trained):
    m, X, W, S = trained
    items = np.random.default_rng(1).permutation(N_ITEMS)
    items = items[(items != 7) & (items != 901)][:500]
    tied = int(np.flatnonzero((S[:, 7] == S[:, 901]) & (S[:, 7] > 0))[0])   # items 7 and 901 tie: candidate order
    for u in (12, tied):
        cand = np.concatenate([items, [901, 7]]) if u == tied else items
        got = m.rank(cand, u, 50)
        np.testing.assert_array_equal(got, cand[np.argsort(-S[u, cand], kind="stable")][:50])
    assert len(m.rank(items, 12)) == 500


@gpu
def test_W_setter_round_trips(cuda_device, trained, data):
    m, X, W, S = trained
    other = RP3beta(num_items=N_ITEMS, num_users=X.shape[0])
    other.train(data, k=8)
    other.W = W.tocoo()
    assert_same_W(other.W, W)
    np.testing.assert_array_equal(other.recommend(np.arange(50), 20), m.recommend(np.arange(50), 20))
    other.W = scipy.sparse.identity(N_ITEMS - 1, format="csr")
    with pytest.raises(ValueError):
        other.recommend(np.arange(3), 10)


def test_train_rejects_bad_arguments_without_a_device():
    X = make_counts(50, 40, 300, seed=2)
    m = RP3beta(num_items=40, num_users=50)
    bad = [{"alpha": v} for v in (-1e-9, 2.000001, float("nan"), float("inf"), -float("inf"))]
    bad += [{"beta": v} for v in (-0.5, 3.0, float("nan"), float("inf"))]
    bad += [{"k": 0}, {"k": 1025}, {"k": True}, {"k": 2.5}]
    for kwargs in bad:
        with pytest.raises(ValueError):
            m.train(X, **kwargs)
    assert m._X is None and m._W_d is None
    with pytest.raises(ValueError, match="square"):
        m.W = scipy.sparse.csr_matrix((40, 41))
    assert m.W is None
    for call in (lambda: m.predict([0], [0]), lambda: m.recommend(np.arange(3), 10)):
        with pytest.raises(ValueError):
            call()


def test_rp3beta_entry_rejects_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call
    need = lib.wmf_rp3beta_train_workspace_bytes(1000, 5000, 100)
    assert need >= 1000 * 100 * 12 + 5000 * 12
    assert lib.wmf_rp3beta_train_workspace_bytes(1000, 5000, 1024) > need
    for n, nnz, k in ((0, 10, 10), (1 << 31, 10, 10), (100, -1, 10), (100, 10, 0), (100, 10, 1025)):
        assert lib.wmf_rp3beta_train_workspace_bytes(n, nnz, k) == 0

    def train(pp=p, pi=p, rows=50, ptp=p, pti=p, n=1000, nnz=5000, du=p, ra=p, cb=p, k=100, wp=p, wi=p, wd=p, ws=p,
              ws_bytes=need):
        return lib.wmf_rp3beta_train(pp, pi, rows, ptp, pti, n, nnz, du, ra, cb, k, wp, wi, wd, ws, ws_bytes, None)
    for k in (0, -1, 1025):
        assert train(k=k) == 1 and "k=" in _lib.last_error()
    for n in (0, -1, 1 << 31):
        assert train(n=n) == 1 and "n=" in _lib.last_error()
    assert train(rows=-1) == 1 and "rows=" in _lib.last_error()
    assert train(nnz=-1) == 1 and "nnz=" in _lib.last_error()
    for name in ("pp", "pi", "ptp", "pti", "du", "ra", "cb", "wp", "wi", "wd"):
        assert train(**{name: None}) == 1 and "null" in _lib.last_error()
    assert train(ws=None) == 2 and "workspace" in _lib.last_error()
    assert train(ws_bytes=need - 1) == 2 and "wmf_rp3beta_train" in _lib.last_error()
