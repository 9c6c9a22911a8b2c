"""Ease.recommend and Ease.eval_ranking (include/wmf_b200.h: wmf_ease_score_topk): exact top-N over each user's unseen
items. Every list must equal, element for element, a NumPy oracle that sums the FP32 products in double in stored order
and orders by (-score, item id); every returned score must be bitwise what Ease.predict returns."""
import numpy as np
import pytest
import scipy.sparse
import torch

from conftest import csr_from, load_golden
from test_gpu_eval_ranking import oracle_means, oracle_per_user
from recmodel_b200 import _lib, build, engine, ranking, utils
from recmodel_b200.ease_model import Ease
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts, split_train_test

gpu = pytest.mark.gpu
N_ITEMS = 1100  # not a multiple of the 128-item panel of the scoring kernel


def oracle_scores(X, W, u):
    """float64 [items]: for each stored entry of row u in stored order, acc += fp32(x_e * W[j_e]) in double."""
    acc = np.zeros(W.shape[1], np.float64)
    for e in range(X.indptr[u], X.indptr[u + 1]):
        acc += (X.data[e] * W[X.indices[e]]).astype(np.float32).astype(np.float64)
    return acc


def oracle_lists(X, W, users, seen, topn):
    out = np.full((len(users), topn), -1, dtype=np.int64)
    for r, u in enumerate(users):
        s = oracle_scores(X, W, u)
        cand = np.setdiff1d(np.arange(W.shape[1]), seen[u])
        best = cand[np.lexsort((cand, -s[cand]))][:topn]
        out[r, :len(best)] = best
    return out


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


@pytest.fixture(scope="module")
def trained():
    """An Ease model trained on a 3000 x 1100 count matrix whose X has an empty row (user 5) and unsorted rows with
    duplicates and explicit zeros (users 0..99), with two equal columns of W (items 7 and 901: an exact tie for every user)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    C = make_counts(3000, N_ITEMS, 90_000, seed=3, planted_rank=6).tolil()
    C.rows[5], C.data[5] = [], []
    X = C.tocsr()
    head = messy_csr([X.indices[X.indptr[u]:X.indptr[u + 1]] for u in range(100)], (100, N_ITEMS), seed=1)
    X = scipy.sparse.vstack([head, X[100:]], format="csr")
    X.has_sorted_indices = False
    assert X.indptr[6] - X.indptr[5] == 0 and not np.all(np.diff(X.indices[X.indptr[0]:X.indptr[1]]) > 0)
    m = Ease(num_items=N_ITEMS, num_users=3000)
    m.train(X, alpha=100.0, verbose=0, cores=1)
    W = m.W.copy()
    W[:, 901] = W[:, 7]
    m.W = W
    return m, X, W


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
def test_recommend_reproduces_the_executed_reference(cuda_device, tmp_path):
    """The reference's own top-10 lists of the golden fixture (its W, its training matrix, nothing excluded)."""
    g = load_golden("ease_f300")
    X = csr_from(g, "train")
    np.save(tmp_path / "W.npy", g["W"])
    m = Ease(num_items=X.shape[1], num_users=X.shape[0])
    m.load_mat(str(tmp_path / "W.npy"), X=X)
    np.testing.assert_array_equal(m.recommend(g["rank_users"], 10), g["rank_top10"])


@gpu
@pytest.mark.parametrize("topn", [1, 10, 100, 1024, N_ITEMS])
def test_recommend_equals_the_oracle(cuda_device, trained, topn):
    m, X, W = trained
    n_users = 60
    seen = seen_lists(n_users, seed=topn)
    Ex = messy_csr(seen, (n_users, N_ITEMS), seed=topn)
    Ex = scipy.sparse.vstack([Ex, scipy.sparse.csr_matrix((X.shape[0] - n_users, N_ITEMS), dtype=np.float32)],
                             format="csr")
    rng = np.random.default_rng(topn)
    users = np.concatenate([rng.permutation(n_users), [5, 5, 0]])       # shuffled, the empty X row, repeats
    got = m.recommend(users, topn, exclude=Ex)
    assert got.dtype == np.int64 and got.shape == (len(users), topn)
    want = oracle_lists(X, W, users, seen, topn)
    np.testing.assert_array_equal(got, want)
    assert np.all(got[users == 3] == -1)
    if topn >= 10:
        assert np.any(got[users % 5 == 2] == -1)                        # padded rows
        r = np.flatnonzero(users == 1)[0]                               # the tie: 7 before 901 wherever both appear
        row = got[r].tolist()
        if 7 in row and 901 in row:
            assert row.index(7) < row.index(901)
    if topn <= _lib.TOPK_MAX:
        users_d = torch.from_numpy(users).to(cuda_device)
        ex = DeviceCSR.from_scipy(Ex, cuda_device)
        ids, scores = engine.ease_score_topk(m._X, m.W_device, users_d, topn, exclude=ex, want_scores=True)
        ids, scores = ids.cpu().numpy(), scores.cpu().numpy()
        np.testing.assert_array_equal(ids, got)
        valid = ids >= 0
        assert np.all(np.isnan(scores[~valid]))
        pred = m.predict(np.repeat(users, topn)[valid.reshape(-1)], ids[valid])
        assert pred.dtype == np.float64
        np.testing.assert_array_equal(scores[valid].view(np.uint64), pred.view(np.uint64))
        np.testing.assert_array_equal(scores[users == 5][valid[users == 5]], 0.0)   # empty X row: every score +0


@gpu
def test_scores_and_lists_independent_of_the_batch(cuda_device, trained):
    m, X, W = trained
    users_d = torch.arange(X.shape[0], device=cuda_device).flip(0)
    Ex = messy_csr(seen_lists(X.shape[0], seed=9), X.shape, seed=9)
    ex = DeviceCSR.from_scipy(Ex, cuda_device)
    for topn in (10, 300):
        ids, scores = engine.ease_score_topk(m._X, m.W_device, users_d, topn, exclude=ex, want_scores=True)
        pieces, u0 = [], 0
        for size in (1, 7, 64, 999, 5000):
            part = users_d[u0:u0 + size]
            if part.numel():
                pieces.append(engine.ease_score_topk(m._X, m.W_device, part, topn, exclude=ex, want_scores=True))
            u0 += size
        assert u0 >= users_d.numel()
        torch.testing.assert_close(ids, torch.cat([p[0] for p in pieces]), rtol=0, atol=0)
        a = scores.cpu().numpy().view(np.uint64)
        b = torch.cat([p[1] for p in pieces]).cpu().numpy().view(np.uint64)
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(m.recommend(np.arange(X.shape[0]), 20, exclude=Ex),
                                  m.recommend(np.arange(X.shape[0]), 20, exclude=ex))


@gpu
@pytest.mark.parametrize("ks", [[10, 50, 5], [1200, 10]])    # the second: the sort path and padding past the items
def test_eval_ranking_equals_the_definitions_in_any_chunking(cuda_device, monkeypatch, ks):
    full = make_counts(2000, N_ITEMS, 60_000, seed=8, planted_rank=6)
    Train, Test = split_train_test(full)
    m = Ease(num_items=N_ITEMS, num_users=2000)
    m.train(Train, alpha=50.0, verbose=0, cores=1)
    K = max(ks)
    users = np.flatnonzero(np.diff(Test.indptr) > 0)
    ids = m.recommend(users, K, exclude=Train)
    sample = users[::97]
    seen = [Train.indices[Train.indptr[u]:Train.indptr[u + 1]] for u in range(Train.shape[0])]
    np.testing.assert_array_equal(ids[::97][:, :min(K, N_ITEMS)], oracle_lists(Train, m.W, sample, seen, min(K, N_ITEMS)))
    want = oracle_per_user(ids, users, Test, ks)
    T = DeviceCSR.from_scipy(Test, cuda_device).sorted()
    got = engine.topn_metrics(torch.from_numpy(ids).to(cuda_device), torch.from_numpy(users).to(cuda_device), T,
                              ks).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    res = m.eval_ranking(Test, topn=ks, exclude=Train)
    means = oracle_means(want, ks)
    assert res["users"] == means["users"] == len(users) and set(res) == set(means)
    for key in means:
        np.testing.assert_allclose(res[key], means[key], rtol=1e-12, atol=1e-15)
    assert res[f"Recall@{K}"] > 0
    assert m.eval_ranking(DeviceCSR.from_scipy(Test, cuda_device), topn=ks,
                          exclude=DeviceCSR.from_scipy(Train, cuda_device)) == res
    real, calls = engine.topn_metrics, []
    monkeypatch.setattr(engine, "topn_metrics", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    for chunk in (K * 13, 1):     # chunks of 13 users, then 1 user
        monkeypatch.setattr(ranking, "EVAL_CHUNK_IDS", chunk)
        calls.clear()
        assert m.eval_ranking(Test, topn=ks, exclude=Train) == res
        assert len(calls) == -(-len(users) // max(1, chunk // K))   # one metrics call per chunk


@gpu
def test_coverage_equals_the_per_user_loop(cuda_device):
    """utils.test_coverage takes recommend for Ease and equals the reference's rank(np.delete(...)) loop. The model has
    no near-tie at any user's 10th place, so the loop's argpartition picks the same set."""
    full = make_counts(1500, N_ITEMS, 40_000, seed=12, planted_rank=6)
    empty = np.flatnonzero(np.diff(full.indptr) == 0)       # an empty row scores every item 0: one entry each
    full = (full + scipy.sparse.csr_matrix((np.ones(len(empty), np.float32), (empty, empty * 7 % N_ITEMS)),
                                           shape=full.shape)).tocsr()
    assert np.diff(full.indptr).min() > 0
    m = Ease(num_items=N_ITEMS, num_users=1500)
    m.train(full, alpha=50.0, verbose=0, cores=1)
    S = full.astype(np.float64) @ m.W.astype(np.float64)
    S[full.nonzero()] = -np.inf
    top = -np.sort(-S, axis=1)[:, :11]
    assert np.all(top[:, 9] - top[:, 10] > 1e-9 * np.abs(top[:, 9]))

    class LoopOnly:
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    got = utils.test_coverage(m, full, 10)
    np.testing.assert_array_equal(got, utils.test_coverage(LoopOnly(), full, 10))
    assert got.sum() == 1500 * 10


@gpu
def test_input_errors(cuda_device, trained):
    m, X, W = trained
    bare = Ease(num_items=N_ITEMS, num_users=3000)
    bare.W = W                                     # load_mat(path) without X: no interaction matrix
    with pytest.raises(ValueError):
        bare.recommend(np.arange(3), 10)
    with pytest.raises(ValueError):
        bare.eval_ranking(X)
    for users in ([-1], [0, X.shape[0]]):
        with pytest.raises(ValueError):
            m.recommend(np.array(users), 10)
        with pytest.raises(ValueError):
            m.eval_ranking(X, users=np.array(users))
    with pytest.raises(ValueError):
        m.recommend(np.arange(3), 10, exclude=scipy.sparse.csr_matrix((X.shape[0], N_ITEMS - 1), dtype=np.float32))
    with pytest.raises(ValueError):
        m.recommend(np.arange(3), 10, exclude=scipy.sparse.csr_matrix((X.shape[0] - 1, N_ITEMS), dtype=np.float32))
    with pytest.raises(ValueError):
        m.eval_ranking(scipy.sparse.csr_matrix((X.shape[0], N_ITEMS + 1), dtype=np.float32))
    with pytest.raises(ValueError):
        m.eval_ranking(scipy.sparse.csr_matrix((X.shape[0] + 1, N_ITEMS), dtype=np.float32))
    with pytest.raises(ValueError):
        m.eval_ranking(X, exclude=scipy.sparse.csr_matrix((X.shape[0], N_ITEMS - 1), dtype=np.float32))
    for topn in ([0], [5, 5], np.arange(1, 18), [[1, 2]], [1.5], [], np.array([True])):
        with pytest.raises(ValueError):
            m.eval_ranking(X, topn=topn)
    assert m.recommend(np.arange(4), 0).shape == (4, 0)
    assert m.recommend(np.array([], dtype=np.int64), 10).shape == (0, 10)
    users_d = torch.arange(4, device=cuda_device)
    with pytest.raises(_lib.WMFLibraryError, match="UNSUPPORTED"):
        engine.ease_score_topk(m._X, m.W_device, users_d, 1025)
    with pytest.raises(_lib.WMFLibraryError, match="UNSUPPORTED"):
        engine.ease_score_topk(m._X, m.W_device, users_d, 0)


def test_ease_score_topk_rejects_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call
    need = lib.wmf_ease_score_topk_workspace_bytes(100, 1000, 10)
    assert need >= 100 * 1000 * 8 and lib.wmf_ease_score_topk_workspace_bytes(100, 0, 10) == 0

    def run(xp=p, xi=p, xd=p, W=p, n=1000, users=p, nu=100, ep=None, ei=None, topn=10, ids=p, sc=None, ws=p,
            ws_bytes=need):
        return lib.wmf_ease_score_topk(xp, xi, xd, W, n, users, nu, ep, ei, topn, ids, sc, ws, ws_bytes, None)
    for n in (0, -1, 1 << 31):
        assert run(n=n) == 1 and "n=" in _lib.last_error()
    assert run(nu=-1) == 1
    for topn in (0, -3, 1025):
        assert run(topn=topn) == 5 and "topn" in _lib.last_error()
    assert run(n=20, topn=21) == 5
    for name in ("xp", "W", "users", "ids"):
        assert run(**{name: None}) == 1 and "null" in _lib.last_error()
    assert run(ws=None) == 2 and "workspace" in _lib.last_error()
    assert run(ws_bytes=need - 1) == 2
    assert run(nu=0, xp=None, users=None, ids=None, ws=None, ws_bytes=0) == 0   # nothing to do, nothing launched
