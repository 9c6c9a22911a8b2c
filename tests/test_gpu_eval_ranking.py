"""WMF.eval_ranking and its kernels (include/wmf_b200.h: wmf_topn_metrics, wmf_topn_metrics_reduce): Recall, Precision,
NDCG, MAP and hit rate at N over each user's unseen items. The per-user values are compared with a NumPy restatement of
the definitions, computed from recommend's host lists and the SciPy test matrix, on the tensor-core, exact and sort
paths; a hand-built case checks the definitions themselves against closed-form values."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse
import torch

from conftest import ROOT
from oracle import wmf_oracle as orc
from recmodel_b200 import WMF, _lib, build, engine, wmf_model
from recmodel_b200.engine import DeviceCSR

gpu = pytest.mark.gpu


def oracle_per_user(ids, users, test, ks):
    """[len(users) x len(ks) x 5] from the definitions: T_u = distinct columns of row u with a non-zero stored value."""
    test = test.tocsr()
    K = ids.shape[1]
    pos = np.arange(1, K + 1, dtype=np.float64)
    disc = 1.0 / np.log2(pos + 1.0)
    out = np.full((len(users), len(ks), 5), np.nan)
    for r, u in enumerate(users):
        lo, hi = test.indptr[u], test.indptr[u + 1]
        T = set(test.indices[lo:hi][test.data[lo:hi] != 0].tolist())
        if not T:
            continue
        hit = np.array([int(x) in T for x in ids[r]], dtype=bool)
        h = np.cumsum(hit)
        for j, k in enumerate(ks):
            m = min(k, len(T))
            dcg = disc[:k][hit[:k]].sum()
            idcg = disc[:m].sum()
            ap = (h[:k] / pos[:k])[hit[:k]].sum()
            out[r, j] = (h[k - 1] / len(T), h[k - 1] / k, dcg / idcg, ap / m, float(h[k - 1] > 0))
    return out


def oracle_means(per_user, ks):
    keep = ~np.isnan(per_user[:, 0, 0])
    res = {}
    for j, k in enumerate(ks):
        for m, name in enumerate(engine.TOPN_METRICS):
            res[f"{name}@{k}"] = per_user[keep, j, m].mean()
    res["users"] = int(keep.sum())
    return res


def make_model(f, bias, ni, nu, seed):
    rng = np.random.default_rng(seed)
    U = (rng.standard_normal((nu, f)) * 0.5).astype(np.float32)
    V = (rng.standard_normal((ni, f)) * 0.5).astype(np.float32)
    m = WMF(num_items=ni, num_users=nu, dim=f - 1 if bias else f, gamma=0.1, weighted=True, bias=bias)
    m.users, m.items = U, V
    return m, U, V


def make_data(U, V, bias, K, seed):
    """(exclude, test) users x items. The test rows mix the user's best unseen items (so that there are hits at every
    depth) with random ones, in shuffled order, with duplicates and explicit zeros. Row kinds by u % 7: empty, zeros only,
    all excluded, a zero copy before a non-zero copy of the same id, a row longer than K, and two mixed rows."""
    nu, ni = U.shape[0], V.shape[0]
    rng = np.random.default_rng(seed)
    ex_rows, t_rows, t_vals = [], [], []
    for u in range(nu):
        seen = rng.choice(ni, size=int(rng.integers(0, max(2, ni // 20))), replace=False)
        if u % 11 == 4:
            seen = rng.choice(ni, size=ni - max(1, K // 3), replace=False)   # fewer than K unseen items: padded list
        s = orc.rank_scores(U, V, np.arange(ni), u, bias)
        unseen = np.setdiff1d(np.argsort(-s, kind="stable"), seen, assume_unique=True)
        best = np.argsort(-s[unseen], kind="stable")
        best = unseen[best]
        kind = u % 7
        if kind == 0 or len(best) == 0:
            items, vals = np.empty(0, np.int64), np.empty(0, np.float32)
        elif kind == 1:
            items = rng.choice(best[:2 * K], size=min(5, len(best)), replace=False)
            vals = np.zeros(len(items), np.float32)
        elif kind == 2:
            items = seen[:7] if len(seen) else np.empty(0, np.int64)
            vals = np.ones(len(items), np.float32)
        elif kind == 3:
            a = best[rng.integers(0, min(len(best), K))]
            b = best[rng.integers(0, min(len(best), K))]
            items = np.array([a, a, b, b, b])
            vals = np.array([0, 2, 0, 0, 0], np.float32)   # a is in T_u through its second copy, b is not
        elif kind == 4:
            items = np.concatenate([best[:min(len(best), K + 5)], rng.choice(ni, size=20)])
            vals = rng.integers(1, 4, size=len(items)).astype(np.float32)
        else:
            pick = best[rng.choice(min(len(best), 3 * K), size=min(len(best), max(1, K // 4)), replace=False)]
            items = np.concatenate([pick, rng.choice(ni, size=10), pick[:3]])          # duplicates
            vals = rng.integers(0, 3, size=len(items)).astype(np.float32)              # a third explicit zeros
        order = rng.permutation(len(items))
        t_rows.append(np.asarray(items, np.int64)[order])
        t_vals.append(np.asarray(vals, np.float32)[order])
        ex_rows.append(rng.permutation(seen))

    def csr(rows, vals):
        indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
        return scipy.sparse.csr_matrix((np.concatenate(vals).astype(np.float32), np.concatenate(rows).astype(np.int32),
                                        indptr), shape=(nu, ni))
    ex = csr(ex_rows, [rng.integers(0, 3, size=len(r)).astype(np.float32) for r in ex_rows])
    return ex, csr(t_rows, t_vals)


CASES = [  # f, bias, ni, ks (out of order): tensor-core path, exact path (f > 128), sort path (K > 1024), K > items
    (64, False, 5000, [50, 10, 100, 1]),
    (33, True, 4096, [20, 5, 3]),
    (256, False, 3000, [5, 100, 20]),
    (64, False, 3000, [1500, 10, 2000]),
    (16, False, 300, [400, 10, 299]),
]


@gpu
@pytest.mark.parametrize("f,bias,ni,ks", CASES)
def test_per_user_metrics_equal_the_oracle(cuda_device, f, bias, ni, ks):
    nu = 60
    K = max(ks)
    m, U, V = make_model(f, bias, ni, nu, seed=ni + f)
    X, Test = make_data(U, V, bias, K, seed=f + K)
    rng = np.random.default_rng(2)
    users = np.concatenate([rng.permutation(nu), rng.integers(0, nu, 13)])    # shuffled, with repeats
    ids = m.recommend(users, K, exclude=X)
    want = oracle_per_user(ids, users, Test, ks)
    T = DeviceCSR.from_scipy(Test, cuda_device).sorted()
    got = engine.topn_metrics(torch.from_numpy(ids).to(cuda_device), torch.from_numpy(users).to(cuda_device), T,
                              ks).cpu().numpy()
    nan = np.isnan(want[:, 0, 0])
    assert nan.sum() >= 2 * (nu // 7) and np.all(np.isnan(got[nan]))          # empty and zeros-only rows
    assert not np.isnan(got[~nan]).any()
    hits = got[~nan][:, :, 1] * np.asarray(ks)                                # Precision@k * k is a hit count
    np.testing.assert_allclose(hits, np.rint(hits), rtol=0, atol=1e-9)
    np.testing.assert_array_equal(np.rint(hits), np.rint(want[~nan][:, :, 1] * np.asarray(ks)))
    np.testing.assert_allclose(got[~nan], want[~nan], rtol=1e-12, atol=0)
    all_excluded = [r for r, u in enumerate(users) if u % 7 == 2 and not nan[r]]
    assert all_excluded and np.all(got[all_excluded] == 0)
    assert got[~nan][:, :, 4].sum() > 0 and (got[~nan][:, :, 2] > 0.5).any()  # the data has hits near the top

    res = m.eval_ranking(Test, topn=ks, exclude=X, users=users)
    means = oracle_means(want, ks)
    assert res["users"] == means["users"] and set(res) == set(means)
    for key in means:
        assert isinstance(res[key], (float, int))
        np.testing.assert_allclose(res[key], means[key], rtol=1e-12, atol=1e-15)


@gpu
def test_hand_built_closed_form(cuda_device):
    """Scores fall with the item id, so the ranking is 0, 1, 2, ... minus the excluded items, and the test items sit at
    known positions. User 0: item 1 excluded, list 0 2 3 4 5, T = {2, 5, 100}: hits at positions 2 and 5. User 1:
    T = {1}, all excluded. User 2: T = {0}, hit at position 1. User 3: empty test row."""
    ni, f = 300, 16
    U = np.zeros((4, f), np.float32)
    U[:, 0] = 1
    V = np.zeros((ni, f), np.float32)
    V[:, 0] = np.arange(ni, 0, -1, dtype=np.float32) / 512
    m = WMF(num_items=ni, num_users=4, dim=f, gamma=0.1, weighted=True)
    m.users, m.items = U, V
    X = scipy.sparse.csr_matrix(([1.0, 1.0], ([0, 1], [1, 1])), shape=(4, ni), dtype=np.float32)
    Test = scipy.sparse.csr_matrix(([1.0, 3.0, 1.0, 2.0, 1.0], ([0, 0, 0, 1, 2], [100, 5, 2, 1, 0])), shape=(4, ni),
                                   dtype=np.float32)
    ks = [5, 1, 2]
    users = np.arange(4)
    ids = m.recommend(users, 5, exclude=X)
    np.testing.assert_array_equal(ids[0], [0, 2, 3, 4, 5])
    got = engine.topn_metrics(torch.from_numpy(ids).to(cuda_device), torch.from_numpy(users).to(cuda_device),
                              DeviceCSR.from_scipy(Test, cuda_device).sorted(), ks).cpu().numpy()
    d = [1 / math.log2(i + 1) for i in range(1, 6)]   # discount of positions 1..5
    want0 = {5: [2 / 3, 2 / 5, (d[1] + d[4]) / (d[0] + d[1] + d[2]), (1 / 2 + 2 / 5) / 3, 1],
             1: [0, 0, 0, 0, 0],
             2: [1 / 3, 1 / 2, d[1] / (d[0] + d[1]), (1 / 2) / 2, 1]}
    want2 = {k: [1, 1 / k, 1, 1, 1] for k in ks}
    for j, k in enumerate(ks):
        np.testing.assert_allclose(got[0, j], want0[k], rtol=1e-12, atol=0)
        np.testing.assert_array_equal(got[1, j], 0)
        np.testing.assert_allclose(got[2, j], want2[k], rtol=1e-12, atol=0)
    assert np.all(np.isnan(got[3]))
    res = m.eval_ranking(Test, topn=ks, exclude=X, users=users)
    assert res["users"] == 3
    np.testing.assert_allclose(res["Recall@5"], (2 / 3 + 0 + 1) / 3, rtol=1e-12)
    np.testing.assert_allclose(res["NDCG@2"], (d[1] / (d[0] + d[1]) + 0 + 1) / 3, rtol=1e-12)
    np.testing.assert_allclose(res["MAP@5"], ((1 / 2 + 2 / 5) / 3 + 0 + 1) / 3, rtol=1e-12)
    np.testing.assert_allclose(res["HitRate@1"], 1 / 3, rtol=1e-12)
    # default users: the rows with stored entries (user 3 is not ranked); the same three users are evaluated
    assert m.eval_ranking(Test, topn=ks, exclude=X) == res


@gpu
def test_eval_ranking_reproducible_and_chunk_independent(cuda_device, monkeypatch):
    ni, nu, ks = 4096, 300, np.array([10, 50, 3])
    m, U, V = make_model(64, False, ni, nu, seed=9)
    X, Test = make_data(U, V, False, 50, seed=9)
    a = m.eval_ranking(Test, topn=ks, exclude=X)
    b = m.eval_ranking(DeviceCSR.from_scipy(Test, cuda_device), topn=ks, exclude=DeviceCSR.from_scipy(X, cuda_device))
    assert a == b
    for ids in (50 * 7, 50, 1):       # chunks of 7 users, then 1 user
        monkeypatch.setattr(wmf_model, "_EVAL_CHUNK_IDS", ids)
        assert m.eval_ranking(Test, topn=ks, exclude=X) == a
    monkeypatch.undo()
    users = np.flatnonzero(np.diff(Test.indptr) > 0)
    assert a["users"] == oracle_means(oracle_per_user(m.recommend(users, 50, exclude=X), users, Test, ks), ks)["users"]
    # nothing excluded: the lists are recommend(users, K) = rank_batch over all items
    c = m.eval_ranking(Test, topn=ks)
    want = oracle_means(oracle_per_user(m.recommend(users, 50), users, Test, ks), ks)
    assert c["users"] == want["users"]
    for key in want:
        np.testing.assert_allclose(c[key], want[key], rtol=1e-12, atol=1e-15)
    assert c["Recall@50"] != a["Recall@50"]
    # an int topn
    assert m.eval_ranking(Test, topn=10, exclude=X) == {k: v for k, v in a.items() if k.endswith("@10") or k == "users"}


@gpu
def test_eval_ranking_input_errors(cuda_device):
    m, U, V = make_model(16, False, 400, 10, seed=4)
    T = scipy.sparse.random(10, 400, density=0.05, format="csr", dtype=np.float32, random_state=0)
    for topn in ([0], [5, 5], np.arange(1, 18), [[1, 2]], [1.5], [], np.array([True])):
        with pytest.raises(ValueError):
            m.eval_ranking(T, topn=topn)
    with pytest.raises(ValueError):
        m.eval_ranking(scipy.sparse.csr_matrix((10, 399), dtype=np.float32))
    with pytest.raises(ValueError):
        m.eval_ranking(T, exclude=scipy.sparse.csr_matrix((11, 400), dtype=np.float32))
    for users in ([-1], [0, 10]):
        with pytest.raises(ValueError):
            m.eval_ranking(T, users=np.array(users))
    taller = scipy.sparse.random(12, 400, density=0.5, format="csr", dtype=np.float32, random_state=1)
    with pytest.raises(ValueError):
        m.eval_ranking(taller)                   # default users past the user factors
    with pytest.raises(ValueError):
        m.eval_ranking(taller, users=np.array([11]))
    assert m.eval_ranking(taller, users=np.arange(10))["users"] == 10


def test_topn_metrics_rejects_bad_arguments_without_a_device():
    build.build()
    lib = _lib.load()
    p = 8   # a non-null address; never dereferenced: every call below fails its checks before any CUDA call
    ks = np.array([10, 1, 5], dtype=np.int32)
    k = ks.ctypes.data

    def run(ids=p, nu=4, K=10, users=p, ip=p, ix=p, dt=p, ksp=k, nk=3, out=p):
        return lib.wmf_topn_metrics(ids, nu, K, users, ip, ix, dt, ksp, nk, out, None)
    assert run(nu=-1) == 1 and "bad sizes" in _lib.last_error()
    assert run(K=0) == 1
    assert run(nk=0) == 1
    many = np.arange(1, 18, dtype=np.int32)
    assert run(K=20, ksp=many.ctypes.data, nk=17) == 1 and "nk=17" in _lib.last_error()
    assert run(K=9) == 1 and "cutoff 10" in _lib.last_error()            # cutoff past K
    zero = np.array([0], dtype=np.int32)
    assert run(ksp=zero.ctypes.data, nk=1) == 1
    twice = np.array([3, 3], dtype=np.int32)
    assert run(ksp=twice.ctypes.data, nk=2) == 1 and "twice" in _lib.last_error()
    assert run(ksp=None) == 1
    for name in ("ids", "users", "ip", "ix", "dt", "out"):
        assert run(**{name: None}) == 1 and "null" in _lib.last_error()
    assert run(nu=0, ids=None, users=None, out=None) == 0                  # nothing to do, nothing launched
    assert lib.wmf_topn_metrics_reduce(p, -1, 3, p, p, 1 << 20, None) == 1
    assert lib.wmf_topn_metrics_reduce(p, 10, 17, p, p, 1 << 20, None) == 1
    assert lib.wmf_topn_metrics_reduce(p, 10, 0, p, p, 1 << 20, None) == 1
    assert lib.wmf_topn_metrics_reduce(p, 10, 3, None, p, 1 << 20, None) == 1
    assert lib.wmf_topn_metrics_reduce(None, 10, 3, p, p, 1 << 20, None) == 1
    assert lib.wmf_topn_metrics_reduce(p, 10, 3, p, None, 0, None) == 2                   # workspace
    need = lib.wmf_topn_metrics_workspace_bytes(1000, 4)
    assert need >= 21 * 8 and lib.wmf_topn_metrics_reduce(p, 1000, 4, p, p, need - 1, None) == 2
    assert lib.wmf_topn_metrics_workspace_bytes(1000, 17) == 0


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, scipy.sparse, torch, torch.distributed as dist
from recmodel_b200 import WMF, wmf_model
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rng = np.random.default_rng(0)
nu, ni = 1001, 6000
m = WMF(num_items=ni, num_users=nu, dim=64, gamma=0.1, weighted=True)
m.users = (rng.standard_normal((nu, 64)) * 0.5).astype(np.float32)
m.items = (rng.standard_normal((ni, 64)) * 0.5).astype(np.float32)
X = scipy.sparse.random(nu, ni, density=0.05, format="csr", dtype=np.float32, random_state=1)
T = scipy.sparse.random(nu, ni, density=0.01, format="csr", dtype=np.float32, random_state=2)
for ks in ([10, 50], [700, 3]):
    a = m.eval_ranking(T, topn=ks, exclude=X, distributed=True)
    b = m.eval_ranking(T, topn=ks, exclude=X)
    assert a == b, (ks, a, b)
wmf_model._EVAL_CHUNK_IDS = 50 * 97
assert m.eval_ranking(T, topn=[10, 50], exclude=X, distributed=True) == m.eval_ranking(T, topn=[10, 50], exclude=X)
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


@gpu
def test_eval_ranking_distributed_equals_local(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc_per_node", "2",
                        f"--master_port={29500 + (os.getpid() + 7) % 2000}", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok 0" in r.stdout and "ok 1" in r.stdout, r.stdout + r.stderr
