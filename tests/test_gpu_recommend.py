"""WMF.recommend: top-N over every item a user has not interacted with, exclusion applied inside the device ranking
(include/wmf_b200.h: wmf_score_topk_exclude). Row k must equal rank(np.delete(arange(I), seen[users[k]]), users[k], N)
element for element, padded with -1, on the tensor-core path, the exact path and the sort path (topn > 1024)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse
import torch

from conftest import ROOT
from oracle import wmf_oracle as orc
from recmodel_b200 import WMF, engine, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts

pytestmark = pytest.mark.gpu


def make_model(f, bias, ni, nu, seed, equal=False):
    rng = np.random.default_rng(seed)
    if equal:
        U, V = np.ones((nu, f), np.float32), np.ones((ni, f), np.float32)
    else:
        U = (rng.standard_normal((nu, f)) * 0.5).astype(np.float32)
        V = (rng.standard_normal((ni, f)) * 0.5).astype(np.float32)
        V[ni // 2] = V[ni // 3]  # an exact tie
    m = WMF(num_items=ni, num_users=nu, dim=f - 1 if bias else f, gamma=0.1, weighted=True, bias=bias)
    m.users, m.items = U, V
    return m, U, V


def seen_lists(U, V, bias, topn, seed):
    """Per user: the items to exclude. Covers no seen items, random subsets, more than ni - topn seen items,
    everything seen, and the user's highest-scoring items all seen."""
    nu, ni = U.shape[0], V.shape[0]
    rng = np.random.default_rng(seed)
    seen = []
    for u in range(nu):
        kind = u % 6
        if kind == 0:
            s = np.empty(0, np.int64)
        elif kind == 1:
            s = rng.choice(ni, size=int(rng.integers(1, max(2, ni // 10))), replace=False)
        elif kind == 2:
            s = rng.choice(ni, size=ni - max(1, topn // 2), replace=False)       # fewer than topn unseen: padded row
        elif kind == 3 and u == 3:
            s = np.arange(ni)                                                    # everything seen
        elif kind == 3:
            s = rng.choice(ni, size=int(rng.integers((ni - topn) // 2, ni - topn)), replace=False)
        elif kind == 4:
            sc = orc.rank_scores(U, V, np.arange(ni), u, bias)
            s = np.argsort(-sc, kind="stable")[:min(ni - 1, 3 * topn)]          # the best items are all seen
        else:
            s = rng.choice(ni, size=int(rng.integers(1, 64)), replace=False)
        seen.append(np.asarray(s, dtype=np.int64))
    return seen


def to_csr(seen, ni, seed):
    """Unsorted rows, duplicate entries and explicit zeros: every stored entry excludes its item."""
    rng = np.random.default_rng(seed)
    rows = []
    for s in seen:
        r = rng.permutation(s)
        if len(r) > 3:
            r = np.concatenate([r, r[:3]])                # duplicates
        rows.append(r)
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    indices = np.concatenate(rows).astype(np.int32) if rows else np.empty(0, np.int32)
    data = rng.integers(0, 3, size=len(indices)).astype(np.float32)  # a third of them explicit zeros
    return scipy.sparse.csr_matrix((data, indices, indptr), shape=(len(seen), ni))


def per_user_rank(m, seen, users, topn):
    ni = m.items.shape[0]
    out = np.full((len(users), topn), -1, dtype=np.int64)
    for k, u in enumerate(users):
        cand = np.delete(np.arange(ni), seen[u])
        if len(cand):
            r = m.rank(cand, int(u), topn)
            out[k, :len(r)] = r
    return out


def check_against_oracle(got, U, V, bias, seen, users, topn):
    ni = V.shape[0]
    for k, u in enumerate(users):
        cand = np.delete(np.arange(ni), seen[u])
        n = min(topn, len(cand))
        assert np.all(got[k, n:] == -1)
        if n == 0:
            continue
        s = orc.rank_scores(U, V, np.arange(ni), u, bias)
        kth = np.sort(s[cand])[-n]
        sel = got[k, :n]
        assert len(set(sel.tolist())) == n and not np.isin(sel, seen[u]).any()
        assert set(cand[s[cand] > kth].tolist()) <= set(sel.tolist()) <= set(cand[s[cand] >= kth].tolist())
        assert np.all(np.diff(s[sel]) <= 0)


CASES = [  # f, bias, ni, topn: tensor-core path (f + bias <= 128, topn <= 512 and <= ni / 32), exact, sort
    (16, False, 300, 9),
    (65, True, 5000, 100),
    (128, False, 26_744, 100),
    (128, False, 100_000, 512),
    (32, False, 4096, 10),
    (256, False, 3000, 100),   # exact path: f > 128
    (128, False, 26_744, 700), # exact path: topn > 512
    (64, False, 3000, 2000),   # sort path: topn > 1024
]


@pytest.mark.parametrize("f,bias,ni,topn", CASES)
def test_recommend_equals_per_user_rank(cuda_device, monkeypatch, f, bias, ni, topn):
    nu = 48
    m, U, V = make_model(f, bias, ni, nu, seed=ni + f + topn)
    seen = seen_lists(U, V, bias, topn, seed=f + topn)
    X = to_csr(seen, ni, seed=ni)
    rng = np.random.default_rng(1)
    users = np.concatenate([rng.permutation(nu), rng.integers(0, nu, 17)])  # shuffled, with repeats
    got = m.recommend(users, topn, exclude=X)
    assert got.dtype == np.int64 and got.shape == (len(users), topn)
    assert np.all(got[users == 3] == -1)  # user 3 has seen everything
    np.testing.assert_array_equal(got, per_user_rank(m, seen, users, topn))
    check_against_oracle(got, U, V, bias, seen, users, topn)
    tc = ((f + bias) <= 128 and topn <= 512 and topn <= ni // 32)
    if tc:
        # no list overflowed: the tensor-core path answered alone, padded rows included
        users_d = torch.from_numpy(users).to(cuda_device)
        ex = DeviceCSR.from_scipy(X, cuda_device).sorted()
        ids, _, fixup = engine.score_topk_exclude(users_d, ex, m.users_device, m.items_device, topn, bias=bias)
        assert int(fixup.item()) == 0
        np.testing.assert_array_equal(ids.cpu().numpy(), got)
        monkeypatch.setenv("WMF_SCORE_EXACT", "1")
        np.testing.assert_array_equal(m.recommend(users, topn, exclude=X), got)


def test_recommend_without_exclusion_is_rank_batch(cuda_device):
    m, U, V = make_model(64, False, 3000, 40, seed=3)
    users = np.array([5, 1, 5, 39, 0])
    np.testing.assert_array_equal(m.recommend(users, 50), m.rank_batch(np.arange(3000), users, 50))
    empty = scipy.sparse.csr_matrix((40, 3000), dtype=np.float32)
    np.testing.assert_array_equal(m.recommend(users, 50, exclude=empty), m.rank_batch(np.arange(3000), users, 50))
    ex = DeviceCSR.from_scipy(empty, cuda_device)  # a DeviceCSR is taken as is
    np.testing.assert_array_equal(m.recommend(users, 50, exclude=ex), m.rank_batch(np.arange(3000), users, 50))


def test_rank_batch_sort_path_maps_positions_to_candidate_ids(cuda_device):
    """topn > 1024 over a permuted subset of the items: the stable device sort ranks candidate positions, and the lists
    must report the candidates' ids, an exact tie in candidate order."""
    ni, nu, topn = 3000, 24, 1500
    m, U, V = make_model(64, False, ni, nu, seed=17)
    cand = np.random.default_rng(17).permutation(ni)[:2400]
    p, q = 5, 2000                                  # a tie between positions 5 and 2000, the later id first in cand
    if cand[p] < cand[q]:
        cand[[p, q]] = cand[[q, p]]
    V[cand[q]] = V[cand[p]]
    m.items = V
    got = m.rank_batch(cand, np.arange(nu), topn)
    assert got.shape == (nu, topn) and got.dtype == cand.dtype
    tied = 0
    for u in range(nu):
        s = m.predict(np.full(len(cand), u), cand)
        assert s[p] == s[q]
        np.testing.assert_array_equal(got[u], cand[np.argsort(-s, kind="stable")][:topn])
        tied += np.isin(cand[[p, q]], got[u]).all()
    assert tied > 0                                 # the tie is inside some lists


def test_recommend_all_equal_scores_overflow(cuda_device):
    """All scores equal: every candidate list overflows, the exact kernels redo the call (counted in fixup_users),
    and ties go to the lowest unseen item ids."""
    ni, nu, topn = 5000, 4, 40
    m, U, V = make_model(16, False, ni, nu, seed=0, equal=True)
    seen = [np.arange(0, 10), np.arange(5, 200, 2), np.empty(0, np.int64), np.arange(ni - 20)]
    X = to_csr(seen, ni, seed=2)
    got = m.recommend(np.arange(nu), topn, exclude=X)
    for u in range(nu):
        want = np.full(topn, -1)
        rest = np.delete(np.arange(ni), seen[u])[:topn]
        want[:len(rest)] = rest
        np.testing.assert_array_equal(got[u], want)
    ex = DeviceCSR.from_scipy(X, cuda_device).sorted()
    _, _, fixup = engine.score_topk_exclude(torch.arange(nu, device=cuda_device), ex, m.users_device, m.items_device,
                                            topn)
    assert int(fixup.item()) == 3  # user 3 has 20 unseen items: its list is complete and needs no redo


def test_recommend_input_errors(cuda_device):
    m, U, V = make_model(16, False, 400, 10, seed=4)
    with pytest.raises(ValueError):
        m.recommend(np.arange(10), 5, exclude=scipy.sparse.csr_matrix((10, 399), dtype=np.float32))
    with pytest.raises(ValueError):
        m.recommend(np.array([0, 10]), 5, exclude=scipy.sparse.csr_matrix((10, 400), dtype=np.float32))
    with pytest.raises(ValueError):
        m.recommend(np.array([-1]), 5, exclude=scipy.sparse.csr_matrix((10, 400), dtype=np.float32))


def test_coverage_with_heavy_users_equals_per_user_loop(cuda_device):
    """utils.test_coverage through recommend equals the reference's per-user loop, with users who have seen more
    than 1024 items (the former batched code needed its per-user fallback for them)."""
    full = make_counts(3000, 2500, 400_000, seed=21)
    assert np.diff(full.indptr).max() > 1024
    m, U, V = make_model(32, False, 2500, 3000, seed=21)

    class LoopOnly:
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    got = utils.test_coverage(m, full, 10)
    np.testing.assert_array_equal(got, utils.test_coverage(LoopOnly(), full, 10))
    assert got.sum() == 3000 * 10


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, scipy.sparse, torch, torch.distributed as dist
from recmodel_b200 import WMF
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
rng = np.random.default_rng(0)
nu, ni = 1001, 6000
m = WMF(num_items=ni, num_users=nu, dim=64, gamma=0.1, weighted=True)
m.users = (rng.standard_normal((nu, 64)) * 0.5).astype(np.float32)
m.items = (rng.standard_normal((ni, 64)) * 0.5).astype(np.float32)
X = scipy.sparse.random(nu, ni, density=0.05, format="csr", dtype=np.float32, random_state=1)
users = rng.permutation(nu)
for topn in (50, 700):
    a = m.recommend(users, topn, exclude=X, distributed=True)
    b = m.recommend(users, topn, exclude=X)
    assert np.array_equal(a, b), topn
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_recommend_distributed_equals_local(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc_per_node", "2",
                        f"--master_port={29500 + os.getpid() % 2000}", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok 0" in r.stdout and "ok 1" in r.stdout, r.stdout + r.stderr
