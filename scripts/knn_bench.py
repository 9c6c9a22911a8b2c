"""ItemKNN training, recommend and eval_ranking at ML-20M shape: the data of scripts/ease_rank_bench.py
(make_counts_cached(138 493, 26 744, 20 M) split 80/20 with utils.train_test_split_sparse_mat), ItemKNN trained on
the train half with k = 100 and cosine similarity, then top-100 over each test user's unseen items (train entries
excluded) and Recall / Precision / NDCG / MAP / hit rate at 10 / 20 / 50 / 100.

One JSON line, all numbers from the same run:
 - train_s: host clock around ItemKNN.train (canonical copy, upload, transpose, device training; ends in a device
   synchronise), median of --train-reps after one warm-up.
 - recommend_ms: device events around the device part of recommend (top-100 of every test user, matrices resident),
   median of the reps after a warm-up. eval_ms: the same for the device part of eval_ranking; eval_api_ms: host clock
   around the public call with SciPy matrices in.
 - kernels_ms_*: torch.profiler device time per kernel of one training and of one recommend, in a separate pass after
   the timed ones.
 - work: sum_u nnz_u^2 (co-occurrence updates of training) and sum over the test users of sum_j |W_j| over their train
   entries j (read-modify-writes of the score tiles), computed here from the data and the trained model.
 - cpu_arm: SciPy B_R^T B (int64 counts of a fixed seeded sample of item rows R against all items) plus per-row NumPy
   cosine and top-k, timed on this host and EXTRAPOLATED to all items by n / |R|.
 - oracle_equal: sampled rows of W (from the CPU arm) and sampled users' lists against the NumPy definitions.

    python scripts/knn_bench.py [--reps 5] [--train-reps 3] [--sample-items 400] [--sample-users 40] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np
import scipy.sparse
import torch

from recommend_bench import gpu_info
from recmodel_b200 import engine, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.knn_model import ItemKNN, _canonical
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, K, TOPN = 138_493, 26_744, 20_000_000, 100, 100
KS = [10, 20, 50, 100]


def cpu_rows(P, P_csr, pop, rows, k):
    """(ids, sims) per item row of ``rows``: the cosine neighbours by the definitions, on the host (P: the binary
    pattern as CSC for the column slice, P_csr the same as CSR)."""
    C = (P[:, rows].T @ P_csr).tocsr()
    C.sort_indices()
    out = []
    for r, a in enumerate(rows):
        b = C.indices[C.indptr[r]:C.indptr[r + 1]].astype(np.int64)
        c = C.data[C.indptr[r]:C.indptr[r + 1]].astype(np.float64)
        keep = (b != a) & (c > 0)
        b, c = b[keep], c[keep]
        s = c / (np.sqrt(pop[a]) * np.sqrt(pop[b]) + 0.0)
        top = np.lexsort((b, -s))[:k]
        top = top[np.argsort(b[top])]
        out.append((b[top], s[top]))
    return out


def oracle_list(X, W, u, topn):
    acc = np.zeros(W.shape[1], np.float64)
    for e in range(X.indptr[u], X.indptr[u + 1]):
        j = X.indices[e]
        lo, hi = W.indptr[j], W.indptr[j + 1]
        acc[W.indices[lo:hi]] += np.float64(np.float32(X.data[e])) * W.data[lo:hi]
    cand = np.delete(np.arange(W.shape[1]), X.indices[X.indptr[u]:X.indptr[u + 1]])
    out = np.full(topn, -1, np.int64)
    best = cand[np.lexsort((cand, -acc[cand]))][:topn]
    out[:len(best)] = best
    return out


def timed(fn, reps, dev):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    out = []
    for _ in range(reps):
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize(dev)
        out.append(ev[0].elapsed_time(ev[1]))
    return out


def profiled(fn, dev):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize(dev)
    kernels = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            kernels[e.key[:80]] = round(t / 1e3, 3)
    return kernels


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--train-reps", type=int, default=3)
    ap.add_argument("--sample-items", type=int, default=400)
    ap.add_argument("--sample-users", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    full = make_counts_cached(USERS, ITEMS, NNZ)
    Train, Test = utils.train_test_split_sparse_mat(full)
    m = ItemKNN(num_items=ITEMS, num_users=USERS, device=dev)
    m.train(Train, k=K)   # warm-up
    torch.cuda.synchronize(dev)
    train_s = []
    for _ in range(args.train_reps):
        t0 = time.perf_counter()
        m.train(Train, k=K)
        torch.cuda.synchronize(dev)
        train_s.append(time.perf_counter() - t0)
    X = m._X
    XT = X.transpose()
    W_d = m._W_device()

    ex = DeviceCSR.from_scipy(Train, dev)
    T = DeviceCSR.from_scipy(Test, dev).sorted()
    users = np.flatnonzero(np.diff(Test.indptr) > 0)
    users_d = torch.from_numpy(users).to(dev)

    def rec():
        return m._recommend_ids(*m._X_and_W(), users_d, TOPN, ex)

    def ev_device():
        return ranking.eval_ranking_sums(lambda u, k, e: m._recommend_ids(*m._X_and_W(), u, k, e), ITEMS, T, ex,
                                         users_d, np.asarray(KS, np.int64))

    ids0 = rec()
    sums0 = ev_device()
    torch.cuda.synchronize(dev)
    train_dev_ms = timed(lambda: engine.knn_train(X, XT, K, "cosine", 0.0), args.train_reps, dev)
    rec_ms, eval_ms, api_ms, same = [], [], [], True
    for _ in range(args.reps):   # the two device paths alternated
        out = []
        rec_ms += timed(lambda: out.append(rec()), 1, dev)
        eval_ms += timed(lambda: out.append(ev_device()), 1, dev)
        same &= bool(torch.equal(out[0], ids0)) and bool(torch.equal(out[1], sums0))
    res = m.eval_ranking(Test, topn=KS, exclude=Train)   # warm-up of the public call
    for _ in range(args.reps):
        t0 = time.perf_counter()
        res = m.eval_ranking(Test, topn=KS, exclude=Train)
        api_ms.append((time.perf_counter() - t0) * 1e3)
    W2 = engine.knn_train(X, XT, K, "cosine", 0.0)
    same_train = all(bool(torch.equal(a, b)) for a, b in zip(W2, W_d))

    kernels_train = profiled(lambda: engine.knn_train(X, XT, K, "cosine", 0.0), dev)
    kernels_rec = profiled(rec, dev)

    # the CPU arm and the oracle, on fixed seeded samples
    Xc = _canonical(Train)
    P = Xc.copy()
    P.data = np.ones_like(P.data, dtype=np.int64)
    P = scipy.sparse.csc_matrix(P.astype(np.int64))
    pop = np.diff(P.indptr).astype(np.float64)
    P_csr = P.tocsr()
    rng = np.random.default_rng(2024)
    rows = np.sort(rng.choice(ITEMS, size=args.sample_items, replace=False))
    t0 = time.perf_counter()
    cpu = cpu_rows(P, P_csr, pop, rows, K)
    cpu_s = time.perf_counter() - t0
    Wh = m.neighbors
    w_ok = all(np.array_equal(Wh.indices[Wh.indptr[a]:Wh.indptr[a + 1]], ids)
               and np.array_equal(Wh.data[Wh.indptr[a]:Wh.indptr[a + 1]].view(np.uint64), sims.view(np.uint64))
               for a, (ids, sims) in zip(rows, cpu))
    sample_u = np.sort(rng.choice(users, size=min(args.sample_users, len(users)), replace=False))
    ids_h = ids0.cpu().numpy()
    pos = np.searchsorted(users, sample_u)
    lists_ok = all(np.array_equal(ids_h[p], oracle_list(Xc, Wh, int(u), TOPN)) for p, u in zip(pos, sample_u))

    nnz_u = np.diff(Xc.indptr).astype(np.int64)
    w_len = np.diff(Wh.indptr).astype(np.int64)
    votes = int(sum(int(w_len[Xc.indices[Xc.indptr[u]:Xc.indptr[u + 1]]].sum()) for u in users))
    rec_med = float(np.median(rec_ms))
    line = {
        "metric": "itemknn_recommend_device_ms", "value": rec_med, "unit": "ms",
        "what": f"ItemKNN (k {K}, cosine, shrink 0) trained on the 80% split of make_counts_cached({USERS}, {ITEMS}, "
                f"{NNZ}); recommend top-{TOPN} over each user's unseen items, {len(users)} test users x {ITEMS} items, "
                f"train entries excluded; device events, median of {args.reps} after a warm-up",
        "train_s": [round(x, 3) for x in train_s], "train_median_s": float(np.median(train_s)),
        "train_device_ms": [round(x, 2) for x in train_dev_ms],
        "train_bitwise_equal_across_runs": bool(same_train),
        "recommend_ms": [round(x, 3) for x in rec_ms],
        "eval_ranking_ks": KS, "eval_ms": [round(x, 3) for x in eval_ms], "eval_median_ms": float(np.median(eval_ms)),
        "eval_api_ms": [round(x, 1) for x in api_ms], "eval_api_median_ms": float(np.median(api_ms)),
        "bitwise_equal_across_reps": bool(same),
        "kernels_ms_one_train_profiled": kernels_train,
        "kernels_ms_one_recommend_profiled": kernels_rec,
        "work": {"cooccurrence_updates_sum_nnz_u_sq": int((nnz_u * nnz_u).sum()),
                 "score_updates_sum_u_sum_j_W_j": votes, "W_nnz": int(Wh.nnz),
                 "train_nnz": int(Xc.nnz), "test_nnz": int(Test.nnz)},
        "cpu_arm": {"what": "SciPy int64 B_R^T B of a seeded sample of item rows R, then per-row NumPy cosine and top-k "
                            "(lexsort), single process on the GPU host; EXTRAPOLATED to all items by n / |R|",
                    "sample_items": int(len(rows)), "sample_s": round(cpu_s, 3),
                    "extrapolated_all_items_s": round(cpu_s / len(rows) * ITEMS, 1)},
        "oracle_equal_sampled_W_rows": bool(w_ok),
        "oracle_equal_sampled_users": bool(lists_ok), "sampled_users": int(len(sample_u)),
        "result": res,
        **info,
    }
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
