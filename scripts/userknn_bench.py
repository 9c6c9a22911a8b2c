"""UserKNN training, recommend and eval_ranking at ML-20M shape: the data of scripts/knn_bench.py
(make_counts_cached(138 493, 26 744, 20 M) split 80/20 with utils.train_test_split_sparse_mat), UserKNN trained on
the train half with k = 100 and cosine similarity, then top-100 over each test user's unseen items (train entries
excluded) and Recall / Precision / NDCG / MAP / hit rate at 10 / 20 / 50 / 100.

One JSON line, all numbers from the same run:
 - train_s: host clock around UserKNN.train (canonical copy, upload, transpose, device training; ends in a device
   synchronise), median of --train-reps after one warm-up. train_device_ms: device events around
   engine.knn_train(X^T, X) alone.
 - recommend_ms: device events around the device part of recommend (top-100 of every test user, matrices resident),
   after a warm-up; median and spread ((max - min) / median). eval_ms: the same for the device part of eval_ranking;
   eval_api_ms: host clock around the public call with SciPy matrices in.
 - kernels_ms_*: torch.profiler device time per kernel of one training and of one recommend, in a separate pass after
   the timed ones.
 - work: sum_i pop_i^2 (co-occurrence updates of training, pop_i the users of item i), and sum over the test users u
   of sum over the neighbours v of u of nnz_v (read-modify-writes of the score tiles), computed here from the data and
   the trained model; score_rate: the latter over the profiled time of userknn_score_tile_kernel.
 - quality: Recall@10, NDCG@10, Recall@100 of UserKNN and of ItemKNN (k 100, cosine) on the same split, same run.
 - cpu_arm: SciPy int64 P_R P^T (the counts of a fixed seeded sample of user rows R against all users) plus per-row
   NumPy cosine and top-k, timed on this host and EXTRAPOLATED to all users by n / |R|.
 - oracle_equal: the neighbour rows of the CPU arm and sampled users' lists against the NumPy definitions.

    python scripts/userknn_bench.py [--reps 5] [--train-reps 3] [--sample-users 200] [--list-users 40] [--out FILE]
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

from knn_bench import cpu_rows, profiled, timed
from recommend_bench import gpu_info
from recmodel_b200 import ItemKNN, UserKNN, engine, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.knn_model import _canonical
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, K, TOPN = 138_493, 26_744, 20_000_000, 100, 100
KS = [10, 20, 50, 100]


def oracle_list(X, N, u, topn):
    """User u's top-n over its unseen items by the definitions: sim(u, v) * x_v summed over the neighbours v of u in
    ascending v, ties to the lower id."""
    acc = np.zeros(X.shape[1], np.float64)
    for e in range(N.indptr[u], N.indptr[u + 1]):
        v = N.indices[e]
        lo, hi = X.indptr[v], X.indptr[v + 1]
        acc[X.indices[lo:hi]] += N.data[e] * X.data[lo:hi].astype(np.float32).astype(np.float64)
    cand = np.delete(np.arange(X.shape[1]), X.indices[X.indptr[u]:X.indptr[u + 1]])
    out = np.full(topn, -1, np.int64)
    best = cand[np.lexsort((cand, -acc[cand]))][:topn]
    out[:len(best)] = best
    return out


def log(msg):
    print(f"[{time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def spread(xs):
    return round((max(xs) - min(xs)) / float(np.median(xs)), 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--train-reps", type=int, default=3)
    ap.add_argument("--sample-users", type=int, default=200)
    ap.add_argument("--list-users", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    full = make_counts_cached(USERS, ITEMS, NNZ)
    Train, Test = utils.train_test_split_sparse_mat(full)
    m = UserKNN(num_items=ITEMS, num_users=USERS, device=dev)
    log("data ready")
    m.train(Train, k=K)   # warm-up
    torch.cuda.synchronize(dev)
    log("warm-up training done")
    train_s = []
    for _ in range(args.train_reps):
        t0 = time.perf_counter()
        m.train(Train, k=K)
        torch.cuda.synchronize(dev)
        train_s.append(time.perf_counter() - t0)
    X = m._X
    XT = X.transpose()
    N_d = m._W_device()

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
    log("warm-up recommend and eval done")
    train_dev_ms = timed(lambda: engine.knn_train(XT, X, K, "cosine", 0.0), args.train_reps, dev)
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
    N2 = engine.knn_train(XT, X, K, "cosine", 0.0)
    same_train = all(bool(torch.equal(a, b)) for a, b in zip(N2, N_d))
    del N2

    log("timed passes done")
    kernels_train = profiled(lambda: engine.knn_train(XT, X, K, "cosine", 0.0), dev)
    kernels_rec = profiled(rec, dev)

    item = ItemKNN(num_items=ITEMS, num_users=USERS, device=dev)
    item.train(Train, k=K)
    res_item = item.eval_ranking(Test, topn=KS, exclude=Train)
    del item

    log("ItemKNN done")
    # the CPU arm and the oracle, on fixed seeded samples: user rows are item rows of X^T
    Xc = _canonical(Train)
    P = Xc.T.tocsr()
    P.data = np.ones_like(P.data, dtype=np.int64)
    P = scipy.sparse.csc_matrix(P.astype(np.int64))   # items x users: column u is user u's pattern
    pop = np.diff(P.indptr).astype(np.float64)        # c_uu, the items of user u
    P_csr = P.tocsr()
    rng = np.random.default_rng(2024)
    rows = np.sort(rng.choice(USERS, size=args.sample_users, replace=False))
    t0 = time.perf_counter()
    cpu = cpu_rows(P, P_csr, pop, rows, K)
    cpu_s = time.perf_counter() - t0
    Nh = m.neighbors
    n_ok = all(np.array_equal(Nh.indices[Nh.indptr[a]:Nh.indptr[a + 1]], ids)
               and np.array_equal(Nh.data[Nh.indptr[a]:Nh.indptr[a + 1]].view(np.uint64), sims.view(np.uint64))
               for a, (ids, sims) in zip(rows, cpu))
    sample_u = np.sort(rng.choice(users, size=min(args.list_users, len(users)), replace=False))
    ids_h = ids0.cpu().numpy()
    pos = np.searchsorted(users, sample_u)
    lists_ok = all(np.array_equal(ids_h[p], oracle_list(Xc, Nh, int(u), TOPN)) for p, u in zip(pos, sample_u))

    nnz_u = np.diff(Xc.indptr).astype(np.int64)
    pop_i = np.diff(Xc.tocsc().indptr).astype(np.int64)
    per_user = np.add.reduceat(np.append(nnz_u[Nh.indices], 0), Nh.indptr[:-1]) * (np.diff(Nh.indptr) > 0)
    votes = int(per_user[users].sum())
    score_key = next((k for k in kernels_rec if "userknn_score_tile_kernel" in k), None)
    score_ms = kernels_rec.get(score_key)
    rec_med = float(np.median(rec_ms))
    pick = ("Recall@10", "NDCG@10", "Recall@100")
    line = {
        "metric": "userknn_recommend_device_ms", "value": rec_med, "unit": "ms",
        "what": f"UserKNN (k {K}, cosine, shrink 0) trained on the 80% split of make_counts_cached({USERS}, {ITEMS}, "
                f"{NNZ}); recommend top-{TOPN} over each user's unseen items, {len(users)} test users x {ITEMS} items, "
                f"train entries excluded; device events, median of {args.reps} after a warm-up (measured)",
        "train_s": [round(x, 3) for x in train_s], "train_median_s": float(np.median(train_s)),
        "train_device_ms": [round(x, 2) for x in train_dev_ms],
        "train_device_median_ms": float(np.median(train_dev_ms)),
        "train_bitwise_equal_across_runs": bool(same_train),
        "recommend_ms": [round(x, 3) for x in rec_ms], "recommend_spread": spread(rec_ms),
        "eval_ranking_ks": KS, "eval_ms": [round(x, 3) for x in eval_ms], "eval_median_ms": float(np.median(eval_ms)),
        "eval_spread": spread(eval_ms),
        "eval_api_ms": [round(x, 1) for x in api_ms], "eval_api_median_ms": float(np.median(api_ms)),
        "bitwise_equal_across_reps": bool(same),
        "kernels_ms_one_train_profiled": kernels_train,
        "kernels_ms_one_recommend_profiled": kernels_rec,
        "work": {"what": "computed from the data and the trained model",
                 "cooccurrence_updates_sum_i_pop_i_sq": int((pop_i * pop_i).sum()),
                 "score_updates_sum_u_sum_v_nnz_v": votes, "neighbors_nnz": int(Nh.nnz),
                 "longest_user_row": int(nnz_u.max()), "median_user_row": float(np.median(nnz_u)),
                 "longest_item_column": int(pop_i.max()),
                 "train_nnz": int(Xc.nnz), "test_nnz": int(Test.nnz)},
        "score_rate_updates_per_s": (votes / (score_ms / 1e3)) if score_ms else None,
        "quality": {"UserKNN": {k: res[k] for k in pick}, "ItemKNN": {k: res_item[k] for k in pick}},
        "cpu_arm": {"what": "SciPy int64 P_R P^T of a seeded sample of user rows R, then per-row NumPy cosine and top-k "
                            "(lexsort), single process on the GPU host; EXTRAPOLATED to all users by n / |R|",
                    "sample_users": int(len(rows)), "sample_s": round(cpu_s, 3),
                    "extrapolated_all_users_s": round(cpu_s / len(rows) * USERS, 1)},
        "oracle_equal_sampled_neighbor_rows": bool(n_ok),
        "oracle_equal_sampled_users": bool(lists_ok), "sampled_users": int(len(sample_u)),
        "result": res,
        "provenance": {"measured": "train_*, recommend_*, eval_*, kernels_ms_*, score_rate_updates_per_s, quality, "
                                   "result, cpu_arm.sample_s, oracle_equal_*, on the card named here",
                       "computed": "work: counted from the data and the trained model, not timed",
                       "extrapolated": "cpu_arm.extrapolated_all_users_s"},
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
