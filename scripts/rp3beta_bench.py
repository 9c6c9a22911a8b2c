"""RP3beta training, recommend and eval_ranking at ML-20M shape: the data of scripts/knn_bench.py
(make_counts_cached(138 493, 26 744, 20 M) split 80/20 with utils.train_test_split_sparse_mat), RP3beta trained on the
train half with alpha = 1, beta = 0.5 and k = 100, then top-100 over each test user's unseen items (train entries
excluded) and Recall / Precision / NDCG / MAP / hit rate at 10 / 20 / 50 / 100.

One JSON line, all numbers from the same run:
 - train_s: host clock around RP3beta.train (canonical copy, scales, upload, transpose, device training; ends in a
   device synchronise), median of --train-reps after one warm-up. train_device_ms: device events around
   engine.rp3beta_train with the matrices and scales resident.
 - recommend_ms / eval_ms: device events around the device parts of recommend and eval_ranking, alternated, after a
   warm-up; eval_api_ms: host clock around the public call with SciPy matrices in.
 - kernels_ms_*: torch.profiler device time per kernel of one training and of one recommend, in a separate pass after
   the timed ones.
 - work: sum_u deg_u^2 (read-modify-writes of the walk), the barrier steps the walk runs (per block the longest row's
   sum over its users of ceil(deg_u / 256), summed over the blocks) for rows grouped by that length, as training runs
   them, and in id order for comparison, and sum over the test users of sum_j |W_j| (read-modify-writes of scoring).
   walk_ns_per_step: the profiled walk kernel time over the steps run.
 - cpu_arm: SciPy float64 Piu[R] @ Pui (Piu = P^T with values du[u], Pui = P) of a fixed seeded sample of item rows R,
   then the two products and per-row NumPy top-k, timed on this host and EXTRAPOLATED to all items by n / |R|.
 - oracle_equal: sampled rows of W against the ordered restatement of the definition (acc[P.indices[row u]] += du[u]
   over the users of a, ascending), and sampled users' lists against the NumPy scores.
 - quality: Recall@10, NDCG@10, Recall@100 of RP3beta and of ItemKNN (k 100, cosine) on the same split, same run.

    python scripts/rp3beta_bench.py [--reps 5] [--train-reps 3] [--sample-items 400] [--sample-users 40] [--out FILE]
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

from knn_bench import oracle_list, profiled, timed
from recommend_bench import gpu_info
from recmodel_b200 import ItemKNN, RP3beta, engine, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.knn_model import _canonical
from recmodel_b200.rp3beta_model import _scale
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, K, TOPN = 138_493, 26_744, 20_000_000, 100, 100
ALPHA, BETA = 1.0, 0.5
KS = [10, 20, 50, 100]
TILE_BYTES, STEP = 64 << 20, 256   # knn_batch's tile budget; threads per walk row (KN_THREADS)


def ordered_row(P, PT, du, ra, cb, a, k):
    """(ids, weights) of row a by the definition: the walk sum in ascending u, the two products, lexsort top-k."""
    acc = np.zeros(P.shape[1], np.float64)
    for u in PT.indices[PT.indptr[a]:PT.indptr[a + 1]]:
        acc[P.indices[P.indptr[u]:P.indptr[u + 1]]] += du[u]
    b = np.flatnonzero(acc > 0)
    b = b[b != a]
    w = (ra[a] * acc[b]) * cb[b]
    top = np.lexsort((b, -w))[:k]
    top = top[np.argsort(b[top])]
    return b[top], w[top]


def cpu_rows(Piu, Pui, ra, cb, rows, k):
    """The CPU arm: SciPy float64 Piu[R] @ Pui, then the products and top-k per row."""
    S = (Piu[rows] @ Pui).tocsr()
    S.sort_indices()
    out = []
    for r, a in enumerate(rows):
        b = S.indices[S.indptr[r]:S.indptr[r + 1]].astype(np.int64)
        s = S.data[S.indptr[r]:S.indptr[r + 1]]
        keep = (b != a) & (s > 0)
        b, s = b[keep], s[keep]
        w = (ra[a] * s) * cb[b]
        top = np.lexsort((b, -w))[:k]
        top = top[np.argsort(b[top])]
        out.append((b[top], w[top]))
    return out


def walk_steps(P, PT, n):
    """(steps run with rows grouped by walk length, steps in id order, per-item walk lengths)."""
    deg = np.diff(P.indptr).astype(np.int64)
    per_entry = (deg[PT.indices] + STEP - 1) // STEP
    chain = np.add.reduceat(np.r_[per_entry, 0], PT.indptr[:-1])[:n] * (np.diff(PT.indptr) > 0)
    B = max(1, min(n, TILE_BYTES // (n * 8)))
    grouped = chain[np.lexsort((np.arange(n), -chain))]
    return (int(sum(grouped[a0:a0 + B].max() for a0 in range(0, n, B))),
            int(sum(chain[a0:a0 + B].max() for a0 in range(0, n, B))), chain)


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
    m = RP3beta(num_items=ITEMS, num_users=USERS, device=dev)
    m.train(Train, alpha=ALPHA, beta=BETA, k=K)   # warm-up
    torch.cuda.synchronize(dev)
    train_s = []
    for _ in range(args.train_reps):
        t0 = time.perf_counter()
        m.train(Train, alpha=ALPHA, beta=BETA, k=K)
        torch.cuda.synchronize(dev)
        train_s.append(time.perf_counter() - t0)
    X = m._X
    XT = X.transpose()
    W_d = m._W_device()
    Xc = _canonical(Train)
    Xc.data = np.ones_like(Xc.data, dtype=np.float32)
    deg = np.diff(Xc.indptr)
    pop = np.bincount(Xc.indices, minlength=ITEMS)
    du, ra, cb = _scale(deg, ALPHA), _scale(pop, ALPHA), _scale(pop, BETA)
    du_d, ra_d, cb_d = (torch.from_numpy(v).to(dev) for v in (du, ra, cb))

    def train_dev():
        return engine.rp3beta_train(X, XT, du_d, ra_d, cb_d, K)

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
    train_dev_ms = timed(train_dev, args.train_reps, dev)
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
    W2 = train_dev()
    same_train = all(bool(torch.equal(a, b)) for a, b in zip(W2, W_d))

    kernels_train = profiled(train_dev, dev)
    kernels_rec = profiled(rec, dev)

    item = ItemKNN(num_items=ITEMS, num_users=USERS, device=dev)
    item.train(Train, k=K)
    res_item = item.eval_ranking(Test, topn=KS, exclude=Train)
    del item

    # the work counts, the CPU arm and the oracle, on fixed seeded samples
    PT = Xc.T.tocsr()
    PT.sort_indices()
    steps_grouped, steps_id_order, chain = walk_steps(Xc, PT, ITEMS)
    walk_ms = next((v for key, v in kernels_train.items() if "userknn_score_tile_kernel" in key), None)
    Piu = scipy.sparse.csr_matrix((du[PT.indices], PT.indices, PT.indptr), shape=PT.shape)
    Pui = Xc.astype(np.float64)
    rng = np.random.default_rng(2024)
    rows = np.sort(rng.choice(ITEMS, size=args.sample_items, replace=False))
    t0 = time.perf_counter()
    cpu = cpu_rows(Piu, Pui, ra, cb, rows, K)
    cpu_s = time.perf_counter() - t0
    Wh = m.W

    def same_row(a, ids, vals):
        lo, hi = Wh.indptr[a], Wh.indptr[a + 1]
        return np.array_equal(Wh.indices[lo:hi], ids) and np.array_equal(Wh.data[lo:hi].view(np.uint64),
                                                                          vals.view(np.uint64))
    w_ok = all(same_row(a, *ordered_row(Xc, PT, du, ra, cb, a, K)) for a in rows)
    cpu_ok = all(same_row(a, ids, vals) for a, (ids, vals) in zip(rows, cpu))
    sample_u = np.sort(rng.choice(users, size=min(args.sample_users, len(users)), replace=False))
    ids_h = ids0.cpu().numpy()
    pos = np.searchsorted(users, sample_u)
    lists_ok = all(np.array_equal(ids_h[p], oracle_list(Xc, Wh, int(u), TOPN)) for p, u in zip(pos, sample_u))

    w_len = np.diff(Wh.indptr).astype(np.int64)
    votes = int(sum(int(w_len[Xc.indices[Xc.indptr[u]:Xc.indptr[u + 1]]].sum()) for u in users))
    deg64 = deg.astype(np.int64)
    pick = ["Recall@10", "NDCG@10", "Recall@100"]
    line = {
        "metric": "rp3beta_recommend_device_ms", "value": float(np.median(rec_ms)), "unit": "ms",
        "what": f"RP3beta (alpha {ALPHA}, beta {BETA}, k {K}) trained on the 80% split of make_counts_cached({USERS}, "
                f"{ITEMS}, {NNZ}); recommend top-{TOPN} over each user's unseen items, {len(users)} test users x "
                f"{ITEMS} items, train entries excluded; device events, median of {args.reps} after a warm-up",
        "train_s": [round(x, 3) for x in train_s], "train_median_s": float(np.median(train_s)),
        "train_device_ms": [round(x, 2) for x in train_dev_ms],
        "train_device_median_ms": float(np.median(train_dev_ms)),
        "train_bitwise_equal_across_runs": bool(same_train),
        "recommend_ms": [round(x, 3) for x in rec_ms],
        "eval_ranking_ks": KS, "eval_ms": [round(x, 3) for x in eval_ms], "eval_median_ms": float(np.median(eval_ms)),
        "eval_api_ms": [round(x, 1) for x in api_ms], "eval_api_median_ms": float(np.median(api_ms)),
        "bitwise_equal_across_reps": bool(same),
        "kernels_ms_one_train_profiled": kernels_train,
        "kernels_ms_one_recommend_profiled": kernels_rec,
        "work": {"walk_updates_sum_deg_u_sq": int((deg64 * deg64).sum()),
                 "walk_steps_run_rows_grouped": steps_grouped, "walk_steps_rows_in_id_order": steps_id_order,
                 "walk_longest_row_steps": int(chain.max()),
                 "walk_ns_per_step": None if walk_ms is None else round(walk_ms * 1e6 / steps_grouped, 2),
                 "score_updates_sum_u_sum_j_W_j": votes, "W_nnz": int(Wh.nnz),
                 "train_nnz": int(Xc.nnz), "test_nnz": int(Test.nnz), "max_pop": int(pop.max()),
                 "max_deg": int(deg.max())},
        "cpu_arm": {"what": "SciPy float64 Piu[R] @ Pui of a seeded sample of item rows R, then per-row NumPy products "
                            "and top-k (lexsort), single process on the GPU host; EXTRAPOLATED to all items by n / |R|",
                    "sample_items": int(len(rows)), "sample_s": round(cpu_s, 3),
                    "extrapolated_all_items_s": round(cpu_s / len(rows) * ITEMS, 1),
                    "equal_to_device_rows": bool(cpu_ok)},
        "oracle_equal_sampled_W_rows": bool(w_ok),
        "oracle_equal_sampled_users": bool(lists_ok), "sampled_users": int(len(sample_u)),
        "quality": {"RP3beta": {k: res[k] for k in pick}, "ItemKNN": {k: res_item[k] for k in pick}},
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
