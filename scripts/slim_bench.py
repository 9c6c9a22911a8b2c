"""SLIM training, recommend and eval_ranking at ML-20M shape: the data of scripts/knn_bench.py
(make_counts_cached(138 493, 26 744, 20 M) split 80/20 with utils.train_test_split_sparse_mat), SLIM trained on the
train half with its defaults (l1 1, l2 10, k 128, max_iter 100, tol 1e-4), then top-100 over each test user's unseen
items (train entries excluded) and Recall / Precision / NDCG / MAP / hit rate at 10 / 20 / 50 / 100.

One JSON line, all numbers from the same run:
 - train_s: host clock around SLIM.train (canonical copy, upload, transpose, candidates, G, descent, W assembly; ends
   in a device synchronise), median of --train-reps after one warm-up. train_device_ms: device events around
   engine.slim_train; candidates_device_ms: the same around its engine.knn_train part alone.
 - split_ms_profiled: torch.profiler device time of one engine.slim_train, split into the dense G (its memset and
   knn_cooc_kernel, less the knn_cooc_kernel of the candidates), the candidates (the kernels of one profiled
   engine.knn_train), the coordinate descent (slim_cd_kernel) and the assembly (the rest: scan, compaction, the
   transpose sort), in a separate pass after the timed ones.
 - sweeps: the distribution of the sweeps per column, and how many columns stopped at max_iter.
 - recommend_ms / eval_ms / eval_api_ms: as in scripts/knn_bench.py.
 - quality: eval_ranking of ItemKNN (k 100, cosine) and Ease (alpha 100) on the same split, in the same run.
 - cpu_arm: scikit-learn ElasticNet(positive=True) on P[:, S_j] (the same restricted problem) for a seeded sample of
   columns, timed on this host and EXTRAPOLATED to all items by n / |sample|; the largest relative difference of its
   solutions to the device's is reported beside it.
 - oracle_equal: sampled columns of W and their sweeps against the NumPy coordinate descent, and sampled users'
   lists against the NumPy scores.

    python scripts/slim_bench.py [--reps 5] [--train-reps 3] [--sample-cols 20] [--cpu-cols 50] [--sample-users 40]
                                 [--out FILE]
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
from recmodel_b200 import Ease, ItemKNN, engine, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.slim_model import SLIM
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, TOPN = 138_493, 26_744, 20_000_000, 100
L1, L2, K, MAX_ITER, TOL = 1.0, 10.0, 128, 100, 1e-4
KS = [10, 20, 50, 100]


def oracle_cd(Gs, b, l1, l2, max_iter, tol):
    """The defined coordinate descent (DESIGN.md 4.7) with scalar float64 steps: (w, sweeps)."""
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


def kernel_ms(kernels, name):
    return sum(v for k, v in kernels.items() if name in k)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--train-reps", type=int, default=3)
    ap.add_argument("--sample-cols", type=int, default=20)
    ap.add_argument("--cpu-cols", type=int, default=50)
    ap.add_argument("--sample-users", type=int, default=40)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    full = make_counts_cached(USERS, ITEMS, NNZ)
    Train, Test = utils.train_test_split_sparse_mat(full)
    m = SLIM(num_items=ITEMS, num_users=USERS, device=dev)
    kw = dict(l1=L1, l2=L2, k=K, max_iter=MAX_ITER, tol=TOL)
    m.train(Train, **kw)   # warm-up
    torch.cuda.synchronize(dev)
    train_s = []
    for _ in range(args.train_reps):
        t0 = time.perf_counter()
        m.train(Train, **kw)
        torch.cuda.synchronize(dev)
        train_s.append(time.perf_counter() - t0)
    X = m._X
    XT = X.transpose()
    W_d = m._W_device()
    sweeps = m.sweeps

    def slim():
        return engine.slim_train(X, XT, K, L1, L2, MAX_ITER, TOL)

    train_dev_ms = timed(slim, args.train_reps, dev)
    cand_dev_ms = timed(lambda: engine.knn_train(X, XT, K, "cosine", 0.0), args.train_reps, dev)
    W2, sweeps2 = slim()
    same_train = all(bool(torch.equal(a, b)) for a, b in zip(W2, W_d)) and np.array_equal(engine.d2h(sweeps2), sweeps)

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

    kernels_train = profiled(slim, dev)
    kernels_cand = profiled(lambda: engine.knn_train(X, XT, K, "cosine", 0.0), dev)
    kernels_rec = profiled(rec, dev)
    total = sum(kernels_train.values())
    cand_ms = sum(kernels_cand.values())
    cd_ms = kernel_ms(kernels_train, "slim_cd_kernel")
    gram_ms = (kernel_ms(kernels_train, "knn_cooc_kernel") - kernel_ms(kernels_cand, "knn_cooc_kernel")
               + kernel_ms(kernels_train, "emset") - kernel_ms(kernels_cand, "emset"))
    split = {"gram": round(gram_ms, 3), "candidates": round(cand_ms, 3), "coordinate_descent": round(cd_ms, 3),
             "assembly": round(total - gram_ms - cand_ms - cd_ms, 3), "total": round(total, 3)}

    knn = ItemKNN(num_items=ITEMS, num_users=USERS, device=dev)
    knn.train(Train, k=100)
    ease = Ease(num_items=ITEMS, num_users=USERS, device=dev)
    ease.train(Train, 100.0, 0, 1)
    quality = {"SLIM": res, "ItemKNN_k100_cosine": knn.eval_ranking(Test, topn=KS, exclude=Train),
               "Ease_alpha100": ease.eval_ranking(Test, topn=KS, exclude=Train)}
    del ease, knn

    # the CPU arm and the oracle, on fixed seeded samples
    Xc = m._X.to_scipy()
    P = scipy.sparse.csc_matrix(Xc.astype(np.int64))
    P.data[:] = 1
    Wh = m.W.tocsc()
    cand = engine.knn_train(X, XT, K, "cosine", 0.0)
    c_ptr, c_idx = engine.d2h(cand[0]), engine.d2h(cand[1])
    rng = np.random.default_rng(2024)
    cols = np.sort(rng.choice(ITEMS, size=args.sample_cols, replace=False))
    w_ok = True
    for j in cols:
        S = c_idx[c_ptr[j]:c_ptr[j + 1]].astype(np.int64)
        PS = P[:, S]
        Gs = (PS.T @ PS).toarray()
        b = (PS.T @ P[:, [j]]).toarray().reshape(-1)
        w, sw = oracle_cd(Gs, b, L1, L2, MAX_ITER, TOL)
        lo, hi = Wh.indptr[j], Wh.indptr[j + 1]
        w_ok &= (np.array_equal(Wh.indices[lo:hi], S[w > 0]) and
                 np.array_equal(Wh.data[lo:hi].view(np.uint64), w[w > 0].view(np.uint64)) and int(sweeps[j]) == sw)
    from sklearn.linear_model import ElasticNet
    cpu_cols = np.sort(rng.choice(ITEMS, size=args.cpu_cols, replace=False))
    Pf = scipy.sparse.csc_matrix(P, dtype=np.float64)
    cpu_s, cpu_diff = 0.0, 0.0
    for j in cpu_cols:
        S = c_idx[c_ptr[j]:c_ptr[j + 1]].astype(np.int64)
        if len(S) == 0:
            continue
        A, y = Pf[:, S], Pf[:, j].toarray().reshape(-1)
        t0 = time.perf_counter()
        en = ElasticNet(alpha=(L1 + L2) / USERS, l1_ratio=L1 / (L1 + L2), positive=True, fit_intercept=False)
        en.fit(A, y)
        cpu_s += time.perf_counter() - t0
        dev_w = Wh[S, j].toarray().reshape(-1)
        nrm = np.linalg.norm(dev_w)
        if nrm > 0:
            cpu_diff = max(cpu_diff, float(np.linalg.norm(en.coef_ - dev_w) / nrm))
    sample_u = np.sort(rng.choice(users, size=min(args.sample_users, len(users)), replace=False))
    ids_h = ids0.cpu().numpy()
    pos = np.searchsorted(users, sample_u)
    Wr = m.W
    lists_ok = all(np.array_equal(ids_h[p], oracle_list(Xc, Wr, int(u), TOPN)) for p, u in zip(pos, sample_u))

    nnz_u = np.diff(Xc.indptr).astype(np.int64)
    lens = np.diff(c_ptr)
    w_len = np.diff(Wr.indptr).astype(np.int64)
    votes = int(sum(int(w_len[Xc.indices[Xc.indptr[u]:Xc.indptr[u + 1]]].sum()) for u in users))
    rec_med = float(np.median(rec_ms))
    line = {
        "metric": "slim_train_device_ms", "value": float(np.median(train_dev_ms)), "unit": "ms",
        "what": f"SLIM (l1 {L1}, l2 {L2}, k {K}, max_iter {MAX_ITER}, tol {TOL}) trained on the 80% split of "
                f"make_counts_cached({USERS}, {ITEMS}, {NNZ}); device events around engine.slim_train, median of "
                f"{args.train_reps} after a warm-up",
        "train_s": [round(x, 3) for x in train_s], "train_median_s": float(np.median(train_s)),
        "train_device_ms": [round(x, 2) for x in train_dev_ms],
        "candidates_device_ms": [round(x, 2) for x in cand_dev_ms],
        "train_bitwise_equal_across_runs": bool(same_train),
        "split_ms_profiled": split,
        "sweeps": {"min": int(sweeps.min()), "median": float(np.median(sweeps)), "mean": float(sweeps.mean()),
                   "p90": float(np.percentile(sweeps, 90)), "p99": float(np.percentile(sweeps, 99)),
                   "max": int(sweeps.max()), "columns_at_max_iter": int((sweeps >= MAX_ITER).sum()),
                   "total": int(sweeps.sum())},
        "candidates": {"mean": float(lens.mean()), "columns_with_fewer_than_k": int((lens < K).sum())},
        "recommend_topn": TOPN, "recommend_ms": [round(x, 3) for x in rec_ms], "recommend_median_ms": rec_med,
        "eval_ranking_ks": KS, "eval_ms": [round(x, 3) for x in eval_ms], "eval_median_ms": float(np.median(eval_ms)),
        "eval_api_ms": [round(x, 1) for x in api_ms], "eval_api_median_ms": float(np.median(api_ms)),
        "bitwise_equal_across_reps": bool(same),
        "kernels_ms_one_train_profiled": kernels_train,
        "kernels_ms_one_candidates_profiled": kernels_cand,
        "kernels_ms_one_recommend_profiled": kernels_rec,
        "work": {"gram_entries": ITEMS * ITEMS, "gram_bytes": ITEMS * ITEMS * 4,
                 "cooccurrence_updates_sum_nnz_u_sq": int((nnz_u * nnz_u).sum()),
                 "gathered_G_S_entries_sum_m_sq": int((lens * lens).sum()),
                 "score_updates_sum_u_sum_j_W_j": votes, "W_nnz": int(Wr.nnz),
                 "train_nnz": int(Xc.nnz), "test_nnz": int(Test.nnz)},
        "quality": quality,
        "cpu_arm": {"what": "scikit-learn ElasticNet(alpha=(l1+l2)/m, l1_ratio=l1/(l1+l2), positive=True, "
                            "fit_intercept=False, default tol) on P[:, S_j] for a seeded sample of columns, single "
                            "process on the GPU host; EXTRAPOLATED to all items by n / |sample|",
                    "sample_cols": int(len(cpu_cols)), "sample_s": round(cpu_s, 3),
                    "extrapolated_all_items_s": round(cpu_s / len(cpu_cols) * ITEMS, 1),
                    "max_rel_diff_to_device_W": cpu_diff},
        "oracle_equal_sampled_W_columns": bool(w_ok), "sampled_columns": int(len(cols)),
        "oracle_equal_sampled_users": bool(lists_ok), "sampled_users": int(len(sample_u)),
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
