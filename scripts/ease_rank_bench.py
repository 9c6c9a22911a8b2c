"""Ease.recommend and Ease.eval_ranking at ML-20M shape: the 20 M-entry synthetic count matrix
(make_counts_cached(138 493, 26 744, 20 M), the data of scripts/eval_ranking_bench.py) split 80/20 with
utils.train_test_split_sparse_mat, Ease trained on the train half (W: 26 744^2 floats, 2.86 GB), then top-100 over each
test user's unseen items (train entries excluded) and Recall / Precision / NDCG / MAP / hit rate at 10 / 20 / 50 / 100.

One JSON line, all numbers from the same run:
 - train_s: host clock around Ease.train (ends in a device synchronise).
 - recommend_ms: device events around the device part of recommend (top-100 of every test user, both matrices
   resident), median of the reps after a warm-up of every shape.
 - eval_ms: device events around the device part of eval_ranking (chunked lists, per-user metrics, one reduce);
   eval_api_ms: host clock around the public call with SciPy matrices in.
 - kernels_ms: torch.profiler device time per kernel of one recommend call, in a separate pass after the timed ones.
 - host_loop: what recommend replaces, the per-user Ease.rank(np.delete(all_items, seen), u, 100) loop of
   utils.test_coverage, timed on a fixed seeded sample of users and EXTRAPOLATED to all test users.
 - work: multiply-adds sum_u nnz_u * n (each reads one float of W), and the bytes of W a user batch touches (the rows
   of W its users' entries name, whole rows, n floats each), computed from the shapes and the data; achieved rates
   over recommend_ms and over the scoring kernel's profiled time.
 - oracle_equal: the sampled users' recommend lists against a NumPy oracle (FP32 products summed in double in stored
   order, ordered by (-score, item id)).

    python scripts/ease_rank_bench.py [--reps 5] [--sample 200] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np
import torch

from recommend_bench import gpu_info
from recmodel_b200 import ranking, utils
from recmodel_b200.ease_model import Ease
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, ALPHA, TOPN = 138_493, 26_744, 20_000_000, 100.0, 100
KS = [10, 20, 50, 100]
TILE_BYTES = 64 << 20   # the score tile budget of wmf_ease_score_topk (csrc/ease.cu: ease_user_batch)


def oracle_list(X, W, u, topn):
    acc = np.zeros(W.shape[1], np.float64)
    for e in range(X.indptr[u], X.indptr[u + 1]):
        acc += (X.data[e] * W[X.indices[e]]).astype(np.float32).astype(np.float64)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sample", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    full = make_counts_cached(USERS, ITEMS, NNZ)
    Train, Test = utils.train_test_split_sparse_mat(full)
    m = Ease(num_items=ITEMS, num_users=USERS, device=dev)
    t0 = time.perf_counter()
    m.train(Train, alpha=ALPHA, verbose=0, cores=1)
    torch.cuda.synchronize(dev)
    train_s = time.perf_counter() - t0

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

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rec()
        torch.cuda.synchronize(dev)
    kernels = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            kernels[e.key[:80]] = round(t / 1e3, 3)

    # the host path recommend replaces, on a fixed seeded sample of test users
    rng = np.random.default_rng(2024)
    sample = np.sort(rng.choice(users, size=min(args.sample, len(users)), replace=False))
    all_items = np.arange(ITEMS)
    t0 = time.perf_counter()
    loop_lists = []
    for u in sample:
        seen = Train.indices[Train.indptr[u]:Train.indptr[u + 1]]
        loop_lists.append(m.rank(np.delete(all_items, seen), int(u), TOPN))
    loop_s = time.perf_counter() - t0
    ids_h = ids0.cpu().numpy()
    pos = np.searchsorted(users, sample)
    Wh = m.W
    oracle_ok = all(np.array_equal(ids_h[p], oracle_list(Train, Wh, int(u), TOPN)) for p, u in zip(pos, sample))
    loop_sets = all(set(ids_h[p].tolist()) == set(np.asarray(l).tolist()) for p, l in zip(pos, loop_lists))

    # work, from the shapes and the data
    nnz_u = np.diff(Train.indptr)[users].astype(np.int64)
    macs = int(nnz_u.sum()) * ITEMS
    ub = max(4, TILE_BYTES // (ITEMS * 8) // 4 * 4)
    batches = -(-len(users) // ub)
    rows_touched = []
    for b in range(batches):
        us = users[b * ub:(b + 1) * ub]
        idx = np.concatenate([Train.indices[Train.indptr[u]:Train.indptr[u + 1]] for u in us])
        rows_touched.append(len(np.unique(idx)))
    w_batch_bytes = np.asarray(rows_touched, np.int64) * ITEMS * 4
    rec_med = float(np.median(rec_ms))
    score_ms = sum(v for k, v in kernels.items() if "ease_score_tile_kernel" in k)
    line = {
        "metric": "ease_recommend_device_ms", "value": rec_med, "unit": "ms",
        "what": f"Ease.recommend top-{TOPN} over each user's unseen items, {len(users)} test users x {ITEMS} items, "
                f"train entries excluded, Ease (alpha {ALPHA}) trained on the 80% split of make_counts_cached({USERS}, "
                f"{ITEMS}, {NNZ}); device events, median of {args.reps} after a warm-up, W (2.86 GB) larger than L2",
        "recommend_ms": [round(x, 3) for x in rec_ms],
        "eval_ranking_ks": KS, "eval_ms": [round(x, 3) for x in eval_ms], "eval_median_ms": float(np.median(eval_ms)),
        "eval_api_ms": [round(x, 1) for x in api_ms], "eval_api_median_ms": float(np.median(api_ms)),
        "bitwise_equal_across_reps": bool(same),
        "kernels_ms_one_recommend_profiled": kernels,
        "host_loop": {"what": "per-user Ease.rank(np.delete(all_items, seen), u, 100), the loop test_coverage ran",
                      "sample_users": int(len(sample)), "sample_s": round(loop_s, 3),
                      "extrapolated_all_test_users_s": round(loop_s / len(sample) * len(users), 1),
                      "same_sets_as_recommend": bool(loop_sets)},
        "oracle_equal_sampled_users": bool(oracle_ok),
        "work": {"multiply_adds": macs, "w_reads_fp32_bytes": macs * 4, "user_batch": int(ub), "batches": int(batches),
                 "w_rows_touched_per_batch_median": int(np.median(rows_touched)),
                 "w_bytes_touched_per_batch_median": int(np.median(w_batch_bytes)),
                 "w_bytes_touched_all_batches": int(w_batch_bytes.sum()),
                 "w_bytes_full": ITEMS * ITEMS * 4,
                 "gmacs_per_s_recommend": round(macs / rec_med / 1e6, 1),
                 "gmacs_per_s_scoring_kernel": round(macs / score_ms / 1e6, 1) if score_ms else None,
                 "w_touched_gb_per_s_scoring_kernel": round(w_batch_bytes.sum() / score_ms / 1e6, 1) if score_ms else None,
                 "w_reads_gb_per_s_scoring_kernel": round(macs * 4 / score_ms / 1e6, 1) if score_ms else None},
        "train_s": round(train_s, 2), "train_nnz": int(Train.nnz), "test_nnz": int(Test.nnz),
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
