"""WMF.eval_ranking at ML-20M shape: the 20 M-entry synthetic count matrix (make_counts_cached(138 493, 26 744, 20 M))
split 80/20 with utils.train_test_split_sparse_mat, WMF f = 128 trained 10 epochs on the train half, then Recall,
Precision, NDCG, MAP and hit rate at 10 / 20 / 50 / 100 over each test user's unseen items (train entries excluded).

One JSON line, all numbers from the same run, the paths alternated rep by rep:
 - device_ms: device events around the ranking + metric work of eval_ranking (both matrices already resident and
   sorted, the test users already on the device): chunked recommend lists, per-user metrics, one reduce.
 - metrics_ms: device events around the metric kernels alone (wmf_topn_metrics + wmf_topn_metrics_reduce) on the lists
   of all test users.
 - api_ms: host clock around the public call with SciPy matrices in (uploads, device sort of both matrices, result).
 - host_path_ms: what the call replaces: WMF.recommend for the test users (lists copied to the host) and the metrics in
   vectorised NumPy; its values are compared with eval_ranking's (max relative difference).

    python scripts/eval_ranking_bench.py [--reps 5] [--out FILE]
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
from recmodel_b200 import WMF, engine, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, DIM, EPOCHS = 138_493, 26_744, 20_000_000, 128, 10
KS = [10, 20, 50, 100]


def numpy_metrics(ids, users, test, ks):
    """The metrics of WMF.eval_ranking from host lists, vectorised over users (what a user writes without it)."""
    t = test.tocsr().copy()
    t.eliminate_zeros()
    t.sum_duplicates()
    n_items = t.shape[1]
    tsize = np.diff(t.indptr)[users].astype(np.float64)
    keep = tsize > 0
    test_keys = np.repeat(np.arange(t.shape[0], dtype=np.int64), np.diff(t.indptr)) * n_items + t.indices
    K = ids.shape[1]
    hit = (ids >= 0) & np.isin(users[:, None].astype(np.int64) * n_items + ids, test_keys)
    h = np.cumsum(hit, axis=1)
    pos = np.arange(1, K + 1, dtype=np.float64)
    disc = 1.0 / np.log2(pos + 1.0)
    cdisc = np.cumsum(disc)
    dcg = np.cumsum(hit * disc, axis=1)
    ap = np.cumsum(hit * (h / pos), axis=1)
    out = {}
    for k in ks:
        m = np.minimum(k, tsize[keep]).astype(np.int64)
        hk = h[keep, k - 1].astype(np.float64)
        out[f"Recall@{k}"] = float(np.mean(hk / tsize[keep]))
        out[f"Precision@{k}"] = float(np.mean(hk / k))
        out[f"NDCG@{k}"] = float(np.mean(dcg[keep, k - 1] / cdisc[m - 1]))
        out[f"MAP@{k}"] = float(np.mean(ap[keep, k - 1] / m))
        out[f"HitRate@{k}"] = float(np.mean(hk > 0))
    out["users"] = int(keep.sum())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    full = make_counts_cached(USERS, ITEMS, NNZ)
    Train, Test = utils.train_test_split_sparse_mat(full)
    m = WMF(num_items=ITEMS, num_users=USERS, dim=DIM, gamma=0.1, weighted=True, device=dev)
    t0 = time.perf_counter()
    m.train(Train, EPOCHS, eval_mat=Test, count_mat=Train, cores=1, stopping_rounds=EPOCHS + 1)
    train_s = time.perf_counter() - t0
    K = max(KS)
    T = DeviceCSR.from_scipy(Test, dev).sorted()
    ex = DeviceCSR.from_scipy(Train, dev).sorted()
    users = np.flatnonzero(np.diff(Test.indptr) > 0)
    users_d = torch.from_numpy(users).to(dev)
    ids_d = m._recommend_ids(users_d, K, ex)

    def device_path():
        return m._eval_ranking_sums(T, ex, users_d, KS)

    def metrics_only():
        return engine.topn_metrics_reduce(engine.topn_metrics(ids_d, users_d, T, KS), len(KS))

    def api():
        return m.eval_ranking(Test, topn=KS, exclude=Train)

    def host_path():
        return numpy_metrics(m.recommend(users, K, exclude=Train), users, Test, KS)

    for _ in range(2):  # warm-up of every shape the timed window uses
        device_path(), metrics_only()
    api()
    host_path()
    times = {"device": [], "metrics": [], "api": [], "host": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    sums = []
    for _ in range(args.reps):
        for name, fn in (("device", device_path), ("metrics", metrics_only)):
            ev[0].record()
            r = fn()
            ev[1].record()
            torch.cuda.synchronize(dev)
            times[name].append(ev[0].elapsed_time(ev[1]))
            sums.append((name, r.cpu().numpy()))
        t0 = time.perf_counter()
        res = api()
        times["api"].append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        host = host_path()
        times["host"].append((time.perf_counter() - t0) * 1e3)
    same_bits = all(np.array_equal(s, sums[0][1]) for _, s in sums)
    rel = max(abs(res[k] - host[k]) / max(abs(host[k]), 1e-300) for k in host)
    line = {
        "metric": "wmf_eval_ranking_device_ms", "value": float(np.median(times["device"])), "unit": "ms",
        "what": f"eval_ranking Recall/Precision/NDCG/MAP/HitRate @ {KS}, {len(users)} test users, {ITEMS} items, f {DIM} "
                f"trained {EPOCHS} epochs on the 80% split of make_counts_cached({USERS}, {ITEMS}, {NNZ}), train entries "
                f"excluded; device events around ranking + metrics with both matrices resident (inputs larger than L2), "
                f"median of {args.reps}, paths alternated",
        "device_ms": [round(x, 3) for x in times["device"]],
        "metrics_ms": [round(x, 4) for x in times["metrics"]],
        "metrics_median_ms": float(np.median(times["metrics"])),
        "api_ms": [round(x, 1) for x in times["api"]], "api_median_ms": float(np.median(times["api"])),
        "host_path_ms": [round(x, 1) for x in times["host"]], "host_path_median_ms": float(np.median(times["host"])),
        "host_path_max_rel_diff": rel, "host_path_agrees_1e-12": bool(rel <= 1e-12),
        "sums_bitwise_equal_across_reps": bool(same_bits),
        "train_s": round(train_s, 2), "test_nnz": int(Test.nnz), "train_nnz": int(Train.nnz),
        "result": res,
        **gpu_info(),
    }
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
