"""Top-100 over each user's unseen items for all users at ML-20M shape (138 493 x 26 744, f = 128), with the
20 M-entry synthetic count matrix as the exclusion matrix. One JSON line: ms of the excluding ranking and of the
plain ranking (alternated in one process), the users whose candidate list made the exact kernels redo the call,
and utils.test_coverage(m, Train, 10) through WMF.recommend against the batched implementation it replaced
(rank_batch of topN + max(seen) items, np.isin on the host, per-user loop past 1024), both results compared.

    python scripts/recommend_bench.py [--reps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np
import torch

from oracle import wmf_oracle as orc
from recmodel_b200 import WMF, _lib, engine, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, DIM, TOPN = 138_493, 26_744, 20_000_000, 128, 100


def coverage_batched_rank(cls, Train, topN):
    """utils.test_coverage before WMF.recommend existed: rank topN + max(seen) items per batch of 4096 users, drop the
    seen ones on the host; a batch whose list would pass 1024 items falls back to one rank call per user."""
    Train = Train.tocsr()
    n_users, n_items = Train.shape
    item_counts = np.zeros(n_users, dtype=np.int32)
    seen_n = np.diff(Train.indptr)
    all_items = np.arange(n_items, dtype=np.int32)
    order = np.argsort(seen_n, kind="stable")
    for b0 in range(0, n_users, 4096):
        users = order[b0:b0 + 4096]
        k = int(topN + seen_n[users].max())
        if k > min(_lib.TOPK_MAX, n_items):
            for user in users:
                lo, hi = Train.indptr[user], Train.indptr[user + 1]
                ranked = np.asarray(cls.rank(users=int(user), items=np.delete(all_items, Train.indices[lo:hi]),
                                             topn=topN)).reshape(-1)
                item_counts[ranked[:topN]] += 1
            continue
        ranked = cls.rank_batch(all_items, users.astype(np.int64), k)
        for row, user in zip(ranked, users):
            lo, hi = Train.indptr[user], Train.indptr[user + 1]
            item_counts[row[~np.isin(row, Train.indices[lo:hi])][:topN]] += 1
    return item_counts


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({type(e).__name__})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    Train = make_counts_cached(USERS, ITEMS, NNZ)
    m = WMF(num_items=ITEMS, num_users=USERS, dim=DIM, gamma=0.1, weighted=True, device=dev)
    rng = np.random.default_rng(5)
    m.users = (rng.standard_normal((USERS, DIM)) * 0.3).astype(np.float32)   # bench.py --workload rank's factors
    m.items = orc.init_items(ITEMS, DIM, False)
    U, V = m.users_device, m.items_device
    users_d = torch.arange(USERS, dtype=torch.int64, device=dev)
    ex = DeviceCSR.from_scipy(Train, dev).sorted()

    def excl():
        return engine.score_topk_exclude(users_d, ex, U, V, TOPN)

    def plain():
        return engine.score_topk(users_d, None, U, V, TOPN)

    for _ in range(2):
        excl(), plain()
    times = {"recommend": [], "score_topk": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(args.reps):  # alternating, one device-event window per call
        for name, fn in (("recommend", excl), ("score_topk", plain)):
            ev[0].record()
            fn()
            ev[1].record()
            torch.cuda.synchronize(dev)
            times[name].append(ev[0].elapsed_time(ev[1]))
    ids, _, fixup = excl()
    fixup_users = int(fixup.item())
    # the public call with host arrays in and out, the exclusion matrix already sorted on the device
    t0 = time.perf_counter()
    rec = m.recommend(np.arange(USERS), TOPN, exclude=ex)
    t_api = (time.perf_counter() - t0) * 1e3
    assert np.array_equal(rec, ids.cpu().numpy())
    # a sample of rows against the exact CUDA-core kernels
    sample = torch.arange(0, USERS, 97, dtype=torch.int64, device=dev)
    tc_ids = engine.score_topk_exclude(sample, ex, U, V, TOPN)[0].cpu().numpy()
    os.environ["WMF_SCORE_EXACT"] = "1"
    exact_ids = engine.score_topk_exclude(sample, ex, U, V, TOPN)[0].cpu().numpy()
    del os.environ["WMF_SCORE_EXACT"]
    # test_coverage: new (recommend) and old (batched rank_batch + host filter), alternated new, old, new
    t0 = time.perf_counter(); cov_new = utils.test_coverage(m, Train, 10); t_new1 = time.perf_counter() - t0
    t0 = time.perf_counter(); cov_old = coverage_batched_rank(m, Train, 10); t_old = time.perf_counter() - t0
    t0 = time.perf_counter(); cov_new2 = utils.test_coverage(m, Train, 10); t_new2 = time.perf_counter() - t0
    seen_n = np.diff(Train.indptr)
    line = {
        "metric": "wmf_recommend_ms", "value": float(np.median(times["recommend"])), "unit": "ms",
        "what": f"top-{TOPN} over unseen items for all {USERS} users, {ITEMS} items, f {DIM}, exclusion matrix "
                f"{Train.nnz} entries (make_counts_cached), engine.score_topk_exclude, device events, median of {args.reps}",
        "recommend_ms": [round(x, 3) for x in times["recommend"]],
        "score_topk_ms": [round(x, 3) for x in times["score_topk"]],
        "score_topk_median_ms": float(np.median(times["score_topk"])),
        "fixup_users": fixup_users,
        "recommend_api_ms": round(t_api, 1),
        "tc_equals_exact_sample": bool(np.array_equal(tc_ids, exact_ids)), "sample_users": int(sample.numel()),
        "users_with_more_than_1014_seen": int((seen_n > _lib.TOPK_MAX - 10).sum()), "max_seen": int(seen_n.max()),
        "test_coverage_new_s": [round(t_new1, 3), round(t_new2, 3)], "test_coverage_old_s": round(t_old, 3),
        "test_coverage_equal": bool(np.array_equal(cov_new, cov_old) and np.array_equal(cov_new, cov_new2)),
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
