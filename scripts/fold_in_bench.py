"""recommend_for and eval_ranking_for of all six models under the strong-generalisation protocol at ML-20M shape:
utils.split_users(make_counts_cached(138 493, 26 744, 20 M), 10 000) holds 10 000 users out of training and splits
each one's history 80/20 into FoldIn (folded in) and Test (predicted). Every model is trained on Train with the settings
of its own bench (WMF: f 128, 10 epochs; Ease: alpha 100; ItemKNN, UserKNN: k 100, cosine; SLIM: l1 1, l2 10, k 128;
RP3beta: alpha 1, beta 0.5, k 100), then ranks the top-100 over each held-out user's unseen items (its FoldIn entries
excluded) and is evaluated at 10 / 20 / 50 / 100.

One JSON line, all numbers from the same run:
 - per model, fold_in_ms: device events around the fold-in of the 10 000 histories (host preparation and upload
   included: for the item models that is all of it; UserKNN adds the transpose of X and wmf_userknn_fold_in, WMF the
   confidence transform, the Gram and the user half-step); rank_ms: device events around the top-100 ranking with the
   folded-in representation resident. Median and spread ((max - min) / median) of --reps after a warm-up, the models
   alternated. api_ms: host clock around the public recommend_for call.
 - eval_ms: device events around the device part of eval_ranking_for with the representation resident; eval_api_ms:
   host clock around the public call (fold-in included).
 - kernels_ms: torch.profiler device time per kernel of one fold-in plus ranking per model, in a separate pass.
 - userknn_work: computed from the data: the counting atomics (sum over the FoldIn entries of the Train users of their
   item), the selection size (rows x training users), and the score read-modify-writes (sum over rows r and v in N'(r)
   of nnz_v).
 - quality: Recall@10, NDCG@10, Recall@100 of the six models on this split.
 - oracle: sampled UserKNN N' rows and lists and ItemKNN lists against the NumPy definitions; sampled WMF factor rows
   against an fp64 solve of their normal equations (row-relative error).

    python scripts/fold_in_bench.py [--reps 5] [--held-out 10000] [--sample 20] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np
import torch

from knn_bench import profiled, timed
from recommend_bench import gpu_info
from oracle import wmf_oracle as orc
from recmodel_b200 import RP3beta, SLIM, WMF, Ease, ItemKNN, UserKNN, ranking, utils
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.knn_model import _canonical
from recmodel_b200.synthetic import make_counts_cached

USERS, ITEMS, NNZ, TOPN = 138_493, 26_744, 20_000_000, 100
KS = [10, 20, 50, 100]


def log(msg):
    print(f"[{time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def spread(xs):
    return round((max(xs) - min(xs)) / float(np.median(xs)), 4)


def oracle_rows(Q, P, pop_u, k, rows):
    """UserKNN N' rows of the definitions (cosine, shrink 0) for the rows ``rows`` of the canonical Q: SciPy int64
    counts, float64 similarities, lexsort((v, -sim))."""
    Pq = Q[rows].astype(np.int64)
    Pq.data[:] = 1
    C = (Pq @ P.T).tocsr()
    C.sort_indices()
    out = []
    for r in range(len(rows)):
        v = C.indices[C.indptr[r]:C.indptr[r + 1]].astype(np.int64)
        c = C.data[C.indptr[r]:C.indptr[r + 1]].astype(np.float64)
        s = c / (np.sqrt(float(Pq.indptr[r + 1] - Pq.indptr[r])) * np.sqrt(pop_u[v]) + 0.0)
        top = np.lexsort((v, -s))[:k]
        top = top[np.argsort(v[top])]
        out.append((v[top], s[top]))
    return out


def oracle_list(acc, seen, topn):
    cand = np.delete(np.arange(len(acc)), seen)
    out = np.full(topn, -1, np.int64)
    best = cand[np.lexsort((cand, -acc[cand]))][:topn]
    out[:len(best)] = best
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--held-out", type=int, default=10_000)
    ap.add_argument("--sample", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gpu_info()
    full = make_counts_cached(USERS, ITEMS, NNZ)
    Train, FoldIn, Test, held = utils.split_users(full, args.held_out)
    n_train, nq = Train.shape[0], FoldIn.shape[0]
    log(f"data ready: {n_train} training users, {nq} held out, {FoldIn.nnz} fold-in and {Test.nnz} test entries")

    models = {}
    m = WMF(num_items=ITEMS, num_users=n_train, dim=128, gamma=0.1, weighted=True, device=dev)
    m.train(Train, 10, eval_mat=Train, count_mat=Train, cores=1, stopping_rounds=11)
    models["WMF"] = m
    m = Ease(num_items=ITEMS, num_users=n_train, device=dev)
    m.train(Train, alpha=100.0, verbose=0, cores=1)
    models["Ease"] = m
    for name, cls, kw in (("ItemKNN", ItemKNN, {"k": 100}), ("UserKNN", UserKNN, {"k": 100}),
                          ("SLIM", SLIM, {"l1": 1.0, "l2": 10.0, "k": 128, "max_iter": 100, "tol": 1e-4}),
                          ("RP3beta", RP3beta, {"alpha": 1.0, "beta": 0.5, "k": 100})):
        m = cls(num_items=ITEMS, num_users=n_train, device=dev)
        m.train(Train, **kw)
        models[name] = m
    torch.cuda.synchronize(dev)
    log("models trained")

    ex = DeviceCSR.from_scipy(FoldIn, dev)
    T = DeviceCSR.from_scipy(Test, dev).sorted()
    users_d = torch.arange(nq, dtype=torch.int64, device=dev)
    eval_users = torch.from_numpy(np.flatnonzero(np.diff(Test.indptr) > 0)).to(dev)
    ks = np.asarray(KS, np.int64)

    def fold(name):
        m = models[name]
        return m._fold_in_device(FoldIn) if name == "WMF" else m._fold_in(FoldIn)

    def rank_fn(name):
        m = models[name]
        if name == "WMF":
            return lambda rep, u, k, e: m._fold_in_rank_ids(rep, u, k, e)
        return lambda rep, u, k, e: m._recommend_ids(*rep, u, k, e)

    reps, ids0, sums0 = {}, {}, {}
    for name in models:   # warm-up of every shape
        reps[name] = fold(name)
        ids0[name] = rank_fn(name)(reps[name], users_d, TOPN, ex)
        sums0[name] = ranking.eval_ranking_sums(lambda u, k, e, n=name: rank_fn(n)(reps[n], u, k, e), ITEMS, T, ex,
                                                eval_users, ks)
        models[name].recommend_for(FoldIn, TOPN)
    torch.cuda.synchronize(dev)
    log("warm-up done")

    t = {name: {"fold_in_ms": [], "rank_ms": [], "api_ms": [], "eval_ms": [], "eval_api_ms": []} for name in models}
    same = {name: True for name in models}
    for _ in range(args.reps):   # the models alternated
        for name in models:
            out = []
            t[name]["fold_in_ms"] += timed(lambda: out.append(fold(name)), 1, dev)
            t[name]["rank_ms"] += timed(lambda: out.append(rank_fn(name)(out[0], users_d, TOPN, ex)), 1, dev)
            t[name]["eval_ms"] += timed(lambda: out.append(ranking.eval_ranking_sums(
                lambda u, k, e: rank_fn(name)(out[0], u, k, e), ITEMS, T, ex, eval_users, ks)), 1, dev)
            same[name] &= bool(torch.equal(out[1], ids0[name])) and bool(torch.equal(out[2], sums0[name]))
            t0 = time.perf_counter()
            lists = models[name].recommend_for(FoldIn, TOPN)
            t[name]["api_ms"].append((time.perf_counter() - t0) * 1e3)
            same[name] &= bool(np.array_equal(lists, ids0[name].cpu().numpy()))
    results = {}
    for _ in range(min(args.reps, 3)):
        for name in models:
            t0 = time.perf_counter()
            results[name] = models[name].eval_ranking_for(FoldIn, Test, topn=KS)
            t[name]["eval_api_ms"].append((time.perf_counter() - t0) * 1e3)
    log("timed passes done")

    kernels = {name: profiled(lambda: rank_fn(name)(fold(name), users_d, TOPN, ex), dev) for name in models}
    log("profiled")

    # UserKNN work, from the data
    Xc = _canonical(Train)
    Qc = _canonical(FoldIn)
    pop_i = np.diff(Xc.tocsc().indptr).astype(np.int64)
    nnz_u = np.diff(Xc.indptr).astype(np.int64)
    Nq = models["UserKNN"]._fold_in(FoldIn)[1]
    n_indptr, n_indices = Nq[0].cpu().numpy(), Nq[1].cpu().numpy()
    votes = int(nnz_u[n_indices].sum())
    atomics = int(pop_i[Qc.indices].sum())
    key = next((k for k in kernels["UserKNN"] if "knn_cooc_kernel" in k), None)
    cooc_ms = kernels["UserKNN"].get(key)

    # sampled oracle checks
    rng = np.random.default_rng(2024)
    rows = np.sort(rng.choice(nq, size=min(args.sample, nq), replace=False))
    P = Xc.astype(np.int64)
    P.data[:] = 1
    n_data = Nq[2].cpu().numpy()
    nb_ok = all(np.array_equal(n_indices[n_indptr[r]:n_indptr[r + 1]], v)
                and np.array_equal(n_data[n_indptr[r]:n_indptr[r + 1]].view(np.uint64), s.view(np.uint64))
                for r, (v, s) in zip(rows, oracle_rows(Qc, P, nnz_u.astype(np.float64), 100, rows)))
    uk_ok, ik_ok = True, True
    W = models["ItemKNN"].neighbors
    for r in rows:
        seen = FoldIn.indices[FoldIn.indptr[r]:FoldIn.indptr[r + 1]]
        acc = np.zeros(ITEMS)
        for e in range(n_indptr[r], n_indptr[r + 1]):
            v = n_indices[e]
            acc[Xc.indices[Xc.indptr[v]:Xc.indptr[v + 1]]] += n_data[e] * Xc.data[Xc.indptr[v]:Xc.indptr[v + 1]].astype(
                np.float64)
        uk_ok &= bool(np.array_equal(ids0["UserKNN"][r].cpu().numpy(), oracle_list(acc, seen, TOPN)))
        acc = np.zeros(ITEMS)
        for e in range(Qc.indptr[r], Qc.indptr[r + 1]):
            j = Qc.indices[e]
            acc[W.indices[W.indptr[j]:W.indptr[j + 1]]] += np.float64(np.float32(Qc.data[e])) * W.data[W.indptr[j]:
                                                                                                    W.indptr[j + 1]]
        ik_ok &= bool(np.array_equal(ids0["ItemKNN"][r].cpu().numpy(), oracle_list(acc, seen, TOPN)))
    w = models["WMF"]
    wrows = np.sort(rng.choice(nq, size=200, replace=False))
    Cp = FoldIn[wrows].astype(np.float32)
    Cp.data = orc.preprocess_counts(Cp.data, "log", np.float32(10), np.float32(1)).astype(np.float32)
    ref = orc.half_step(w.items.astype(np.float64), Cp, 0.1, dtype=np.float64)
    got = reps["WMF"][torch.from_numpy(wrows).to(dev)].cpu().numpy().astype(np.float64)
    wmf_err = float(np.max(np.linalg.norm(got - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-30)))
    log("oracle checks done")

    pick = ("Recall@10", "NDCG@10", "Recall@100")
    per_model = {}
    for name in models:
        d = t[name]
        per_model[name] = {
            "fold_in_ms": [round(x, 3) for x in d["fold_in_ms"]], "fold_in_median_ms": float(np.median(d["fold_in_ms"])),
            "fold_in_spread": spread(d["fold_in_ms"]),
            "rank_ms": [round(x, 3) for x in d["rank_ms"]], "rank_median_ms": float(np.median(d["rank_ms"])),
            "rank_spread": spread(d["rank_ms"]),
            "api_ms": [round(x, 1) for x in d["api_ms"]], "api_median_ms": float(np.median(d["api_ms"])),
            "eval_ms": [round(x, 3) for x in d["eval_ms"]], "eval_median_ms": float(np.median(d["eval_ms"])),
            "eval_api_ms": [round(x, 1) for x in d["eval_api_ms"]],
            "eval_api_median_ms": float(np.median(d["eval_api_ms"])),
            "bitwise_equal_across_reps": bool(same[name]),
            "kernels_ms_one_fold_in_and_rank_profiled": kernels[name],
            "quality": {k: results[name][k] for k in pick}, "result": results[name],
        }
    uk = per_model["UserKNN"]
    line = {
        "metric": "userknn_recommend_for_device_ms", "value": uk["fold_in_median_ms"] + uk["rank_median_ms"],
        "unit": "ms",
        "what": f"recommend_for top-{TOPN} of {nq} held-out users (split_users(make_counts_cached({USERS}, {ITEMS}, "
                f"{NNZ}), {args.held_out}), 80% of each history folded in and excluded), six models trained on the "
                f"{n_train} other users; value: UserKNN fold-in + ranking, device events, medians of {args.reps} after "
                f"a warm-up (measured)",
        "models": per_model,
        "userknn_work": {"what": "computed from the data and the folded-in neighbours",
                         "counting_atomics_sum_over_fold_in_entries_of_item_pop": atomics,
                         "selection_doubles_rows_x_training_users": int(nq) * int(n_train),
                         "score_updates_sum_r_sum_v_nnz_v": votes, "fold_in_neighbors_nnz": int(n_indptr[-1]),
                         "fold_in_nnz": int(Qc.nnz)},
        "userknn_cooc_rate_atomics_per_s": (atomics / (cooc_ms / 1e3)) if cooc_ms else None,
        "oracle": {"userknn_neighbor_rows_equal": bool(nb_ok), "userknn_lists_equal": bool(uk_ok),
                   "itemknn_lists_equal": bool(ik_ok), "sampled_rows": int(len(rows)),
                   "wmf_max_row_rel_err_vs_fp64_200_rows": wmf_err},
        "data": {"train_users": int(n_train), "held_out": int(nq), "fold_in_nnz": int(FoldIn.nnz),
                 "test_nnz": int(Test.nnz), "train_nnz": int(Train.nnz)},
        "provenance": {"measured": "models.*: *_ms, kernels_ms_*, quality, result, bitwise_equal_*; oracle.*, "
                                   "userknn_cooc_rate_atomics_per_s, on the card named here",
                       "computed": "userknn_work: counted from the data, not timed"},
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
