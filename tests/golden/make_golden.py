"""Generate tests/golden/*.npz by EXECUTING the unmodified reference.

    WMF_REFERENCE_ROOT=<checkout of titoeb/RecModel> python tests/golden/make_golden.py

Runs the reference's RecModel/wmf_model.py through oracle/ref_shim.py on small seeded
synthetic inputs (recmodel_b200.synthetic) and stores inputs + reference outputs. The
committed .npz files are what the oracle and the CUDA path are checked against; the tests
need no copy of the reference.
"""
import io
import os
import sys
from contextlib import redirect_stdout

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))

from conftest import array_digest  # noqa: E402
from oracle.ref_shim import load_reference_wmf  # noqa: E402
from recmodel_b200.synthetic import make_counts, split_train_test  # noqa: E402


def csr_parts(prefix, m):
    return {f"{prefix}_indptr": m.indptr.astype(np.int64), f"{prefix}_indices": m.indices.astype(np.int32),
            f"{prefix}_data": m.data.astype(np.float32), f"{prefix}_shape": np.array(m.shape, dtype=np.int64)}


def quiet(fn, *a, **k):
    with redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def case_weighted(name, users, items, nnz, dim, bias, iterations, seed, mode="log", planted=6):
    WMF = load_reference_wmf()
    full = make_counts(users, items, nnz, seed=seed, planted_rank=planted)
    tr, te = split_train_test(full, train=0.8, seed=1993)
    out = {}
    out.update(csr_parts("train", tr))
    out.update(csr_parts("test", te))
    m = WMF(num_items=items, num_users=users, dim=dim, gamma=0.1, weighted=True, bias=bias, seed=1993)
    out["items0"] = m.items.copy()
    # one half-step each way straight through the reference's recompute_factors*
    C = tr.copy()
    C.data = 10 * np.log(1 + 1 * C.data) if mode == "log" else 10 * C.data
    CT = C.T.tocsr()
    if bias:
        u1 = m.recompute_factors_bias(m.items.copy(), C.copy(), 0.1, cores=1)
        i1 = m.recompute_factors_bias(u1.copy(), CT.copy(), 0.1, cores=1)
    else:
        u1 = m.recompute_factors(m.items, C, 0.1)
        i1 = m.recompute_factors(u1, CT, 0.1)
    out["users_half1"], out["items_half1"] = u1, i1
    # full train() with the reference's own loop
    it = quiet(m.train, tr.copy(), iterations=iterations, eval_mat=te, count_mat=tr.copy(), cores=1,
               stopping_rounds=99, pre_process_count=mode)
    out["train_iter"] = np.int64(it)
    out["users_final"], out["items_final"] = m.users.copy(), m.items.copy()
    out["mse_final"] = np.float64(m.eval_prec(te))
    out["rmse_final"] = np.float64(m.eval_prec(te, metric="rmse"))
    out["mae_final"] = np.float64(m.eval_prec(te, metric="mae"))
    # early stopping: returned epoch index with a tight patience
    m2 = WMF(num_items=items, num_users=users, dim=dim, gamma=0.1, weighted=True, bias=bias, seed=1993)
    it2 = quiet(m2.train, tr.copy(), iterations=12, eval_mat=te, count_mat=tr.copy(), cores=1,
                stopping_rounds=2, pre_process_count=mode)
    out["early_iter"] = np.int64(it2)
    out["early_mse"] = np.float64(m2.eval_prec(te))
    # predict / rank / eval_topn on the trained model m
    rng = np.random.default_rng(5)
    pu = rng.integers(0, users, size=257)
    pi = rng.integers(0, items, size=257)
    out["pred_users"], out["pred_items"] = pu, pi
    out["pred"] = m.predict(pu, pi)
    all_items = np.arange(items)
    rk_users = rng.integers(0, users, size=16)
    out["rank_users"] = rk_users
    out["rank_top10"] = np.stack([m.rank(all_items, int(u), 10) for u in rk_users])
    out["rank_scores"] = np.stack([m.predict(int(u), all_items) for u in rk_users])
    near = max(items - 3, 1)  # the argsort branch (topn >= len/2)
    out["rank_near_full"] = np.stack([m.rank(all_items, int(u), near) for u in rk_users[:4]])
    topn = np.array([4, 10, 20])
    rec = m.eval_topn(te.copy(), topn=topn, rand_sampled=100, cores=1, random_state=7)
    out["topn"] = topn
    out["recall"] = np.array([rec[f"Recall@{k}"] for k in topn], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "iter", it, "early", it2, "mse", out["mse_final"], "recall", out["recall"])


def case_unweighted(name, users, items, nnz, dim, iterations, seed):
    WMF = load_reference_wmf()
    full = make_counts(users, items, nnz, seed=seed, planted_rank=4)
    tr, te = split_train_test(full, train=0.8, seed=1993)
    out = {}
    out.update(csr_parts("train", tr))
    out.update(csr_parts("test", te))
    m = WMF(num_items=items, num_users=users, dim=dim, gamma=0.1, weighted=None, bias=False, seed=1993)
    out["items0"] = m.items.copy()
    it = quiet(m.train, tr.copy(), iterations=iterations, eval_mat=te, cores=1, stopping_rounds=99)
    out["train_iter"] = np.int64(it)
    out["users_final"], out["items_final"] = m.users.copy(), m.items.copy()
    out["mse_final"] = np.float64(m.eval_prec(te))
    m1 = WMF(num_items=items, num_users=users, dim=dim, gamma=0.1, weighted=None, bias=False, seed=1993)
    quiet(m1.train, tr.copy(), iterations=1, eval_mat=te, cores=1, stopping_rounds=99)
    out["users_ep1"], out["items_ep1"] = m1.users.copy(), m1.items.copy()
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "iter", it, "mse", out["mse_final"])


def case_half_steps(name, users, items, nnz, dim, seed):
    """A larger fixture for the tensor-core shapes: only the two half-steps of the reference (no train loop). The
    inputs are not stored (tests/conftest.py::load_golden_2000x1500 regenerates them and checks them against the
    digests), nor the item half-step beyond every fifth row, so that each file stays under 1 MB."""
    WMF = load_reference_wmf()
    full = make_counts(users, items, nnz, seed=seed, planted_rank=8)
    parts = csr_parts("train", full)
    m = WMF(num_items=items, num_users=users, dim=dim, gamma=0.1, weighted=True, bias=False, seed=1993)
    items0 = m.items.copy()
    C = full.copy()
    C.data = 10 * np.log(1 + 1 * C.data)
    u1 = m.recompute_factors(m.items, C, 0.1)
    i1 = m.recompute_factors(u1, C.T.tocsr(), 0.1)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), users_half1=u1,
                        train_sha256=np.str_(array_digest(parts["train_indptr"], parts["train_indices"], parts["train_data"])),
                        items0_sha256=np.str_(array_digest(items0)))
    rows = np.arange(0, items, 5, dtype=np.int64)
    np.savez_compressed(os.path.join(HERE, name + "_items.npz"), items_half1_rows=rows, items_half1=i1[rows])
    print(name, u1.shape, i1.shape)


def case_ease(name, users, items, nnz, alpha, seed):
    """EASE (SURVEY.md 8f N4): the reference's Ease.train / predict / rank executed through the shim (its Cython
    predictor compiled from the reference sources into /tmp by oracle/ref_shim.load_reference_ease)."""
    from oracle.ref_shim import load_reference_ease
    Ease = load_reference_ease()
    full = make_counts(users, items, nnz, seed=seed, planted_rank=5)
    tr, te = split_train_test(full, train=0.8, seed=1993)
    out = {}
    out.update(csr_parts("train", tr))
    out.update(csr_parts("test", te))
    m = Ease(num_items=items, num_users=users)
    quiet(m.train, tr.copy(), alpha=alpha, verbose=0, cores=1)
    out["alpha"] = np.float64(alpha)
    out["W"] = m.W.copy()
    rng = np.random.default_rng(6)
    pu = rng.integers(0, users, size=300).astype(np.int32)
    pi = rng.integers(0, items, size=300).astype(np.int32)
    out["pred_users"], out["pred_items"] = pu, pi
    out["pred"] = np.asarray(m.predict(pu, pi), dtype=np.float64)
    rk_users = rng.integers(0, users, size=12)
    out["rank_users"] = rk_users
    out["rank_top10"] = np.stack([m.rank(np.arange(items), int(u), 10) for u in rk_users])
    topn = np.array([4, 10, 20])
    rec = m.eval_topn(te.copy(), topn=topn, rand_sampled=100, cores=1, random_state=7)
    out["topn"] = topn
    out["recall"] = np.array([rec[f"Recall@{k}"] for k in topn], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(name, "W absmax", np.abs(out["W"]).max(), "recall", out["recall"])


if __name__ == "__main__":
    if "--ease-only" in sys.argv:
        case_ease("ease_f300", 400, 300, 12000, 50.0, seed=17)
        sys.exit(0)
    if "--large-only" in sys.argv:
        case_half_steps("weighted_nobias_f128_2000x1500", 2000, 1500, 150_000, 128, seed=18)
        sys.exit(0)
    case_weighted("weighted_nobias_f16", 300, 200, 6000, 16, False, 3, seed=11)
    case_weighted("weighted_bias_f8", 240, 160, 5000, 8, True, 3, seed=12)
    case_weighted("weighted_nobias_f64_linear", 200, 150, 6000, 64, False, 2, seed=13, mode="linear")
    case_weighted("weighted_bias_f64", 160, 130, 5000, 64, True, 2, seed=14)
    case_weighted("weighted_nobias_f128", 150, 260, 9000, 128, False, 2, seed=15)
    case_unweighted("unweighted_f12", 260, 180, 5000, 12, 3, seed=16)
    case_ease("ease_f300", 400, 300, 12000, 50.0, seed=17)
    case_half_steps("weighted_nobias_f128_2000x1500", 2000, 1500, 150_000, 128, seed=18)
