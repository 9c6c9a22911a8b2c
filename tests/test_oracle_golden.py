"""The oracle (oracle/wmf_oracle.py) against the golden vectors produced by the executed
reference (tests/golden/make_golden.py). CPU only."""
import numpy as np
import pytest

from conftest import WEIGHTED_CASES, csr_from, load_golden, load_golden_2000x1500, row_rel_err
from oracle import wmf_oracle as orc

HALF_STEP_TOL = 1e-4  # BASELINE.json north_star: 1e-4 relative per half-step


def _prep(g, mode):
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    C = tr.copy()
    C.data = orc.preprocess_counts(C.data, mode, 10, 1)
    return tr, te, C, C.T.tocsr()


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_init_matches_reference(name, dim, bias, mode):
    g = load_golden(name)
    items0 = orc.init_items(int(g["train_shape"][1]), dim, bias, seed=1993)
    assert items0.dtype == np.float32
    np.testing.assert_array_equal(items0, g["items0"])


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_half_steps_fp32_and_fp64(name, dim, bias, mode):
    g = load_golden(name)
    _, _, C, CT = _prep(g, mode)
    step = orc.half_step_bias if bias else orc.half_step
    u32 = step(g["items0"], C, 0.1, np.float32)
    assert u32.dtype == np.float32
    assert row_rel_err(u32, g["users_half1"]) < 1e-5  # same NumPy calls: rounding of BLAS only
    i32 = step(g["users_half1"], CT, 0.1, np.float32)
    assert row_rel_err(i32, g["items_half1"]) < 1e-5
    # the fp64 restatement bounds the reference's own fp32 noise floor (SURVEY.md §8c)
    # On these deliberately tiny, rank-deficient cases (f close to the row counts) the bias
    # formula's fp32 noise reaches 1.2e-4 by itself; realistic shapes sit at <= 4.4e-5.
    u64 = step(g["items0"], C, 0.1, np.float64)
    assert row_rel_err(u64, g["users_half1"]) < (3 * HALF_STEP_TOL if bias else HALF_STEP_TOL)


def test_half_step_bias_does_not_mutate():
    g = load_golden("weighted_bias_f8")
    _, _, C, _ = _prep(g, "log")
    Y = g["items0"].copy()
    orc.half_step_bias(Y, C, 0.1)
    np.testing.assert_array_equal(Y, g["items0"])


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_train_loop_and_metrics(name, dim, bias, mode):
    g = load_golden(name)
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    users, items, it, trace = orc.train(g["items0"], tr, int(g["train_iter"]) + 1, te, count_mat=tr, gamma=0.1,
                                        weighted=True, bias=bias, stopping_rounds=99, pre_process_count=mode)
    assert it == int(g["train_iter"])
    assert row_rel_err(users, g["users_final"]) < 1e-3  # several half-steps compound
    assert row_rel_err(items, g["items_final"]) < 1e-3
    assert abs(float(trace[-1]) - float(g["mse_final"])) < 1e-4 * float(g["mse_final"])
    U, V = g["users_final"], g["items_final"]
    assert float(orc.eval_prec(U, V, te, bias)) == pytest.approx(float(g["mse_final"]), rel=1e-6)
    assert float(orc.eval_prec(U, V, te, bias, "rmse")) == pytest.approx(float(g["rmse_final"]), rel=1e-6)
    assert float(orc.eval_prec(U, V, te, bias, "mae")) == pytest.approx(float(g["mae_final"]), rel=1e-6)
    assert orc.eval_prec_f64(U, V, te, bias) == pytest.approx(float(g["mse_final"]), rel=1e-5)
    with pytest.raises(ValueError):
        orc.eval_prec(U, V, te, bias, "nope")


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES[:2])
def test_early_stopping_epoch(name, dim, bias, mode):
    g = load_golden(name)
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    _, _, it, _ = orc.train(g["items0"], tr, 12, te, count_mat=tr, gamma=0.1, weighted=True, bias=bias,
                            stopping_rounds=2, pre_process_count=mode)
    assert it == int(g["early_iter"])


def test_bad_preprocess_mode():
    with pytest.raises(ValueError):
        orc.preprocess_counts(np.ones(3, np.float32), "sqrt")


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_predict_bit_exact_and_pairwise_restatement(name, dim, bias, mode):
    g = load_golden(name)
    U, V = g["users_final"], g["items_final"]
    p = orc.predict(U, V, g["pred_users"], g["pred_items"], bias)
    np.testing.assert_array_equal(p, g["pred"])
    # explicit restatement of NumPy's pairwise order
    if bias:
        prod = U[:, 1:][g["pred_users"]] * V[:, 1:][g["pred_items"]]
        q = orc.pairwise_sum_rows(prod) + U[:, 0][g["pred_users"]] + V[:, 0][g["pred_items"]]
    else:
        q = orc.pairwise_sum_rows(U[g["pred_users"]] * V[g["pred_items"]])
    np.testing.assert_array_equal(q, g["pred"])
    with pytest.raises(ValueError):
        orc.predict(U, V, [1, 2, 3], [1, 2], bias)


@pytest.mark.parametrize("n", [1, 5, 7, 8, 9, 16, 63, 64, 65, 127, 128, 129, 200, 256, 257, 300])
def test_pairwise_sum_matches_numpy(n):
    rng = np.random.default_rng(n)
    P = (rng.standard_normal((33, n)) * 10 ** rng.uniform(-3, 3, size=(33, n))).astype(np.float32)
    np.testing.assert_array_equal(orc.pairwise_sum_rows(P), P.sum(axis=1))


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_rank_matches_reference(name, dim, bias, mode):
    g = load_golden(name)
    U, V = g["users_final"], g["items_final"]
    all_items = np.arange(V.shape[0])
    for k, u in enumerate(g["rank_users"]):
        s = orc.rank_scores(U, V, all_items, int(u), bias)
        np.testing.assert_array_equal(s, g["rank_scores"][k])
        top = orc.rank(U, V, all_items, int(u), 10, bias)
        assert set(top.tolist()) == set(g["rank_top10"][k].tolist())
        np.testing.assert_array_equal(s[top], s[g["rank_top10"][k]])  # same order up to ties
    near = max(V.shape[0] - 3, 1)
    for k, u in enumerate(g["rank_users"][:4]):
        top = orc.rank(U, V, all_items, int(u), near, bias)
        np.testing.assert_array_equal(top, g["rank_near_full"][k])


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES[:2])
def test_eval_topn_protocol(name, dim, bias, mode):
    g = load_golden(name)
    U, V = g["users_final"], g["items_final"]
    te = csr_from(g, "test")

    def rank_fn(items, user, topn):
        return orc.rank(U, V, items, user, topn, bias)

    rec = orc.eval_topn(rank_fn, V.shape[0], te, g["topn"], rand_sampled=100, random_state=7)
    got = np.array([rec[f"Recall@{k}"] for k in g["topn"]], dtype=np.float64)
    np.testing.assert_allclose(got, g["recall"], atol=1e-7)
    with pytest.raises(ValueError):
        orc.eval_topn(rank_fn, V.shape[0], te, [10])


def test_unweighted_against_reference():
    g = load_golden("unweighted_f12")
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    users, items, it, trace = orc.train(g["items0"], tr, 1, te, gamma=0.1, weighted=None, dim=12, stopping_rounds=99)
    assert row_rel_err(users, g["users_ep1"]) < 1e-4
    assert row_rel_err(items, g["items_ep1"]) < 1e-4
    users, items, it, trace = orc.train(g["items0"], tr, 3, te, gamma=0.1, weighted=None, dim=12, stopping_rounds=99)
    assert it == int(g["train_iter"])
    assert float(trace[-1]) == pytest.approx(float(g["mse_final"]), rel=1e-3)


def test_unweighted_with_bias_raises_like_reference():
    # wmf_model.py:85 adds np.eye(dim) to a (dim+1)x(dim+1) Gram: shape error
    Y = np.ones((5, 4), np.float32)
    import scipy.sparse
    R = scipy.sparse.random(6, 5, density=0.5, format="csr", dtype=np.float32, random_state=0)
    with pytest.raises(ValueError):
        orc.unweighted_half_step(Y, R, 0.1, dim=3)


def test_algorithmic_bytes_match_survey():
    # SURVEY.md §8d: cfg2 = 20.97 GB / epoch
    b = orc.epoch_bytes(20_000_000, 138_493, 26_744, 128)
    assert abs(b / 1e9 - 20.97) < 0.02


def test_reference_constructor_and_half_step_golden():
    """The reference's WMF constructed with its default seed, and its recompute_factors from there, as stored by
    tests/golden/make_golden.py: this package's WMF starts from the same factors, and the oracle's half-step
    reproduces the reference's to BLAS rounding."""
    from recmodel_b200 import WMF
    g = load_golden("weighted_nobias_f16")
    _, _, C, _ = _prep(g, "log")
    m = WMF(num_items=C.shape[1], num_users=C.shape[0], dim=16, gamma=0.1, weighted=True)
    np.testing.assert_array_equal(m.items, g["items0"])
    assert row_rel_err(orc.half_step(m.items, C, 0.1), g["users_half1"]) < 1e-5


# ------------------------------------------------------------------------------- larger f = 128 fixture, EASE (N4)
def test_large_f128_half_steps_fp32_and_fp64():
    """2000 x 1500 fixture of the executed reference (tests/golden/make_golden.py::case_half_steps): the oracle's
    fp32 arithmetic reproduces it to BLAS rounding, the fp64 restatement within the first-half-step noise."""
    g = load_golden_2000x1500()
    C = csr_from(g, "train")
    C.data = orc.preprocess_counts(C.data)
    rows = slice(0, 300)
    u32 = orc.half_step(g["items0"], C[rows], 0.1)
    assert row_rel_err(u32, g["users_half1"][rows]) < 2e-4   # same formula, thread-count dependent BLAS rounding
    u64 = orc.half_step(g["items0"], C[rows], 0.1, np.float64)
    assert row_rel_err(g["users_half1"][rows], u64) < 5e-4


def test_ease_oracle_matches_executed_reference():
    g = load_golden("ease_f300")
    X = csr_from(g, "train")
    W = orc.ease_train(X, float(g["alpha"]))
    assert W.dtype == np.float32 and np.all(np.diag(W) == 0)
    scale = np.abs(g["W"]).max()
    assert np.max(np.abs(W - g["W"])) < 1e-5 * scale            # same LAPACK call, same dtype
    W64 = orc.ease_train(X, float(g["alpha"]), np.float64)
    assert np.max(np.abs(g["W"] - W64)) < 1e-4 * scale          # the reference's own fp32 noise
    pred = orc.ease_predict(X, g["W"], g["pred_users"], g["pred_items"])
    np.testing.assert_array_equal(pred, g["pred"])              # restated accumulation order is bit-exact
    for k, u in enumerate(g["rank_users"][:6]):
        np.testing.assert_array_equal(orc.ease_rank(X, g["W"], np.arange(X.shape[1]), int(u), 10), g["rank_top10"][k])
