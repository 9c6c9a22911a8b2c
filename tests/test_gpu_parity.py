"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on the same seeded
inputs and against the committed golden vectors of the executed reference.

Bars (BASELINE.json north_star): factors within 1e-4 relative per half-step (row-wise L2),
predict bit-exact, top-N index sets identical, Recall within 0.005 absolute.
"""
import numpy as np
import pytest
import scipy.sparse
import torch

from conftest import ROOT, WEIGHTED_CASES, csr_from, ledger_add, load_golden, load_golden_2000x1500, row_rel_err
from oracle import wmf_oracle as orc
from recmodel_b200 import WMF, _lib, engine
from recmodel_b200.engine import DeviceCSR
from recmodel_b200.synthetic import make_counts, make_counts_cached, split_train_test

pytestmark = pytest.mark.gpu

HALF_STEP_TOL = 1e-4
# "tcgen05": conjugate gradients on the matrix in tensor memory (the product); "tcgen05_direct": the same pipeline with
# every system factorised in tensor memory (the fallback of the former, kept tested on its own)
ALGOS = [("simt", _lib.ALGO_SIMT), ("tcgen05", _lib.ALGO_TCGEN05), ("tcgen05_direct", _lib.ALGO_TCGEN05_DIRECT)]
TC_ALGOS = (_lib.ALGO_TCGEN05, _lib.ALGO_TCGEN05_DIRECT)


def dev(a, cuda_device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)


def tc_supported(f, bias):
    return bool(_lib.load().wmf_als_half_step_supports(_lib.ALGO_TCGEN05, int(f), int(bool(bias))))


def half_step_tol(Y, C, ref32, bias):
    """1e-4, widened only where the reference's own fp32 arithmetic is noisier than that
    against the fp64 restatement (tiny rank-deficient fixtures)."""
    step = orc.half_step_bias if bias else orc.half_step
    x64 = step(Y, C, 0.1, np.float64)
    noise = row_rel_err(ref32, x64)
    return x64, max(HALF_STEP_TOL, 2.0 * noise)


def check_half_step(case, algo_name, X, ref32, x64, steady=False):
    """Record (error vs the fp32 reference, error vs the fp64 restatement, the reference's own fp32 noise, the
    tolerance used) in the parity ledger and apply the bar. The tcgen05 path (the product) is gated at PLAIN 1e-4
    against fp64; against the fp32 reference the bar is 1e-4 unless the reference itself is further than that from
    fp64 on this input (first half-steps from the all-positive initialisation), where 1.5 x its noise applies.
    The CUDA-core cross-check kernel solves the unwhitened system like the reference and shares its conditioning:
    max(1e-4, 2 x noise)."""
    noise = row_rel_err(ref32, x64)
    err32, err64 = row_rel_err(X, ref32), row_rel_err(X, x64)
    if algo_name.startswith("tcgen05"):
        tol64, tol32 = HALF_STEP_TOL, max(HALF_STEP_TOL, 1.5 * noise)
    else:
        tol64 = tol32 = HALF_STEP_TOL if steady else max(HALF_STEP_TOL, 2.0 * noise)
    ledger_add(case, algo_name, err_vs_ref32=err32, err_vs_fp64=err64, ref_noise=noise, tol_vs_fp64=tol64, tol_vs_ref32=tol32)
    print(f"{case} [{algo_name}]: vs fp64 {err64:.2e} (tol {tol64:.1e}), vs ref32 {err32:.2e} (tol {tol32:.1e}), ref noise {noise:.2e}")
    assert err64 < tol64, (case, algo_name, err64, tol64)
    assert err32 < tol32, (case, algo_name, err32, tol32)
    return err64


def run_half_step(Y, C, bias, algo, cuda_device, use_row_order=True):
    Yd = dev(Y, cuda_device)
    Cd = DeviceCSR.from_scipy(C, cuda_device)
    G = engine.gram(Yd, 0.1, ones_col0=bias)
    X = engine.half_step(Cd, Yd, G, bias=bias, algo=algo, use_row_order=use_row_order)
    torch.cuda.synchronize()
    return X.cpu().numpy(), G.cpu().numpy()


# ------------------------------------------------------------------------------- K6, K1
def test_device_is_b200(cuda_device):
    assert _lib.require_device() >= 100
    assert torch.cuda.get_device_capability(0)[0] == 10


def test_preprocess_matches_numpy(cuda_device):
    x = np.random.default_rng(0).integers(1, 50, size=100_003).astype(np.float32)
    for mode in ("log", "linear"):
        d = engine.preprocess_(dev(x, cuda_device).clone(), mode, 10, 1).cpu().numpy()
        np.testing.assert_allclose(d, orc.preprocess_counts(x, mode, 10, 1), rtol=3e-7)
    with pytest.raises(ValueError):
        engine.preprocess_(dev(x, cuda_device), "sqrt", 10, 1)


@pytest.mark.parametrize("n,f,ones", [(1, 8, False), (1000, 16, False), (3706, 65, True), (26_744, 128, False),
                                      (5000, 129, True), (777, 256, False), (300, 257, True)])
def test_gram_matches_fp64(cuda_device, n, f, ones):
    Y = np.random.default_rng(n + f).random((n, f)).astype(np.float32)
    G = engine.gram(dev(Y, cuda_device), 0.1, ones_col0=ones).cpu().numpy()
    Y64 = Y.astype(np.float64)
    if ones:
        Y64[:, 0] = 1
    ref = Y64.T @ Y64 + 0.1 * np.eye(f)
    assert np.max(np.abs(G - ref) / np.abs(ref).max()) < 1.5e-7  # one fp32 rounding of the largest entry
    G2 = engine.gram(dev(Y, cuda_device), 0.1, ones_col0=ones).cpu().numpy()
    np.testing.assert_array_equal(G, G2)  # deterministic reduction order


@pytest.mark.parametrize("n,f,ones", [(26_744, 128, False), (3706, 65, True), (700, 16, False), (31, 8, False)])
def test_gram_block_partials_reproduce_gram(cuda_device, n, f, ones):
    """Row-sharded Gram: block partials computed shard by shard (foreign blocks zero) and summed reproduce
    the one-call Gram bit for bit, for any split into whole blocks (include/wmf_b200.h)."""
    from recmodel_b200 import sharding
    Y = (np.random.default_rng(n).standard_normal((n, f)) * 0.5 + 0.3).astype(np.float32)
    Yd = dev(Y, cuda_device)
    G = engine.gram(Yd, 0.1, ones_col0=ones).cpu().numpy()
    B = engine.gram_block_rows(n)
    counts = np.random.default_rng(1).integers(0, 50, n)
    for world in (2, 3, 8):
        bounds = sharding.balanced_row_partition(counts, world, f, align=B)
        assert all(b % B == 0 or b == n for b in bounds)
        total = None
        for g in range(world):
            part = engine.gram_partials(Yd[int(bounds[g]):int(bounds[g + 1])], int(bounds[g]), n, ones_col0=ones)
            total = part if total is None else total + part  # what the sum all-reduce does (x + 0 is exact)
        G2 = engine.gram_from_partials(total, n, 0.1).cpu().numpy()
        np.testing.assert_array_equal(G, G2)
    np.testing.assert_array_equal(G, G.T)


@pytest.mark.parametrize("rows,cols,nnz", [(700, 450, 20_000), (3, 70_000, 5_000), (5000, 1, 800), (6040, 3706, 1_000_000),
                                           (40, 300_000, 90_000)])
def test_transpose_matches_scipy(cuda_device, rows, cols, nnz):
    """N1: the library's stable radix sort by column reproduces count_mat.T.tocsr() (wmf_model.py:128) exactly:
    row pointer, ascending row ids inside every output row, values."""
    C = make_counts(rows, cols, nnz, seed=21)
    CT = DeviceCSR.from_scipy(C, cuda_device).transpose().to_scipy()
    ref = C.T.tocsr()
    np.testing.assert_array_equal(CT.indptr, ref.indptr)
    np.testing.assert_array_equal(CT.indices, ref.indices)
    np.testing.assert_array_equal(CT.data, ref.data)


def test_transpose_unsorted_duplicates_and_canonical(cuda_device):
    """Unsorted column order inside rows, duplicate (row, column) entries and empty rows: the transpose keeps every
    entry (SciPy does not sum duplicates either) in CSR traversal order; two transposes give sorted indices."""
    rng = np.random.default_rng(4)
    rows, cols = 300, 200
    lens = rng.integers(0, 40, rows)
    lens[[3, 77]] = 0
    indptr = np.concatenate([[0], np.cumsum(lens)])
    indices = np.concatenate([rng.integers(0, cols, n) for n in lens]).astype(np.int32)   # unsorted, with repeats
    data = rng.random(indptr[-1]).astype(np.float32)
    C = scipy.sparse.csr_matrix((data, indices, indptr), shape=(rows, cols))
    Cd = DeviceCSR(dev(indptr.astype(np.int64), cuda_device), dev(indices, cuda_device), dev(data, cuda_device), (rows, cols))
    CT = Cd.transpose().to_scipy()
    ref = C.T.tocsr()   # csc -> csr: counting sort in traversal order, duplicates kept
    np.testing.assert_array_equal(CT.indptr, ref.indptr)
    np.testing.assert_array_equal(CT.indices, ref.indices)
    np.testing.assert_array_equal(CT.data, ref.data)
    canon = Cd.canonical().to_scipy()
    assert canon.shape == C.shape and canon.nnz == C.nnz
    assert all(np.all(np.diff(canon.indices[canon.indptr[r]:canon.indptr[r + 1]]) >= 0) for r in range(rows))
    assert abs(canon - C).max() < 1e-6
    empty = DeviceCSR(torch.zeros(6, dtype=torch.int64, device=cuda_device), torch.empty(0, dtype=torch.int32, device=cuda_device),
                      torch.empty(0, dtype=torch.float32, device=cuda_device), (5, 9)).transpose()
    assert empty.shape == (9, 5) and int(empty.indptr.abs().sum()) == 0


# ------------------------------------------------------------------------------- K2
@pytest.mark.parametrize("algo_name,algo", ALGOS)
@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_half_step_vs_reference_golden(cuda_device, name, dim, bias, mode, algo_name, algo):
    f = dim + 1 if bias else dim
    if algo in TC_ALGOS and not tc_supported(f, bias):
        pytest.skip("shape not taken by the tcgen05 path")
    g = load_golden(name)
    C = csr_from(g, "train")
    C.data = orc.preprocess_counts(C.data, mode, 10, 1)
    CT = C.T.tocsr()
    step = orc.half_step_bias if bias else orc.half_step
    X, _ = run_half_step(g["items0"], C, bias, algo, cuda_device)
    check_half_step(f"golden/{name}/users_half1", algo_name, X, g["users_half1"], step(g["items0"], C, 0.1, np.float64))
    Xi, _ = run_half_step(g["users_half1"], CT, bias, algo, cuda_device)
    check_half_step(f"golden/{name}/items_half1", algo_name, Xi, g["items_half1"],
                    step(g["users_half1"], CT, 0.1, np.float64))


@pytest.mark.parametrize("algo_name,algo", ALGOS)
@pytest.mark.parametrize("users,items,nnz,dim,bias", [
    (6040, 3706, 1_000_000, 64, True),     # config 1 in full (ML-1M shape, bias)
    (6040, 3706, 1_000_000, 64, False),
    (3000, 2000, 300_000, 128, False),     # config-2 arithmetic (f=128) at an oracle-sized shape
    (1500, 1200, 150_000, 128, True),
])
def test_half_step_vs_oracle_realistic(cuda_device, users, items, nnz, dim, bias, algo_name, algo):
    f = dim + 1 if bias else dim
    if algo in TC_ALGOS and not tc_supported(f, bias):
        pytest.skip("shape not taken by the tcgen05 path")
    C = make_counts_cached(users, items, nnz, seed=31)
    C.data = orc.preprocess_counts(C.data)
    CT = C.T.tocsr()
    Y = orc.init_items(items, dim, bias)
    step = orc.half_step_bias if bias else orc.half_step
    # First half-step from the all-positive U[0,1) initialisation: the worst-conditioned one.
    # The reference's own fp32 arithmetic is 4e-5 (no bias) .. 1.2e-4 (bias) away from the fp64
    # restatement here, so the bar is: no further from fp64 than max(1e-4, 2 x that noise), and
    # within the same distance of the fp32 reference.
    rows = slice(0, min(users, 1500))
    ref_u = step(Y, C[rows], 0.1)
    X, _ = run_half_step(Y, C, bias, algo, cuda_device)
    case = f"realistic/{users}x{items}/f{f}{'b' if bias else ''}"
    check_half_step(case + "/first_user_half_step", algo_name, X[rows], ref_u, step(Y, C[rows], 0.1, np.float64))
    # second half-step from mixed-sign factors (the steady-state regime): plain 1e-4
    full_u = X if users <= 1500 else step(Y, C, 0.1)
    sel = slice(0, min(items, 800))
    ref_i = step(full_u, CT[sel], 0.1)
    Xi, _ = run_half_step(full_u, CT[sel], bias, algo, cuda_device)
    check_half_step(case + "/item_half_step", algo_name, Xi, ref_i, step(full_u, CT[sel], 0.1, np.float64), steady=True)


@pytest.mark.parametrize("algo_name,algo", ALGOS)
@pytest.mark.parametrize("f,bias", [(8, False), (9, True), (64, False), (65, True), (128, False), (129, True),
                                    (200, False), (256, False), (257, True)])
def test_half_step_edge_rows(cuda_device, f, bias, algo_name, algo):
    """Empty rows, 1-entry rows, a row much longer than f, unsorted column order, explicit zero
    weights (SURVEY.md §4 unit level)."""
    if algo in TC_ALGOS and not tc_supported(f, bias):
        pytest.skip("shape not taken by the tcgen05 path")
    rng = np.random.default_rng(f)
    N = 900
    lens = [0, 1, 1, 0, 2, 5, 33, 700, 0, 17, 64, 3, 0]
    indptr = np.concatenate([[0], np.cumsum(lens)])
    indices = np.concatenate([rng.permutation(N)[:n] for n in lens]).astype(np.int32)  # unsorted inside rows
    data = (rng.random(indptr[-1]) * 20).astype(np.float32)
    data[::7] = 0.0
    C = scipy.sparse.csr_matrix((data, indices, indptr), shape=(len(lens), N))
    Y = (rng.standard_normal((N, f)) * 0.3).astype(np.float32)
    if bias:
        Y[:, 0] = rng.random(N).astype(np.float32)
    step = orc.half_step_bias if bias else orc.half_step
    ref = step(Y, C, 0.1)
    X, _ = run_half_step(Y, C, bias, algo, cuda_device)
    assert np.all(X[np.array(lens) == 0] == 0)
    check_half_step(f"edge_rows/f{f}{'b' if bias else ''}", algo_name, X, ref, step(Y, C, 0.1, np.float64))
    X2, _ = run_half_step(Y, C, bias, algo, cuda_device, use_row_order=False)
    np.testing.assert_array_equal(X, X2)  # processing order never changes a row's arithmetic


@pytest.mark.parametrize("algo_name,algo", ALGOS)
def test_half_step_indefinite_falls_back_to_lu(cuda_device, algo_name, algo):
    """Negative confidence weights make A indefinite; the reference's sgesv still solves it."""
    if algo in TC_ALGOS and not tc_supported(64, False):
        pytest.skip("shape not taken by the tcgen05 path")
    rng = np.random.default_rng(5)
    N, f = 400, 64
    C = scipy.sparse.random(40, N, density=0.2, format="csr", dtype=np.float32, random_state=3)
    C.data = (-(C.data * 30) - 5).astype(np.float32)
    Y = (rng.standard_normal((N, f)) * 0.4).astype(np.float32)
    ref = orc.half_step(Y, C, 0.1)
    x64, tol = half_step_tol(Y, C, ref, False)
    X, _ = run_half_step(Y, C, False, algo, cuda_device)
    assert np.all(np.isfinite(X))
    err = row_rel_err(X, x64)
    ledger_add("indefinite_negative_weights/f64", algo_name, err_vs_ref32=row_rel_err(X, ref), err_vs_fp64=err,
               ref_noise=row_rel_err(ref, x64), tol_vs_fp64=max(tol, 1e-3), tol_vs_ref32=None)
    assert err < max(tol, 1e-3)  # indefinite systems: conditioning-limited (LU kernel on both paths)
    if algo in TC_ALGOS:  # every row with entries went through the per-row fix-up list, none through a redo
        flags, fixed = engine.half_step_status()
        assert fixed == int((np.diff(C.indptr) > 0).sum()) and (flags & 2) == 0


@pytest.mark.parametrize("f", [32, 128, 200])
def test_half_step_cg_falls_back_to_factorisation(cuda_device, f):
    """Weights in the thousands (linear preprocessing of large counts) put the whitened systems at condition numbers
    the conjugate gradients do not resolve within their product budget: those rows are factorised in tensor memory
    instead (the block Gauss-Jordan that WMF_ALGO_TCGEN05_DIRECT applies to every row), from the untouched matrix.
    Both algorithms then agree with the fp64 restatement to the conditioning-limited noise of fp32 and with each other;
    on the reference's own weightings no row takes the fallback."""
    if not tc_supported(f, False):
        pytest.skip("shape not taken by the tcgen05 path")
    C = make_counts(700, 500, 60_000, seed=11)
    rng = np.random.default_rng(8)
    C.data = (C.data * rng.uniform(500.0, 4000.0, size=C.nnz)).astype(np.float32)   # d up to 2e4
    Y = orc.init_items(500, f, False)
    ref = orc.half_step(Y, C, 0.1)
    x64, tol = half_step_tol(Y, C, ref, False)
    X, _ = run_half_step(Y, C, False, _lib.ALGO_TCGEN05, cuda_device)
    fallback = engine.half_step_used_fallback()
    Xd, _ = run_half_step(Y, C, False, _lib.ALGO_TCGEN05_DIRECT, cuda_device)
    assert np.all(np.isfinite(X)) and np.all(np.isfinite(Xd))
    noise = row_rel_err(ref, x64)
    e_cg, e_direct = row_rel_err(X, x64), row_rel_err(Xd, x64)
    ledger_add(f"heavy_weights/f{f}", "tcgen05", err_vs_ref32=row_rel_err(X, ref), err_vs_fp64=e_cg, ref_noise=noise,
               tol_vs_fp64=tol, tol_vs_ref32=None)
    ledger_add(f"heavy_weights/f{f}", "tcgen05_direct", err_vs_ref32=row_rel_err(Xd, ref), err_vs_fp64=e_direct, ref_noise=noise,
               tol_vs_fp64=tol, tol_vs_ref32=None)
    print(f"heavy weights f={f}: factorisation used: {fallback}; vs fp64: cg path {e_cg:.2e}, direct {e_direct:.2e}, "
          f"reference {noise:.2e} (tol {tol:.1e})")
    assert fallback, "no row took the factorisation: the fallback is not exercised"
    assert e_cg < tol and e_direct < tol
    # the reference's weighting: nothing falls back
    C2 = make_counts(700, 500, 60_000, seed=11)
    C2.data = orc.preprocess_counts(C2.data)
    run_half_step(Y, C2, False, _lib.ALGO_TCGEN05, cuda_device)
    assert not engine.half_step_used_fallback()


def test_half_step_split_rows(cuda_device):
    """Rows longer than wmf_als_row_split_entries() are accumulated by several CTAs (tcgen05 path) and their
    partial Grams summed in segment order: same accuracy bar, bitwise independent of the schedule and of
    which other rows share the launch (row sharding)."""
    f = 128
    if not tc_supported(f, False):
        pytest.skip("shape not taken by the tcgen05 path")
    split = int(_lib.load().wmf_als_row_split_entries())
    rng = np.random.default_rng(77)
    N, R = 70_000, 1200
    lens = rng.integers(0, 120, R)
    lens[[3, 40, 41, 700, 1199]] = [6 * split + 5, split + 1, split, 2 * split + 1000, 3 * split]
    indptr = np.concatenate([[0], np.cumsum(lens)])
    indices = np.concatenate([np.sort(rng.choice(N, n, replace=False)) for n in lens]).astype(np.int32)
    data = orc.preprocess_counts(rng.integers(1, 6, indptr[-1]).astype(np.float32))
    C = scipy.sparse.csr_matrix((data, indices, indptr), shape=(R, N))
    Y = (rng.standard_normal((N, f)) * 0.2).astype(np.float32)
    X, _ = run_half_step(Y, C, False, _lib.ALGO_TCGEN05, cuda_device)
    assert np.all(np.isfinite(X))
    check = np.array([3, 40, 41, 700, 1199, 0, 1, 2, 500])
    ref = orc.half_step(Y, C[check], 0.1)
    check_half_step("split_rows/f128", "tcgen05", X[check], ref, orc.half_step(Y, C[check], 0.1, np.float64))
    Xs, _ = run_half_step(Y, C, False, _lib.ALGO_SIMT, cuda_device)
    assert row_rel_err(X, Xs) < HALF_STEP_TOL
    X2, _ = run_half_step(Y, C, False, _lib.ALGO_TCGEN05, cuda_device, use_row_order=False)
    np.testing.assert_array_equal(X, X2)
    Xa, _ = run_half_step(Y, C[:650], False, _lib.ALGO_TCGEN05, cuda_device)
    np.testing.assert_array_equal(Xa, X[:650])
    Xb, _ = run_half_step(Y, C[650:], False, _lib.ALGO_TCGEN05, cuda_device)
    np.testing.assert_array_equal(Xb, X[650:])


def test_half_step_full_size_properties(cuda_device):
    """Config 2 at full size (138 493 x 26 744, 20 M entries, f=128): size-independent checks.
    (1) normal-equation residual of sampled rows in fp64; (2) bitwise determinism;
    (3) a 2-way row shard reproduces the unsharded rows bit for bit."""
    users, items, nnz, f = 138_493, 26_744, 20_000_000, 128
    C = make_counts_cached(users, items, nnz)
    C.data = orc.preprocess_counts(C.data)
    Y = orc.init_items(items, f, False)
    Yd = dev(Y, cuda_device)
    Cd = DeviceCSR.from_scipy(C, cuda_device)
    G = engine.gram(Yd, 0.1)
    X = engine.half_step(Cd, Yd, G).cpu().numpy()
    assert np.all(np.isfinite(X))
    G64 = Y.astype(np.float64).T @ Y.astype(np.float64) + 0.1 * np.eye(f)
    G32 = np.dot(Y.T, Y) + np.float32(0.1) * np.eye(f, dtype=np.float32)
    worst = worst_noise = 0.0
    rows = np.concatenate([np.random.default_rng(1).integers(0, users, 48), [int(np.argmax(np.diff(C.indptr)))]])
    for r in rows:
        lo, hi = C.indptr[r], C.indptr[r + 1]
        if lo == hi:
            assert np.all(X[r] == 0)
            continue
        Yr = Y[C.indices[lo:hi]].astype(np.float64)
        d = C.data[lo:hi].astype(np.float64)
        A = G64 + (Yr * d[:, None]).T @ Yr
        x = np.linalg.solve(A, (d + 1) @ Yr)
        # the reference's own fp32 arithmetic for this row (np.dot / sgesv), as the noise yardstick
        Yr32 = Y[C.indices[lo:hi]]
        x32 = np.linalg.solve(np.dot(Yr32.T, Yr32 * C.data[lo:hi, None]) + G32, np.dot(C.data[lo:hi] + 1, Yr32))
        noise = np.linalg.norm(x32 - x) / np.linalg.norm(x)
        worst_noise = max(worst_noise, noise)
        worst = max(worst, np.linalg.norm(X[r] - x) / np.linalg.norm(x))
    print(f"full size: worst gpu-vs-fp64 {worst:.2e}; reference fp32-vs-fp64 on the same rows {worst_noise:.2e}")
    ledger_add("cfg2_full/first_user_half_step(49 rows)", "tcgen05", err_vs_ref32=None, err_vs_fp64=worst,
               ref_noise=worst_noise, tol_vs_fp64=HALF_STEP_TOL, tol_vs_ref32=None)
    assert worst < HALF_STEP_TOL
    X2 = engine.half_step(Cd, Yd, G).cpu().numpy()
    np.testing.assert_array_equal(X, X2)
    half = users // 2
    Xa = engine.half_step(Cd.row_slice(0, half), Yd, G).cpu().numpy()
    np.testing.assert_array_equal(Xa, X[:half])
    # (4) item side: the heaviest rows (50k-110k entries) are where an accumulation bias shows (the tensor core
    # truncates its fp32 accumulation; long rows are cut into segments summed with round-to-nearest adds)
    Xd = torch.from_numpy(X).to(cuda_device)
    CTd = Cd.transpose()
    Gi = engine.gram(Xd, 0.1)
    Xi = engine.half_step(CTd, Xd, Gi).cpu().numpy()
    CT = C.T.tocsr()
    lens = np.diff(CT.indptr)
    order = np.argsort(-lens)
    X64 = X.astype(np.float64)
    Gi64 = X64.T @ X64 + 0.1 * np.eye(f)
    worst_i = 0.0
    for r in np.concatenate([order[:3], order[200:202], order[5000:5002]]):
        lo, hi = CT.indptr[r], CT.indptr[r + 1]
        Yr = X64[CT.indices[lo:hi]]
        d = CT.data[lo:hi].astype(np.float64)
        x = np.linalg.solve(Gi64 + (Yr * d[:, None]).T @ Yr, (d + 1) @ Yr)
        worst_i = max(worst_i, np.linalg.norm(Xi[r] - x) / np.linalg.norm(x))
    print(f"full size, item side: worst gpu-vs-fp64 over rows of {lens[order[0]]} .. {lens[order[5001]]} entries {worst_i:.2e}")
    ledger_add("cfg2_full/item_half_step(heaviest rows)", "tcgen05", err_vs_ref32=None, err_vs_fp64=worst_i,
               ref_noise=None, tol_vs_fp64=HALF_STEP_TOL / 2, tol_vs_ref32=None)
    assert worst_i < HALF_STEP_TOL / 2
    Xib = engine.half_step(CTd.row_slice(0, items // 3), Xd, Gi).cpu().numpy()
    np.testing.assert_array_equal(Xib, Xi[:items // 3])


# ------------------------------------------------------------------------------- R8, K3
@pytest.mark.parametrize("f,bias", [(5, False), (7, True), (16, False), (64, False), (65, True), (128, False),
                                    (129, True), (200, False), (256, False), (257, True), (300, False)])
def test_predict_bit_exact(cuda_device, f, bias):
    rng = np.random.default_rng(f)
    U = (rng.standard_normal((300, f)) * 10 ** rng.uniform(-2, 2, (300, f))).astype(np.float32)
    V = (rng.standard_normal((500, f)) * 10 ** rng.uniform(-2, 2, (500, f))).astype(np.float32)
    us, it = rng.integers(0, 300, 4001), rng.integers(0, 500, 4001)
    m = WMF(num_items=500, num_users=300, dim=f - 1 if bias else f, gamma=0.1, weighted=True, bias=bias)
    m.users, m.items = U, V
    np.testing.assert_array_equal(m.predict(us, it), orc.predict(U, V, us, it, bias))
    np.testing.assert_array_equal(m.predict(7, np.arange(500)), orc.predict(U, V, 7, np.arange(500), bias))
    with pytest.raises(ValueError):
        m.predict([1, 2, 3], [1, 2])


@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_predict_and_metrics_vs_golden(cuda_device, name, dim, bias, mode):
    g = load_golden(name)
    te = csr_from(g, "test")
    m = WMF(num_items=g["items_final"].shape[0], num_users=g["users_final"].shape[0], dim=dim, gamma=0.1,
            weighted=True, bias=bias)
    m.users, m.items = g["users_final"], g["items_final"]
    np.testing.assert_array_equal(m.predict(g["pred_users"], g["pred_items"]), g["pred"])
    assert float(m.eval_prec(te)) == pytest.approx(float(g["mse_final"]), rel=2e-6)
    assert float(m.eval_prec(te, "rmse")) == pytest.approx(float(g["rmse_final"]), rel=2e-6)
    assert float(m.eval_prec(te, metric="MAE")) == pytest.approx(float(g["mae_final"]), rel=2e-6)
    with pytest.raises(ValueError):
        m.eval_prec(te, "nope")
    te0 = te.copy()
    te0.data[::3] = 0.0  # explicit zeros are skipped like nonzero() does
    ref = orc.eval_prec_f64(g["users_final"], g["items_final"], te0, bias)
    assert float(m.eval_prec(te0)) == pytest.approx(ref, rel=2e-6)


def test_sddmm_loss_large_and_deterministic(cuda_device):
    C = make_counts_cached(6040, 3706, 1_000_000, seed=31)
    rng = np.random.default_rng(2)
    U = (rng.standard_normal((6040, 128)) * 0.2).astype(np.float32)
    V = (rng.standard_normal((3706, 128)) * 0.2).astype(np.float32)
    Cd = DeviceCSR.from_scipy(C, cuda_device)
    s1 = engine.sddmm_loss(Cd, dev(U, cuda_device), dev(V, cuda_device)).cpu().numpy()
    s2 = engine.sddmm_loss(Cd, dev(U, cuda_device), dev(V, cuda_device)).cpu().numpy()
    np.testing.assert_array_equal(s1, s2)
    assert s1[2] == C.nnz
    assert s1[0] / s1[2] == pytest.approx(orc.eval_prec_f64(U, V, C, False), rel=1e-9)


# ------------------------------------------------------------------------------- R10
@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_rank_vs_golden(cuda_device, name, dim, bias, mode):
    g = load_golden(name)
    V = g["items_final"]
    m = WMF(num_items=V.shape[0], num_users=g["users_final"].shape[0], dim=dim, gamma=0.1, weighted=True, bias=bias)
    m.users, m.items = g["users_final"], V
    all_items = np.arange(V.shape[0])
    for k, u in enumerate(g["rank_users"]):
        top = m.rank(all_items, int(u), 10)
        assert top.dtype == all_items.dtype and len(top) == 10
        assert set(top.tolist()) == set(g["rank_top10"][k].tolist())
        s = g["rank_scores"][k]
        np.testing.assert_array_equal(s[top], s[g["rank_top10"][k]])  # same order up to exact ties
    lst = m.rank(all_items, [int(u) for u in g["rank_users"]], 10)
    assert isinstance(lst, list) and len(lst) == len(g["rank_users"])
    for k in range(len(lst)):
        np.testing.assert_array_equal(lst[k], m.rank(all_items, int(g["rank_users"][k]), 10))
    near = max(V.shape[0] - 3, 1)
    for k, u in enumerate(g["rank_users"][:4]):
        s = g["rank_scores"][k]
        top = m.rank(all_items, int(u), near)
        np.testing.assert_array_equal(s[top], s[g["rank_near_full"][k]])
    assert len(m.rank(all_items, 3)) == V.shape[0]           # topn=None ranks everything
    assert len(m.rank(all_items[:5], 3, 50)) == 5            # topn > len(items) returns len(items)
    sub = np.array([9, 3, 3, 17, 4], dtype=np.int32)         # duplicates + caller's dtype
    out = m.rank(sub, 2, 3)
    assert out.dtype == np.int32 and set(out.tolist()) <= set(sub.tolist())


@pytest.mark.parametrize("f,bias,ni,topn", [(64, False, 3706, 100), (128, False, 26_744, 100), (65, True, 5000, 20),
                                            (257, True, 1500, 1024), (16, False, 40, 40), (128, False, 3000, 2000)])
def test_rank_sets_bit_exact_vs_oracle(cuda_device, f, bias, ni, topn):
    rng = np.random.default_rng(ni + f)
    nu = 37
    U = (rng.standard_normal((nu, f)) * 0.5).astype(np.float32)
    V = (rng.standard_normal((ni, f)) * 0.5).astype(np.float32)
    V[ni // 2] = V[ni // 3]  # an exact tie
    m = WMF(num_items=ni, num_users=nu, dim=f - 1 if bias else f, gamma=0.1, weighted=True, bias=bias)
    m.users, m.items = U, V
    cand = np.arange(ni)
    got = m.rank_batch(cand, np.arange(nu), topn)
    for u in range(nu):
        s = orc.rank_scores(U, V, cand, u, bias)
        kth = np.sort(s)[-topn]
        must = set(np.nonzero(s > kth)[0].tolist())
        may = set(np.nonzero(s >= kth)[0].tolist())
        sel = set(got[u].tolist())
        assert len(sel) == topn and must <= sel <= may
        assert np.all(np.diff(s[got[u]]) <= 0)  # descending


def test_rank_all_equal_scores_ties_by_position(cuda_device):
    m = WMF(num_items=300, num_users=2, dim=8, gamma=0.1, weighted=True)
    m.users, m.items = np.ones((2, 8), np.float32), np.ones((300, 8), np.float32)
    np.testing.assert_array_equal(m.rank(np.arange(300), 0, 7), np.arange(7))


@pytest.mark.parametrize("f,bias,ni,topn,shuffled", [(128, False, 26_744, 100, False), (65, True, 9000, 50, True),
                                                     (32, False, 4096, 128, False), (127, True, 3000, 10, True)])
def test_rank_tensor_core_path_equals_exact_path(cuda_device, monkeypatch, f, bias, ni, topn, shuffled):
    """K4/K5: tcgen05 candidate generation + exact rescoring must return the exact path's lists, element for
    element (same sets, same order, ties by candidate position). The exact path is the one the tests above pin
    against the oracle; WMF_SCORE_EXACT=1 forces it."""
    rng = np.random.default_rng(7 * ni + f)
    nu = 300
    scale = np.float32(10.0 ** rng.uniform(-3, 2))  # the power-of-two operand scaling must not matter
    U = (rng.standard_normal((nu, f)) * scale).astype(np.float32)
    V = (rng.standard_normal((ni, f)) * 0.3).astype(np.float32)
    V[ni // 2] = V[ni // 3]                      # an exact tie
    V[7] = 0                                     # a zero row
    m = WMF(num_items=ni, num_users=nu, dim=f - 1 if bias else f, gamma=0.1, weighted=True, bias=bias)
    m.users, m.items = U, V
    cand = rng.permutation(ni)[: ni - 17] if shuffled else np.arange(ni)
    assert _lib.load().wmf_score_topk_workspace_bytes(nu, len(cand), topn) > nu * len(cand) * 4  # tc scratch included
    got = m.rank_batch(cand, np.arange(nu), topn)
    monkeypatch.setenv("WMF_SCORE_EXACT", "1")
    ref = m.rank_batch(cand, np.arange(nu), topn)
    np.testing.assert_array_equal(got, ref)
    for u in (0, 5, nu - 1):                      # and the exact path itself against the oracle
        s = orc.rank_scores(U, V, cand, u, bias)
        pos = {int(c): k for k, c in enumerate(cand)}
        np.testing.assert_array_equal(np.sort(s[[pos[int(i)] for i in ref[u]]])[::-1], np.sort(s)[::-1][:topn])


def test_rank_tensor_core_overflow_falls_back_to_exact(cuda_device):
    """More than 1024 candidates within the error band (all scores equal): the flag makes the exact kernels
    redo the call, ties by position."""
    ni = 5000
    m = WMF(num_items=ni, num_users=3, dim=16, gamma=0.1, weighted=True)
    m.users, m.items = np.ones((3, 16), np.float32), np.ones((ni, 16), np.float32)
    out = m.rank_batch(np.arange(ni), np.arange(3), 40)
    np.testing.assert_array_equal(out, np.tile(np.arange(40), (3, 1)))


# ------------------------------------------------------------------------------- R2, R11, R12
@pytest.mark.parametrize("algo_name", ["simt", "tcgen05"])
@pytest.mark.parametrize("name,dim,bias,mode", WEIGHTED_CASES)
def test_train_vs_reference_golden(cuda_device, name, dim, bias, mode, algo_name, capsys):
    f = dim + 1 if bias else dim
    if algo_name == "tcgen05" and not tc_supported(f, bias):
        pytest.skip("shape not taken by the tcgen05 path")
    g = load_golden(name)
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    tr_before = tr.copy()
    m = WMF(num_items=tr.shape[1], num_users=tr.shape[0], dim=dim, gamma=0.1, weighted=True, bias=bias, seed=1993,
            algo=algo_name)
    it = m.train(tr.copy(), iterations=int(g["train_iter"]) + 1, eval_mat=te, count_mat=tr, cores=1,
                 stopping_rounds=99, pre_process_count=mode)
    assert it == int(g["train_iter"])
    assert (tr != tr_before).nnz == 0  # inputs are never mutated
    # several half-steps compound; the per-half-step bar is checked above
    ill = name in ("weighted_bias_f64", "weighted_nobias_f128", "weighted_nobias_f64_linear")
    tol = 2e-2 if ill else 2e-3
    assert row_rel_err(m.users, g["users_final"]) < tol
    assert row_rel_err(m.items, g["items_final"]) < tol
    assert float(m.eval_prec(te)) == pytest.approx(float(g["mse_final"]), rel=1e-3)
    if not ill:
        m2 = WMF(num_items=tr.shape[1], num_users=tr.shape[0], dim=dim, gamma=0.1, weighted=True, bias=bias,
                 algo=algo_name)
        assert m2.train(tr, iterations=12, eval_mat=te, count_mat=tr, cores=4, stopping_rounds=2,
                        pre_process_count=mode) == int(g["early_iter"])
        rec = m.eval_topn(te.copy(), topn=g["topn"], rand_sampled=100, cores=1, random_state=7)
        got = np.array([rec[f"Recall@{k}"] for k in g["topn"]], dtype=np.float64)
        assert np.max(np.abs(got - g["recall"])) <= 0.005


def test_train_argument_errors(cuda_device):
    g = load_golden("weighted_nobias_f16")
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    m = WMF(num_items=tr.shape[1], num_users=tr.shape[0], dim=16, gamma=0.1, weighted=True)
    with pytest.raises(ValueError):
        m.train(tr, 1, eval_mat=te, count_mat=tr, pre_process_count="sqrt")
    with pytest.raises(ValueError):
        m.train(tr, 1, eval_mat=te, count_mat=tr, cores=0)
    with pytest.raises(AttributeError):
        m.train(tr, 1, eval_mat=None, count_mat=tr, cores=1)
    mb = WMF(num_items=tr.shape[1], num_users=tr.shape[0], dim=16, gamma=0.1, weighted=False, bias=True)
    with pytest.raises(ValueError):
        mb.train(tr, 1, eval_mat=te)


def test_recompute_factors_methods(cuda_device):
    g = load_golden("weighted_bias_f8")
    C = csr_from(g, "train")
    C.data = orc.preprocess_counts(C.data)
    m = WMF(num_items=C.shape[1], num_users=C.shape[0], dim=8, gamma=0.1, weighted=True, bias=True)
    Y = g["items0"].copy()
    X = m.recompute_factors_bias(Y, C, 0.1, cores=1)
    check_half_step("recompute_factors_bias/f9", "tcgen05", X, g["users_half1"],
                    orc.half_step_bias(g["items0"], C, 0.1, np.float64))
    assert np.all(Y[:, 0] == 1)  # the reference overwrites the caller's bias column (wmf_model.py:331)
    g2 = load_golden("weighted_nobias_f16")
    C2 = csr_from(g2, "train")
    C2.data = orc.preprocess_counts(C2.data)
    m2 = WMF(num_items=C2.shape[1], num_users=C2.shape[0], dim=16, gamma=0.1, weighted=True)
    assert row_rel_err(m2.recompute_factors(g2["items0"], C2, 0.1), g2["users_half1"]) < HALF_STEP_TOL
    assert row_rel_err(m2.recompute_factors_par(g2["items0"], C2, 0.1, cores=4), g2["users_half1"]) < HALF_STEP_TOL


def test_unweighted_vs_golden(cuda_device):
    g = load_golden("unweighted_f12")
    tr, te = csr_from(g, "train"), csr_from(g, "test")
    m = WMF(num_items=tr.shape[1], num_users=tr.shape[0], dim=12, gamma=0.1)  # weighted=None -> unweighted
    assert m.train(tr, 1, eval_mat=te, cores=1, stopping_rounds=99) == 0
    assert row_rel_err(m.users, g["users_ep1"]) < 5e-4
    assert row_rel_err(m.items, g["items_ep1"]) < 5e-4
    m = WMF(num_items=tr.shape[1], num_users=tr.shape[0], dim=12, gamma=0.1)
    assert m.train(tr, 3, eval_mat=te, cores=1, stopping_rounds=99) == int(g["train_iter"])
    assert float(m.eval_prec(te)) == pytest.approx(float(g["mse_final"]), rel=2e-3)


@pytest.mark.parametrize("dim,bias,items,rs", [(16, False, 800, 200), (12, True, 90, 60), (128, False, 3000, 1000)])
def test_eval_topn_device_equals_host_loop(cuda_device, dim, bias, items, rs):
    """SURVEY.md 8f N2: the batched device protocol (one scoring pass + wmf_rank_ahead) returns exactly what the
    reference's loop of rank calls returns (base_model.py:51-148), same RNG draws. The small-catalogue case draws
    lists with many repeated ids (90 items, 61 draws), which exercises the `item in top` duplicate rule."""
    from recmodel_b200.base_model import RecModel
    users = 400
    full = make_counts(users, items, min(users * items // 8, 30_000), seed=5, planted_rank=4)
    tr, te = split_train_test(full)
    m = WMF(num_items=items, num_users=users, dim=dim, gamma=0.1, weighted=True, bias=bias)
    m.train(tr, 2, eval_mat=te, count_mat=tr, cores=1, stopping_rounds=99)
    topn = np.array([1, 5, 20])
    dev_res = m.eval_topn(te.copy(), topn=topn, rand_sampled=rs, random_state=11)
    host_res = RecModel.eval_topn(m, te.copy(), topn=topn, rand_sampled=rs, random_state=11)
    assert dev_res.keys() == host_res.keys()
    for k in dev_res:
        assert float(dev_res[k]) == float(host_res[k]), (k, dev_res[k], host_res[k])
    # exact score ties: all-equal factors make every score equal, so only positions decide
    m.users = np.ones_like(m.users)
    m.items = np.ones_like(m.items)
    dev_res = m.eval_topn(te.copy(), topn=topn, rand_sampled=rs, random_state=12)
    host_res = RecModel.eval_topn(m, te.copy(), topn=topn, rand_sampled=rs, random_state=12)
    for k in dev_res:
        assert float(dev_res[k]) == float(host_res[k]), (k, dev_res[k], host_res[k])
    with pytest.raises(ValueError):
        m.eval_topn(te, topn=[10])


def test_coverage_and_split_mirror_reference_utils(cuda_device):
    """SURVEY.md 8f N3: utils.test_coverage batched on the device equals the reference's per-user loop, and
    train_test_split_sparse_mat keeps the reference's RNG semantics (utils.py:3-37)."""
    from recmodel_b200 import utils
    full = make_counts(700, 300, 20_000, seed=8, planted_rank=5)  # users >= items: the reference sizes the counts by users
    tr, te = utils.train_test_split_sparse_mat(full, train=0.8, seed=1993)
    np.random.seed(1993)
    mask = np.random.rand(full.nnz) < 0.8
    assert tr.nnz == int(mask.sum()) and te.nnz == full.nnz - tr.nnz and (tr + te != full).nnz == 0
    m = WMF(num_items=300, num_users=700, dim=16, gamma=0.1, weighted=True)
    m.train(tr, 2, eval_mat=te, count_mat=tr, cores=1, stopping_rounds=99)
    got = utils.test_coverage(m, tr, 10)

    class LoopOnly:  # no rank_batch: forces the reference's per-user loop through the same device rank
        def rank(self, items, users, topn=None):
            return m.rank(items, users, topn)
    ref = utils.test_coverage(LoopOnly(), tr, 10)
    np.testing.assert_array_equal(got, ref)
    assert got.shape == (700,) and got.sum() == 700 * 10


def test_recall_quality_planted_structure(cuda_device):
    """End-to-end quality: Recall@20 on a planted low-rank matrix vs the oracle trained the same
    way (north_star: within 0.005 absolute)."""
    full = make_counts(1200, 800, 60_000, seed=41, planted_rank=8)
    tr, te = split_train_test(full)
    m = WMF(num_items=800, num_users=1200, dim=16, gamma=0.1, weighted=True)
    m.train(tr, 4, eval_mat=te, count_mat=tr, cores=1, stopping_rounds=99)
    U, V, _, _ = orc.train(orc.init_items(800, 16, False), tr, 4, te, count_mat=tr, gamma=0.1, stopping_rounds=99)
    topn = np.array([20])
    ours = m.eval_topn(te.copy(), topn=topn, rand_sampled=200, cores=1, random_state=3)["Recall@20"]
    ref = orc.eval_topn(lambda it, u, k: orc.rank(U, V, it, u, k), 800, te, topn, rand_sampled=200,
                        random_state=3)["Recall@20"]
    assert ref > 0.3
    assert abs(float(ours) - float(ref)) <= 0.005


# ------------------------------------------------------------------------------- K2, dual kernel / routing
@pytest.mark.parametrize("f,bias", [(16, False), (64, False), (65, True), (128, False), (129, True), (192, False),
                                    (256, False)])
def test_half_step_dual_rows_every_length(cuda_device, f, bias):
    """Rows of every length 1 .. dual_max + 8 (the routing boundary included), a few long ones, an empty one and
    one with a stored zero weight (it must stay off the dual side, whose right-hand side divides by sqrt(d)):
    the tcgen05 pipeline (dual kernel for short rows; primal kernel or CUDA-core kernel for the rest) against the
    fp64 restatement at plain 1e-4, steady-state-like mixed-sign factors and the all-positive first-epoch kind."""
    nd = int(_lib.load().wmf_als_dual_max_entries())
    rng = np.random.default_rng(1000 + f)
    N = 1500
    lens = list(range(1, nd + 9)) + [0, 150, 400, 1100, 5]
    indptr = np.concatenate([[0], np.cumsum(lens)])
    indices = np.concatenate([np.sort(rng.choice(N, n, replace=False)) for n in lens]).astype(np.int32)
    data = orc.preprocess_counts(rng.integers(1, 6, indptr[-1]).astype(np.float32))
    data[indptr[len(lens) - 1] + 2] = 0.0  # the 5-entry row holds a zero weight
    C = scipy.sparse.csr_matrix((data, indices, indptr), shape=(len(lens), N))
    step = orc.half_step_bias if bias else orc.half_step
    for kind in ("positive", "mixed"):
        Y = rng.random((N, f)).astype(np.float32) if kind == "positive" else (rng.standard_normal((N, f)) * 0.3).astype(np.float32)
        if bias:
            Y[:, 0] = (rng.random(N) * 0.5).astype(np.float32)   # beta < d: all weights stay positive
        X, _ = run_half_step(Y, C, bias, _lib.ALGO_TCGEN05, cuda_device)
        flags, fixed = engine.half_step_status()
        assert np.all(X[np.array(lens) == 0] == 0) and np.all(np.isfinite(X))
        check_half_step(f"dual_rows/f{f}{'b' if bias else ''}/{kind}", "tcgen05", X, step(Y, C, 0.1), step(Y, C, 0.1, np.float64))
        assert (flags & 2) == 0
        # only a negative weight needs the CUDA-core kernel: with biases the stored zero becomes 0 - beta < 0
        assert fixed == (1 if bias else 0)
        X2, _ = run_half_step(Y, C, bias, _lib.ALGO_TCGEN05, cuda_device, use_row_order=False)
        np.testing.assert_array_equal(X, X2)
        Xa, _ = run_half_step(Y, C[:40], bias, _lib.ALGO_TCGEN05, cuda_device)   # row sharding never changes a row's bits
        np.testing.assert_array_equal(Xa, X[:40])


# ------------------------------------------------------------------------------- larger golden fixture, EASE (N4)
@pytest.mark.parametrize("algo_name,algo", ALGOS)
def test_half_step_vs_reference_golden_2000x1500(cuda_device, algo_name, algo):
    """The executed reference at 2000 x 1500, f = 128 (tests/golden/make_golden.py::case_half_steps): both tensor-core
    kernels (dual for the short rows, primal for the rest) against reference output, not only against the oracle."""
    g = load_golden_2000x1500()
    C = csr_from(g, "train")
    C.data = orc.preprocess_counts(C.data)
    CT = C.T.tocsr()
    X, _ = run_half_step(g["items0"], C, False, algo, cuda_device)
    rows = np.arange(0, 2000, 5)
    check_half_step("golden/2000x1500_f128/users_half1", algo_name, X[rows], g["users_half1"][rows],
                    orc.half_step(g["items0"], C[rows], 0.1, np.float64))
    Xi, _ = run_half_step(g["users_half1"], CT, False, algo, cuda_device)
    rows = g["items_half1_rows"]
    check_half_step("golden/2000x1500_f128/items_half1", algo_name, Xi[rows], g["items_half1"],
                    orc.half_step(g["users_half1"], CT[rows], 0.1, np.float64), steady=True)


def test_ease_vs_reference_golden(cuda_device):
    """N4: Ease.train / predict / rank / eval_topn on the device against the executed reference (its Cython predictor
    compiled from the reference sources when the fixture was made)."""
    from recmodel_b200.ease_model import Ease
    g = load_golden("ease_f300")
    X, te = csr_from(g, "train"), csr_from(g, "test")
    m = Ease(num_items=X.shape[1], num_users=X.shape[0])
    m.train(X.copy(), alpha=float(g["alpha"]), verbose=0, cores=1)
    W = m.W
    scale = np.abs(g["W"]).max()
    W64 = orc.ease_train(X, float(g["alpha"]), np.float64)
    err_ref, err64, noise = np.abs(W - g["W"]).max() / scale, np.abs(W - W64).max() / scale, np.abs(g["W"] - W64).max() / scale
    print(f"EASE W: vs reference {err_ref:.2e}, vs fp64 {err64:.2e}; reference vs fp64 {noise:.2e}")
    assert W.dtype == np.float32 and np.all(np.diag(W) == 0)
    assert err64 < 1e-4 and err_ref < 1e-4
    # prediction arithmetic is bit-exact given the same W
    m.W = g["W"]
    np.testing.assert_array_equal(m.predict(g["pred_users"], g["pred_items"]), g["pred"])
    for k, u in enumerate(g["rank_users"]):
        np.testing.assert_array_equal(m.rank(np.arange(X.shape[1]), int(u), 10), g["rank_top10"][k])
    rec = m.eval_topn(te.copy(), topn=g["topn"], rand_sampled=100, cores=1, random_state=7)
    np.testing.assert_allclose([rec[f"Recall@{k}"] for k in g["topn"]], g["recall"], atol=1e-12)
    assert m.predict(np.array([], dtype=np.int32), np.array([], dtype=np.int32)).shape == (1,)


def test_bench_dump_outputs_reproducible(cuda_device, tmp_path):
    """bench.py --dump-outputs: the factors of the last timed epoch, identical from run to run (the end-to-end leg
    that follows leaves them alone), and --steps sets the number of timed steps of both legs."""
    import json
    import os
    import subprocess
    import sys
    dumps = []
    for k, extra in enumerate((["--steps", "3"], ["--steps", "3", "--no-e2e"])):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "ml1m",
                              "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(k)), *extra],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
        assert len(lines) == 1, lines
        d = json.loads(lines[0])
        assert d["steps"] == 3 and d["value"] > 0
        if k == 0:
            assert len(d["e2e"]["ms_steps_rank0"]) == 3
        dumps.append({n: np.load(tmp_path / str(k) / f"{n}.npy") for n in ("users", "items")})
    for n, shape in (("users", (6040, 64)), ("items", (3706, 64))):
        a, b = dumps[0][n], dumps[1][n]
        assert a.dtype == np.float32 and a.shape == shape and np.all(np.isfinite(a)) and np.any(a != 0)
        np.testing.assert_array_equal(a, b)


def test_ease_larger_matrix_against_fp64(cuda_device):
    """A catalogue that spans many panels of the blocked inverse (1 100 items, not a multiple of the 64-wide panel)."""
    from recmodel_b200.ease_model import Ease
    X = make_counts(3000, 1100, 90_000, seed=3, planted_rank=6)
    m = Ease(num_items=1100, num_users=3000)
    m.train(X, alpha=100.0, verbose=0, cores=1)
    W64 = orc.ease_train(X, 100.0, np.float64)
    W32 = orc.ease_train(X, 100.0)
    scale = np.abs(W64).max()
    err, noise = np.abs(m.W - W64).max() / scale, np.abs(W32 - W64).max() / scale
    print(f"EASE 1100 items: gpu vs fp64 {err:.2e}; numpy fp32 vs fp64 {noise:.2e}")
    assert err < max(1e-4, 3 * noise)
