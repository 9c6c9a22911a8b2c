"""Dual kernel packs: up to four short rows share one solver group's accumulator on its block diagonal. A row's
result must not depend on its partners: every row of a packed half-step equals, bit for bit, the same row solved
alone, and stays within the 1e-4 bar of the fp64 restatement."""
import numpy as np
import pytest
import scipy.sparse
import torch

from conftest import row_rel_err
from oracle import wmf_oracle as orc
from recmodel_b200 import _lib, engine
from recmodel_b200.engine import DeviceCSR

pytestmark = pytest.mark.gpu

N_ITEMS = 500
# 1, 2 and 3 slices of 32 TMEM lanes (n rounded up to 16), both sides of every slice boundary
BASE_LENS = [1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 95, 96]
WIDE_LENS = [97, 112, 127, 128]   # 4 slices: the dual kernel takes up to 128 entries above f = 128
SHORT = BASE_LENS * 2 + [1, 8, 20, 30, 9, 24, 3, 31, 12]
# (rows, pack shapes they make). Between them every shape occurs: an odd 2-slice row with 2, 1 and 0 spare 1-slice
# rows, 3-slice rows with and without a partner, full and partial fours of 1-slice rows ({4} at f > 128).
MIXES = {
    "short": (SHORT, {"3,1", "2,2", "1,1,1,1", "1,1,1"}),
    "short_odd2": (SHORT + [40], {"3,1", "2,2", "2,1,1", "1,1,1,1", "1"}),
    "balanced_odd2": (BASE_LENS + [70, 80], {"3,1", "2,2", "2,1"}),
    "long_odd2": (BASE_LENS + [65, 70, 80, 90, 96] * 3 + [40, 48, 50, 56], {"3,1", "3", "2,2", "2"}),
}


def pack_shapes(lens):
    """The slice counts of the packs tc_pack_dual_kernel makes of these rows (restated to check the mixes above)."""
    c = [sum(1 for n in lens if (n + 31) // 32 == k) for k in (1, 2, 3, 4)]
    m31 = min(c[0], c[2])
    shapes = ["4"] * c[3] + ["3,1"] * m31 + ["3"] * (c[2] - m31) + ["2,2"] * (c[1] // 2)
    r1 = c[0] - m31
    if c[1] % 2:
        m21 = min(r1, 2)
        shapes.append("2" + ",1" * m21)
        r1 -= m21
    shapes += ["1,1,1,1"] * (r1 // 4) + ([",".join(["1"] * (r1 % 4))] if r1 % 4 else [])
    return set(shapes)


def matrix(lens, rng, weights=None):
    lens = list(lens)
    rng.shuffle(lens)
    indptr = np.concatenate([[0], np.cumsum(lens)])
    indices = np.concatenate([np.sort(rng.choice(N_ITEMS, n, replace=False)) for n in lens]).astype(np.int32)
    data = orc.preprocess_counts(rng.integers(1, 6, indptr[-1]).astype(np.float32)) if weights is None else weights(indptr)
    return scipy.sparse.csr_matrix((data, indices, indptr), shape=(len(lens), N_ITEMS))


def factors(f, bias, rng):
    Y = (rng.standard_normal((N_ITEMS, f)) * 0.3).astype(np.float32)
    if bias:
        Y[:, 0] = (rng.random(N_ITEMS) * 0.5).astype(np.float32)   # beta < d: every weight stays positive (dual side)
    return Y


def half_step(Y, C, bias, cuda_device):
    Yd = torch.from_numpy(Y).to(cuda_device)
    G = engine.gram(Yd, 0.1, ones_col0=bias)
    X = engine.half_step(DeviceCSR.from_scipy(C, cuda_device), Yd, G, bias=bias, algo=_lib.ALGO_TCGEN05)
    torch.cuda.synchronize()
    return X.cpu().numpy()


def solo(Y, C, bias, cuda_device):
    """Each row of C solved alone (a one-row slice: a pack of its own)."""
    return np.concatenate([half_step(Y, C[i:i + 1], bias, cuda_device) for i in range(C.shape[0])])


@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("f", [16, 64, 128, 256])
@pytest.mark.parametrize("mix", sorted(MIXES))
def test_packed_rows_equal_solo_rows(cuda_device, f, bias, mix):
    """Every mix after every other one in the same process: the pack table is not cleared between calls, so an entry
    left from an earlier, larger call would show up here as a wrong or extra row."""
    rng = np.random.default_rng(f + 7 * bias + 100 * sorted(MIXES).index(mix))
    lens, shapes = MIXES[mix]
    lens = lens + (WIDE_LENS * 2 if f > 128 else [])
    assert pack_shapes(lens) == (shapes | {"4"} if f > 128 else shapes)
    assert max(lens) <= int(_lib.load().wmf_als_dual_max_entries()) or f > 128   # every row is a dual row
    C = matrix(lens, rng)
    Y = factors(f, bias, rng)
    X = half_step(Y, C, bias, cuda_device)
    flags, fixed = engine.half_step_status()
    assert flags & 2 == 0 and fixed == 0 and not engine.half_step_used_fallback()
    np.testing.assert_array_equal(X, solo(Y, C, bias, cuda_device))
    step = orc.half_step_bias if bias else orc.half_step
    err = row_rel_err(X, step(Y, C, 0.1, np.float64))
    print(f"packed dual rows f={f} bias={bias} {mix}: vs fp64 {err:.2e}")
    assert err < 1e-4


@pytest.mark.parametrize("f", [128, 256])
def test_heavy_row_falls_back_inside_its_pack(cuda_device, f):
    """A row with weights spread over four decades (up to 2e4) does not converge within the conjugate-gradient budget
    and is factorised in tensor memory at its own lanes and columns; the other systems of its pack keep their solo
    bits. (Its n x n system has rank n <= f: at smaller f, CG would converge in at most f + 1 products.)"""
    rng = np.random.default_rng(31 + f)
    lens = [96, 20, 40, 44, 10, 12, 14, 16, 90, 30]   # the heavy 96-entry row shares a pack with a 1-slice row
    heavy = {}

    def weights(indptr):
        d = orc.preprocess_counts(rng.integers(1, 6, indptr[-1]).astype(np.float32))
        k = int(np.argmax(np.diff(indptr) == 96))
        heavy["row"] = k
        lo, hi = indptr[k], indptr[k + 1]
        d[lo:hi] = np.exp(rng.uniform(0.0, np.log(2e4), hi - lo)).astype(np.float32)
        return d

    C = matrix(lens, np.random.default_rng(5), weights)
    k = heavy["row"]
    Y = factors(f, False, rng)
    X = half_step(Y, C, False, cuda_device)
    assert engine.half_step_used_fallback(), "the heavy row did not take the factorisation"
    Xs = solo(Y, C, False, cuda_device)
    others = np.arange(C.shape[0]) != k
    np.testing.assert_array_equal(X[others], Xs[others])
    np.testing.assert_array_equal(X[k], Xs[k])
    ref = orc.half_step(Y, C, 0.1)
    x64 = orc.half_step(Y, C, 0.1, np.float64)
    tol = max(1e-4, 2.0 * row_rel_err(ref, x64))   # the bar of test_half_step_cg_falls_back_to_factorisation
    err = row_rel_err(X, x64)
    print(f"heavy row f={f}: vs fp64 {err:.2e} (tol {tol:.1e})")
    assert np.all(np.isfinite(X)) and err < tol
