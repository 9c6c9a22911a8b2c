"""Host-side logic: constructor parity with the reference, row partitioning, the gloo
world_size=2 exchange, the synthetic generator and the split. CPU only."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse

from conftest import ROOT, load_golden
from recmodel_b200 import WMF, WMFModel, sharding, train_test_split_sparse_mat
from recmodel_b200.synthetic import make_counts


def test_constructor_matches_reference_init():
    g = load_golden("weighted_bias_f8")
    m = WMF(num_items=g["items0"].shape[0], num_users=int(g["train_shape"][0]), dim=8, gamma=0.1, weighted=True,
            bias=True, seed=1993)
    np.testing.assert_array_equal(m.items, g["items0"])
    assert m.users is None and m.dim == 8 and m.gamma == 0.1 and m.weighted is True and m.dtype == "float32"
    assert WMFModel is WMF
    with pytest.raises(ValueError):
        WMF(5, 4, 3, 0.1, dtype="float64")


def test_synthetic_generator_is_deterministic_and_canonical():
    a = make_counts(300, 200, 5000, seed=3)
    b = make_counts(300, 200, 5000, seed=3)
    assert a.nnz == 5000 and (a != b).nnz == 0
    assert a.has_sorted_indices
    for r in range(a.shape[0]):
        idx = a.indices[a.indptr[r]:a.indptr[r + 1]]
        assert np.all(np.diff(idx) > 0)
    assert a.data.dtype == np.float32 and a.data.min() >= 1 and a.data.max() <= 5


def test_split_keeps_reference_rng_semantics():
    m = make_counts(200, 150, 4000, seed=4)
    tr, te = train_test_split_sparse_mat(m, train=0.8, seed=1993)
    assert tr.nnz + te.nnz == m.nnz and (tr.multiply(te)).nnz == 0
    np.random.seed(1993)
    mask = np.random.rand(m.nnz) < 0.8
    assert tr.nnz == int(mask.sum())
    assert m.nnz == 4000  # the input is not zeroed (SURVEY.md §4 item 3)


def test_balanced_row_partition_properties():
    rng = np.random.default_rng(0)
    counts = (rng.pareto(1.2, size=5000) * 20).astype(np.int64)
    for world in (1, 2, 4, 8):
        b = sharding.balanced_row_partition(counts, world, 128)
        assert len(b) == world + 1 and b[0] == 0 and b[-1] == len(counts) and np.all(np.diff(b) >= 0)
        cost = sharding.row_costs(counts, 128)
        per = np.array([cost[b[g]:b[g + 1]].sum() for g in range(world)])
        assert per.max() <= cost.sum() / world + cost.max() + 1e-6
    assert list(sharding.balanced_row_partition(np.zeros(0), 4, 16)) == [0, 0, 0, 0, 0]
    # aligned to the Gram block height (sharding.sharded_gram): inner boundaries are whole blocks
    for world in (2, 3, 8):
        b = sharding.balanced_row_partition(counts, world, 128, align=32)
        assert b[0] == 0 and b[-1] == len(counts) and np.all(np.diff(b) >= 0) and np.all(b[:-1] % 32 == 0)
        per = np.array([cost[b[g]:b[g + 1]].sum() for g in range(world)])
        assert per.max() <= cost.sum() / world + 2 * cost.max() + np.sort(cost)[-32:].sum()


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
from recmodel_b200 import sharding
from oracle import wmf_oracle as orc
from recmodel_b200.synthetic import make_counts
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank, world = sharding.dist_info()
C = make_counts(90, 60, 1500, seed=9); C.data = orc.preprocess_counts(C.data)
CT = C.T.tocsr()
Y = orc.init_items(60, 8, False)
ub = sharding.balanced_row_partition(np.diff(C.indptr), world, 8)
ib = sharding.balanced_row_partition(np.diff(CT.indptr), world, 8)
# each rank solves only its rows (the oracle stands in for the kernel on CPU), then all-gather
Xl = orc.half_step(Y, C[ub[rank]:ub[rank+1]], 0.1)
users = sharding.all_gather_rows(torch.from_numpy(Xl), ub).numpy()
Il = orc.half_step(users, CT[ib[rank]:ib[rank+1]], 0.1)
items = sharding.all_gather_rows(torch.from_numpy(Il), ib).numpy()
ref_u = orc.half_step(Y, C, 0.1); ref_i = orc.half_step(ref_u, CT, 0.1)
assert np.array_equal(users, ref_u) and np.array_equal(items, ref_i), "sharded != single"
# Gram of the new factors from block partials: each rank fills the blocks of its own rows (NumPy stands in
# for wmf_gram_partials), zeros elsewhere, one sum all-reduce, blocks added in block order
from recmodel_b200 import engine
B = engine.gram_block_rows(90)
ub2 = sharding.balanced_row_partition(np.diff(C.indptr), world, 8, align=B)
assert all(int(b) % B == 0 for b in ub2[:-1])
nb = -(-90 // B)
def block(b, X):
    Xb = X[b * B:(b + 1) * B].astype(np.float64)
    return Xb.T @ Xb
part = torch.zeros((nb, 8, 8), dtype=torch.float64)
for b in range(int(ub2[rank]) // B, -(-int(ub2[rank + 1]) // B)):
    part[b] = torch.from_numpy(block(b, ref_u))
sharding.all_reduce_sum_(part)
single = np.zeros((8, 8)); summed = np.zeros((8, 8))
for b in range(nb):
    single = single + block(b, ref_u); summed = summed + part[b].numpy()
assert np.array_equal(single, summed), "block partial exchange changed the Gram"
# peer-memory exchange is a GPU feature: on CPU / gloo the buffers are unavailable and callers take the collective path
assert sharding.PeerBuffers.create(90, 60, 8, torch.device("cpu")) is None
s = torch.tensor([1.0 + rank, 2.0, 3.0], dtype=torch.float64)
sharding.all_reduce_sum_(s)
assert s.tolist() == [3.0, 4.0, 6.0]
dist.destroy_process_group()
print("ok", rank)
"""


def test_two_rank_gloo_sharded_epoch_equals_single(tmp_path):
    port = 29500 + (os.getpid() % 2000)
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                              text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"ok {r}" in o, o


def test_utils_mirror_reference_semantics():
    """recmodel_b200.utils (SURVEY.md 8f N3) on the host: the split keeps the reference's RNG semantics
    (utils.py:21-27) and test_coverage's per-user loop counts what the reference's loop counts (utils.py:3-18),
    checked with a model whose rank is a fixed score table."""
    from recmodel_b200 import utils
    full = make_counts(60, 40, 600, seed=3)
    tr, te = utils.train_test_split_sparse_mat(full, train=0.8, seed=1993)
    np.random.seed(1993)
    mask = np.random.rand(full.nnz) < 0.8
    assert tr.nnz == int(mask.sum()) and te.nnz == full.nnz - tr.nnz and (tr + te != full).nnz == 0
    assert full.nnz == 600  # the input is left alone

    scores = np.random.default_rng(0).random((60, 40))

    class Table:
        def rank(self, items, users, topn=None):
            items = np.asarray(items)
            order = np.argsort(-scores[users, items], kind="stable")
            return items[order][:topn]

    got = utils.test_coverage(Table(), tr, 5)
    want = np.zeros(60, dtype=np.int32)  # the reference sizes the counts by the number of users
    for u in range(60):
        seen = tr.indices[tr.indptr[u]:tr.indptr[u + 1]]
        cand = np.delete(np.arange(40), seen)
        want[cand[np.argsort(-scores[u, cand], kind="stable")][:5]] += 1
    np.testing.assert_array_equal(got, want)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) needs no GPU and prints exactly one JSON
    line with the contract's keys: same metric / unit / config as our arm, `impl`, a `cpu_baseline` that describes
    the run and an `e2e` object without copies."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "ml1m",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "wmf_nnz_updates_per_sec_per_epoch" and d["unit"] == "nnz-updates/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("WMF weighted ALS epoch, 6040x3706") and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["gpu_launches"] == 0


def test_bench_rejects_bad_step_counts_and_reference_dumps():
    """Argument errors end the bench before any work (exit status 2, no result line)."""
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "ml1m", *extra],
                             capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr)


def test_bench_dump_outputs_stays_within_budget(tmp_path):
    """bench.py --dump-outputs: an output larger than its share of the budget keeps a fixed, ascending sample of its
    rows (the same on every call); smaller outputs are written whole."""
    import bench
    big = np.arange(70_000 * 128, dtype=np.float32).reshape(70_000, 128)   # 35.8 MB, over its half of the budget
    small = np.random.default_rng(1).random((300, 128)).astype(np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"users": big, "items": small})
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == ["items.npy", "users.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES
    u = np.load(tmp_path / "a" / "users.npy")
    assert u.dtype == np.float32 and u.shape[1] == 128 and 60_000 < u.shape[0] < 70_000
    assert np.all(np.diff(u[:, 0]) > 0)   # distinct rows in ascending order
    np.testing.assert_array_equal(u, big[(u[:, 0] / 128).astype(np.int64)])
    np.testing.assert_array_equal(u, np.load(tmp_path / "b" / "users.npy"))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "items.npy"), small)
