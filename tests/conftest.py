import hashlib
import os
import sys

import numpy as np
import pytest
import scipy.sparse

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


# ---- parity ledger: every half-step comparison of the GPU run is recorded and written to
# gpurun_out/r02_parity.json at session end (copied to profiles/ from the B200 run)
PARITY_LEDGER = []


def ledger_add(case, algo, **fields):
    rec = {"case": case, "algo": algo}
    rec.update({k: (float(v) if v is not None else None) for k, v in fields.items()})
    PARITY_LEDGER.append(rec)


def pytest_sessionfinish(session, exitstatus):
    if not PARITY_LEDGER:
        return
    import json
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, os.environ.get("WMF_LEDGER_NAME", "r02_parity.json")), "w") as fh:
        json.dump({"bar": 1e-4, "measure": "max over rows of ||x - ref|| / ||ref||", "records": PARITY_LEDGER}, fh, indent=1)


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    return {k: z[k] for k in z.files}


def array_digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def load_golden_2000x1500():
    """The reference's two half-steps at 2000 x 1500, f = 128 (tests/golden/make_golden.py::case_half_steps) in the
    layout of load_golden(). Only the reference's outputs are stored, to keep the files small: the user half-step in
    full (the item half-step's input) and the item half-step on the rows in ``items_half1_rows``. The inputs are
    regenerated from their seeds and checked against digests of what the reference was given."""
    from oracle.wmf_oracle import init_items
    from recmodel_b200.synthetic import make_counts
    g = load_golden("weighted_nobias_f128_2000x1500")
    g.update(load_golden("weighted_nobias_f128_2000x1500_items"))
    C = make_counts(2000, 1500, 150_000, seed=18, planted_rank=8)
    g.update(train_indptr=C.indptr.astype(np.int64), train_indices=C.indices.astype(np.int32),
             train_data=C.data.astype(np.float32), train_shape=np.array(C.shape, dtype=np.int64))
    g["items0"] = init_items(1500, 128, False, seed=1993)
    assert array_digest(g["train_indptr"], g["train_indices"], g["train_data"]) == str(g["train_sha256"]), \
        "recmodel_b200.synthetic.make_counts no longer generates the matrix the reference was given"
    assert array_digest(g["items0"]) == str(g["items0_sha256"]), \
        "oracle.wmf_oracle.init_items no longer generates the factors the reference was given"
    return g


def csr_from(g, prefix):
    shape = tuple(int(x) for x in g[f"{prefix}_shape"])
    nnz = len(g[f"{prefix}_data"])
    ptr_t = np.int32 if nnz < 2**31 - 1 else np.int64
    return scipy.sparse.csr_matrix((g[f"{prefix}_data"], g[f"{prefix}_indices"], g[f"{prefix}_indptr"].astype(ptr_t)),
                                   shape=shape)


def row_rel_err(a, b):
    """max over rows of ||a_r - b_r|| / max(||b_r||, tiny): the per-half-step parity measure."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    num = np.linalg.norm(a - b, axis=1)
    den = np.maximum(np.linalg.norm(b, axis=1), 1e-30)
    zero = np.linalg.norm(b, axis=1) == 0
    return float(np.max(np.where(zero, np.linalg.norm(a, axis=1), num / den))) if len(a) else 0.0


WEIGHTED_CASES = [
    ("weighted_nobias_f16", 16, False, "log"),
    ("weighted_bias_f8", 8, True, "log"),
    ("weighted_nobias_f64_linear", 64, False, "linear"),
    ("weighted_bias_f64", 64, True, "log"),
    ("weighted_nobias_f128", 128, False, "log"),
]


@pytest.fixture(scope="session")
def cuda_device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")
