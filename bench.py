#!/usr/bin/env python
"""bench.py - WMF nnz-updates/s per epoch (BASELINE.json's metric), default workload ML-20M shape (config 2).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU arithmetic (oracle port)
    python bench.py --workload netflix|powerlaw256|rank ...   # BASELINE.json configs 3, 4 (scaled) and 5
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/*.npy

A "step" is one ALS epoch (user half-step + item half-step, each with its Gram) over a synthetic count matrix,
weighted, log preprocessing; metric = 2*nnz / t_epoch. `value` is measured with the matrices resident in HBM;
`e2e` is the same metric through the public `WMF.train` call with HOST (SciPy/NumPy) buffers, so it pays the H2D
upload, the device transpose, the epoch, the fused eval and the D2H read-back of the factors every step. Under
torchrun the rows are partitioned across the ranks (strong scaling: same matrix at every N) and factor shards are
exchanged after every half-step. Workload `rank` (config 5) times top-100 ranking of every user instead
(metric users/s, tensor roofline).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True   # the bench writes nothing into the source tree, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: users, items, nnz, dim, where the matrix is generated, BASELINE.json config
    "ml20m": (138_493, 26_744, 20_000_000, 128, "host", "configs[1]: ML-20M shape"),
    "netflix": (480_189, 17_770, 100_000_000, 128, "device", "configs[2]: Netflix shape"),
    "powerlaw256": (1_000_000, 100_000, 100_000_000, 256, "device",
                    "configs[3] at 1/10 of every dimension (the 10 M x 1 M, 1 B-entry matrix needs 8 GPUs)"),
    "powerlaw1b": (10_000_000, 1_000_000, 1_000_000_000, 256, "device",
                   "configs[3]: power-law 10 M x 1 M, 1 B entries, dim 256 (row-sharded; needs several GPUs)"),
    "rank": (138_493, 26_744, 20_000_000, 128, "host", "configs[4]: top-100 for all users, ML-20M shape"),
    "ml1m": (6040, 3706, 1_000_000, 64, "host", "debugging only; never the reported config"),
}
GAMMA, ALPHA, BETA = 0.1, 10, 1
L2_NOTE = "inputs larger than L2, no flush (CSR + transpose + factors streamed every epoch)"
DUMP_BYTES = 64_000_000   # --dump-outputs writes at most this much in all


def dump_outputs(dirname, arrays):
    """Write each float32 array as <dirname>/<name>.npy. An array larger than its equal share of DUMP_BYTES keeps a
    fixed sample of its rows (seed 0, ascending), the same rows for the same workload on every run and build."""
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096   # room for the .npy header
    for name, a in arrays.items():
        if a.nbytes > share:
            keep = share // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_config(name):
    """The `config` object both arms print (identical keys and values for one workload)."""
    users, items, nnz, dim, _, what = WORKLOADS[name]
    return {"workload": f"WMF weighted ALS epoch, {users}x{items}, {nnz} nnz, dim {dim}, log preprocessing "
                        f"(BASELINE.json {what})" if name != "rank" else
                        f"top-100 ranking of all {users} users over {items} items, dim {dim} (BASELINE.json {what})",
            "users": users, "items": items, "nnz": nnz, "dim": dim, "weighted": True, "bias": False,
            "preprocess": "log", "gamma": GAMMA, "l2": L2_NOTE}


def source_hash():
    """Hash of the CUDA sources the library is built from (ties a committed ncu capture to the code it measured)."""
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "recmodel_b200", "csrc")
    for fn in sorted(os.listdir(csrc)):
        if fn.endswith((".cu", ".cuh")):
            with open(os.path.join(csrc, fn), "rb") as fh:
                h.update(fn.encode() + b"\0" + fh.read())
    return h.hexdigest()[:16]


def load_traffic():
    """DRAM bytes (read + write) of the half-step kernels of one epoch from the committed `ncu --set full` capture,
    or None when the capture was taken from other sources than the ones this library is built from."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    try:
        with open(path) as fh:
            t = json.load(fh)
        if t.get("source_hash") != source_hash():
            return None, f"capture {t.get('source_hash')} does not match the built sources {source_hash()}"
        return float(t["epoch_dram_bytes"]), "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum, profiles/r02_ncu_traffic.json"
    except Exception:
        return None, "no capture"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as fh:
                p = json.load(fh)
            return p, "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synth_host(workload):
    from recmodel_b200.synthetic import make_counts_cached
    users, items, nnz, dim = WORKLOADS[workload][:4]
    return make_counts_cached(users, items, nnz), dim


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's arithmetic (oracle port, NumPy + BLAS + LAPACK, all host threads)
# --------------------------------------------------------------------------------------------
def cpu_epoch_sample(C, CT, dim, frac, threads, seed=0, eval_mat=None):
    """Time the oracle's two half-steps (and its eval_prec, as the reference's epoch does at wmf_model.py:163) on a
    RANDOM row sample (fixed seed) holding ~frac of the rows of either side; extrapolate linearly in rows to one
    epoch. Returns (nnz-updates/s, seconds per epoch, description)."""
    from oracle import wmf_oracle as orc
    try:
        from threadpoolctl import threadpool_limits
    except Exception:  # pragma: no cover
        threadpool_limits = None
    users, items = C.shape
    rng = np.random.default_rng(seed)
    nu, ni = max(1, int(users * frac)), max(1, int(items * frac))
    su = np.sort(rng.choice(users, nu, replace=False))
    si = np.sort(rng.choice(items, ni, replace=False))
    Y = orc.init_items(items, dim, False)
    Cs, CTs = C[su], CT[si]
    ctx = threadpool_limits(limits=threads) if threadpool_limits else None
    try:
        t0 = time.perf_counter()
        Xu = orc.half_step(Y, Cs, GAMMA)
        t_u = time.perf_counter() - t0
        # item side needs user factors for all users: reuse the sample's rows cyclically (same cost)
        Ufull = np.resize(Xu, (users, dim)).astype(np.float32, copy=False)
        t0 = time.perf_counter()
        Xi = orc.half_step(Ufull, CTs, GAMMA)
        t_i = time.perf_counter() - t0
        t_e = 0.0
        if eval_mat is not None:  # eval_prec over the evaluation matrix (base_model.py:150-179), timed in full
            Ifull = np.resize(Xi, (items, dim)).astype(np.float32, copy=False)
            t0 = time.perf_counter()
            orc.eval_prec(Ufull, Ifull, eval_mat, False)
            t_e = time.perf_counter() - t0
    finally:
        if ctx is not None:
            ctx.__exit__(None, None, None)
    t_epoch = t_u * users / nu + t_i * items / ni + t_e
    desc = (f"oracle port (NumPy/BLAS/LAPACK per-row loop of wmf_model.py:213-240), extrapolated: {nu} of {users} user "
            f"rows (random, seed {seed}) in {t_u:.2f}s + {ni} of {items} item rows in {t_i:.2f}s, scaled linearly in rows"
            + (f", + eval_prec over {eval_mat.nnz} held-out entries in {t_e:.2f}s (not scaled)" if eval_mat is not None else ""))
    return 2.0 * C.nnz / t_epoch, t_epoch, desc


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return  # under torchrun only rank 0 measures the CPU arm
    from oracle import wmf_oracle as orc
    from recmodel_b200.synthetic import split_train_test
    if WORKLOADS[args.workload][4] != "host" or args.workload == "rank":
        print(json.dumps({"impl": "reference", "unavailable": f"workload {args.workload} has no CPU arm (matrix generated "
                                                              "on the device / ranking-only workload)"}), flush=True)
        return
    C, dim = synth_host(args.workload)
    tr, te = split_train_test(C, train=0.8, seed=1993)
    C = C.copy()
    C.data = orc.preprocess_counts(C.data, "log", ALPHA, BETA)
    CT = C.T.tocsr()
    threads = os.cpu_count() or 1
    frac = args.cpu_frac if args.cpu_frac else 0.1  # ~10 % of the rows each way: a few seconds of CPU work per step
    for _ in range(args.warmup):
        cpu_epoch_sample(C, CT, dim, frac / 4, threads)
    t_eps, desc = [], ""
    for k in range(args.steps):
        _, t_ep, desc = cpu_epoch_sample(C, CT, dim, frac, threads, seed=k, eval_mat=te)
        t_eps.append(t_ep)
    value = 2.0 * C.nnz / float(np.mean(t_eps))  # consistent with ms_per_step
    line = {
        "impl": "reference", "metric": "wmf_nnz_updates_per_sec_per_epoch", "value": value, "unit": "nnz-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(t_eps)) * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload),
        "run": {"impl": "oracle port of the reference's NumPy path (the Python reference cannot travel to the GPU box)",
                "extrapolated": True, "host_threads": threads},
        "cpu_baseline": {"value": value, "unit": "nnz-updates/s", "cores": threads, "kind": "port", "sample": desc,
                         "extrapolated": True},
        "e2e": {"value": value, "unit": "nnz-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def pin_csr(m):
    """The same scipy CSR matrix with its three arrays in page-locked host memory (NumPy views of pinned torch
    tensors): WMF.train then DMAs straight out of them instead of staging a copy."""
    import scipy.sparse
    import torch

    def pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    out = scipy.sparse.csr_matrix((pin(m.data), pin(m.indices), pin(m.indptr)), shape=m.shape, copy=False)
    out.has_sorted_indices = m.has_sorted_indices
    return out


def make_device_matrix(workload, device):
    """(DeviceCSR of raw counts, host CSR or None). Host-generated workloads are uploaded; the large ones are
    generated on the device with the same recipe."""
    from recmodel_b200.engine import DeviceCSR
    users, items, nnz, dim, where, _ = WORKLOADS[workload]
    if where == "host":
        C_host, _ = synth_host(workload)
        return DeviceCSR.from_scipy(C_host, device), C_host
    from recmodel_b200.synthetic import make_counts_device
    indptr, cols, data = make_counts_device(users, items, nnz, device)
    return DeviceCSR(indptr, cols, data, (users, items)), None


def run_rank(args, device, world, rank):
    """Config 5: top-100 for every user over all items (wmf_model.py:25-47), tcgen05 candidate GEMM + exact rescoring."""
    import torch
    import torch.distributed as dist
    from recmodel_b200 import WMF
    from oracle import wmf_oracle as orc
    users, items, _, dim = WORKLOADS["rank"][:4]
    m = WMF(num_items=items, num_users=users, dim=dim, gamma=GAMMA, weighted=True, bias=False, device=device)
    rng = np.random.default_rng(5)
    m.users = (rng.standard_normal((users, dim)) * 0.3).astype(np.float32)
    m.items = orc.init_items(items, dim, False)
    per = -(-users // world)
    mine = np.arange(rank * per, min(users, (rank + 1) * per), dtype=np.int64)
    cand = np.arange(items)
    from recmodel_b200 import engine
    users_d = torch.from_numpy(mine).to(device)
    cand_d = torch.from_numpy(cand.astype(np.int64)).to(device)
    U, V = m.users_device, m.items_device
    for _ in range(args.warmup):
        engine.score_topk(users_d, cand_d, U, V, 100)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    sampler = ClockSampler(device.index)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        ids = engine.score_topk(users_d, cand_d, U, V, 100)
    e1.record()
    torch.cuda.synchronize(device)
    # the last step's top-100 item ids of this rank's users (ids below 2**24 are exact in float32)
    outputs = {"topk_ids": ids.float().cpu().numpy()} if args.dump_outputs and rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    # e2e: the public rank_batch call with host arrays in and out
    t0 = time.perf_counter()
    out = m.rank_batch(cand, mine, 100)
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    if rank == 0:
        peaks, kind = load_peaks()
        ms_v = float(ms.item())
        flops = 2.0 * users * items * dim          # the score matrix once (SURVEY.md 8d); the kernel runs the GEMM twice
        line = {"metric": "wmf_rank_users_per_sec", "value": users / (ms_v * 1e-3), "unit": "users/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_v, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16 candidates + f32 exact rescoring", "data": "synthetic",
                "config": workload_config("rank"),
                "run": {"parallelism": f"users split x{world}" if world > 1 else "single GPU", "topn": 100},
                "roofline": {"bound": "tensor", "achieved": flops / (ms_v * 1e-3) / 1e12,
                             "peak": float(peaks["bf16_tflops_sustained"]), "unit": "TFLOP/s",
                             "frac": flops / (ms_v * 1e-3) / 1e12 / float(peaks["bf16_tflops_sustained"]), "traffic": None,
                             "peak_kind": kind + " (sustained bf16; fp16 runs at the same rate)",
                             "note": "algorithmic flops 2*U*I*f; the kernel computes the score tiles twice (pass 1: "
                                     "block maxima, pass 2: candidates), so the tensor pipe does twice this work"},
                "cpu_baseline": None,
                "e2e": {"value": users / float(t_e2e.item()), "unit": "users/s", "h2d_bytes_per_step": int(mine.nbytes + cand.nbytes),
                        "d2h_bytes_per_step": int(out.nbytes), "ms_per_step": float(t_e2e.item()) * 1e3,
                        "what": "WMF.rank_batch(all items, this rank's users, 100) with host arrays"},
                "gpu_launches": None, "clocks": clocks}
        print(json.dumps(line), flush=True)
        if outputs:
            dump_outputs(args.dump_outputs, outputs)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from recmodel_b200 import WMF, _lib, engine, sharding
    from recmodel_b200.synthetic import split_train_test

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    _lib.require_device()
    if args.workload == "rank":
        run_rank(args, device, world, rank)
        finish(world, device)
        return
    algo = {"auto": _lib.ALGO_AUTO, "simt": _lib.ALGO_SIMT, "tcgen05": _lib.ALGO_TCGEN05,
            "tcgen05_direct": _lib.ALGO_TCGEN05_DIRECT}[args.algo]
    users, items, _, dim, where, _ = WORKLOADS[args.workload]
    f = dim

    # synthetic data: rank 0 generates host matrices (cached on disk), the others wait and load the cache
    if where == "host" and rank == 0:
        synth_host(args.workload)
    if world > 1:
        dist.barrier()
    C_full, C_host = make_device_matrix(args.workload, device)
    nnz = C_full.nnz

    # ---- resident setup (not timed): preprocess, transpose, shard
    raw_counts = C_full.data.clone() if C_host is None else None
    engine.preprocess_(C_full.data, "log", ALPHA, BETA)
    CT_full = C_full.transpose()
    if world > 1:
        ucounts = (C_full.indptr[1:] - C_full.indptr[:-1]).cpu().numpy()
        icounts = (CT_full.indptr[1:] - CT_full.indptr[:-1]).cpu().numpy()
        ub = sharding.balanced_row_partition(ucounts, world, f, align=engine.gram_block_rows(users))
        ib = sharding.balanced_row_partition(icounts, world, f, align=engine.gram_block_rows(items))
        C = C_full.row_slice(int(ub[rank]), int(ub[rank + 1]))
        CT = CT_full.row_slice(int(ib[rank]), int(ib[rank + 1]))
    else:
        ub = ib = None
        C, CT = C_full, CT_full
    C.row_order, CT.row_order  # noqa: B018
    # the model's own initialisation (wmf_model.py:11-17, bit-reproduced on the host)
    model = WMF(num_items=items, num_users=users, dim=dim, gamma=GAMMA, weighted=True, bias=False, device=device,
                algo=args.algo)
    items_d = model.items_device.clone()
    from recmodel_b200.epoch import ResidentEpoch
    launch_mode = "python" if args.no_graphs else "4 CUDA graphs per epoch"
    try:
        loop = ResidentEpoch(C, CT, items_d, GAMMA, bias=False, algo=algo, ub=ub, ib=ib, graphs=not args.no_graphs)
    except Exception as exc:  # graph capture refused (driver / NCCL combination): same launches issued from Python
        if args.no_graphs:
            raise
        print(f"[bench] CUDA graph capture failed ({type(exc).__name__}: {exc}); launching the epoch from Python",
              file=sys.stderr, flush=True)
        torch.cuda.synchronize(device)
        launch_mode = "python (graph capture failed)"
        loop = ResidentEpoch(C, CT, items_d, GAMMA, bias=False, algo=algo, ub=ub, ib=ib, graphs=False)
    ev_pairs = []

    def epoch(record=False):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if record else None
        loop.step(e)
        if record:
            ev_pairs.append(e)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for _ in range(args.warmup):
        epoch()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        epoch(record=True)
    stop.record()
    sync_all()
    # the factors the last epoch left (full matrices on every rank), before the legs below run anything else
    outputs = {"users": loop.users.cpu().numpy(), "items": loop.items.cpu().numpy()} if args.dump_outputs and rank == 0 else None
    elapsed_ms = torch.tensor([start.elapsed_time(stop)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = float(elapsed_ms.item()) / args.steps
    value = 2.0 * nnz / (ms_per_step * 1e-3)

    # dominant stage = the two half-steps (whitening, tensor-core kernels, unwhitening); device time per stage
    t_user = float(np.mean([e[0].elapsed_time(e[1]) for e in ev_pairs]))
    t_item = float(np.mean([e[2].elapsed_time(e[3]) for e in ev_pairs]))
    # algorithmic bytes of THIS rank's two half-steps (SURVEY.md 8d, without the Gram's read of Y, which belongs to
    # the separate Gram kernel)
    bytes_user = C.nnz * (4 * f + 8) + C.shape[0] * (4 * f + 4)
    bytes_item = CT.nnz * (4 * f + 8) + CT.shape[0] * (4 * f + 4)
    peaks, peak_kind = load_peaks()
    peak = float(peaks["hbm_gbs"])
    achieved = (bytes_user + bytes_item) / ((t_user + t_item) * 1e-3) / 1e9
    flops = (C.nnz + CT.nnz) * (2.0 * f * f + 2 * f) + (C.shape[0] + CT.shape[0]) * (f ** 3 / 3.0 + 2.0 * f * f)
    # what the tensor pipe executes: 3 FP16 passes of the Gram (n f^2 MACs each, every row counted in its primal form;
    # the solves are conjugate gradients on the CUDA cores), reported against the sustained bf16 peak; under
    # --algo tcgen05_direct the 3 TF32 passes of the rank-8 Gauss-Jordan updates (~f^3 / 2 MACs per row) come on top
    tensor_flops = 3 * 2.0 * f * f * (C.nnz + CT.nnz)
    if args.algo == "tcgen05_direct":
        tensor_flops += 3 * 1.0 * f ** 3 * (C.shape[0] + CT.shape[0])
    launches_per_epoch = loop.launches_per_epoch

    # ---- eval_prec alone (SURVEY.md 8d: reported separately): MSE over the stored entries of the count matrix
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u_lo, u_hi = (0, users) if ub is None else (int(ub[rank]), int(ub[rank + 1]))
    engine.sddmm_loss(C, loop.users[u_lo:u_hi], loop.items)
    e0.record()
    for _ in range(3):
        engine.sddmm_loss(C, loop.users[u_lo:u_hi], loop.items)
    e1.record()
    torch.cuda.synchronize(device)
    eval_ms = e0.elapsed_time(e1) / 3
    eval_bytes = C.nnz * (2 * 4 * f + 12)

    # ---- e2e through the public API with host buffers (rank-local timing, max over ranks)
    times, d2h, h2d, marks = [float("nan")], 0, 0, []
    if not args.no_e2e:
        if C_host is None:  # device-generated workload: bring the raw counts to the host once (not timed)
            import scipy.sparse
            C_host = scipy.sparse.csr_matrix((raw_counts.cpu().numpy(), C_full.indices.cpu().numpy(),
                                              C_full.indptr.cpu().numpy()), shape=(users, items))
        del C_full, CT_full, raw_counts
        tr_host, te_host = split_train_test(C_host, train=0.8, seed=1993)
        if not args.pageable:
            tr_host, te_host = pin_csr(tr_host), pin_csr(te_host)   # the contract's e2e inputs: pinned host memory

        def e2e_step():
            t0 = time.perf_counter()
            model.train(tr_host, iterations=1, eval_mat=te_host, count_mat=tr_host, cores=1, stopping_rounds=99)
            u, i = model.users, model.items  # D2H of the result
            return time.perf_counter() - t0, u.nbytes + i.nbytes + 24

        e2e_step()  # warm-up (allocator, pinned staging)
        sync_all()
        e2e_step()  # second warm-up: pinned staging / host allocator caches reach steady state
        sync_all()
        times, marks = [], []
        for _ in range(args.steps):
            sync_all()
            t, d2h = e2e_step()
            times.append(t)
            marks.append([(k, round(v, 2)) for k, v in model.last_train_stats.get("host_marks_ms", [])]
                         + [("train() returned", round(model.last_train_stats.get("total_ms", 0.0), 2)), ("step", round(t * 1e3, 2))])
        if os.environ.get("WMF_BENCH_PROFILE"):   # development: where does the host spend an e2e step?
            import cProfile
            import pstats
            pr = cProfile.Profile()
            pr.enable()
            e2e_step()
            pr.disable()
            pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(30)
        h2d = (tr_host.nnz * 8 + (users + 1) * 8) + (te_host.nnz * 8 + (users + 1) * 8)
        e2e_nnz = tr_host.nnz
    else:
        e2e_nnz = nnz
    # the median step: the GPU box's host is shared, and one step in three or four stalls for tens of ms in the
    # host-side upload (every step and the mean are in the line)
    t_e2e = torch.tensor([float(np.median(times))], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = 2.0 * e2e_nnz / float(t_e2e.item()) if not args.no_e2e else float("nan")

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline and where == "host":
            from oracle import wmf_oracle as orc  # cpu_baseline leg only
            Cp = C_host.copy()
            Cp.data = orc.preprocess_counts(Cp.data, "log", ALPHA, BETA)
            threads = os.cpu_count() or 1
            v, _, desc = cpu_epoch_sample(Cp, Cp.T.tocsr(), dim, 0.3, threads)  # ~10-15 s of host work
            cpu = {"value": v, "unit": "nnz-updates/s", "cores": threads, "kind": "port", "sample": desc, "extrapolated": True}
        traffic, traffic_note = load_traffic() if (world == 1 and args.workload == "ml20m") else (None, "not captured for this run")
        line = {
            "metric": "wmf_nnz_updates_per_sec_per_epoch", "value": value, "unit": "nnz-updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload),
            "run": {"algo": args.algo, "parallelism": f"row-sharded x{world}" if world > 1 else "single GPU",
                    "launch": launch_mode, "exchange": loop.exchange_mode,
                    "solver": ("block Gauss-Jordan in tensor memory" if args.algo == "tcgen05_direct" else
                               "conjugate gradients on the system matrix in tensor memory (relative residual 1e-6; "
                               "rows that do not converge in 64 products are factorised in tensor memory)")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_note": traffic_note + "; algorithmic bytes = %d" % (bytes_user + bytes_item),
                         "peak_kind": peak_kind, "kernel": "als half-step stage (whiten, dual + primal tcgen05 kernels, unwhiten; 2 per epoch)",
                         "ms_user_half_step": t_user, "ms_item_half_step": t_item,
                         "fp32_equiv_tflops": flops / ((t_user + t_item) * 1e-3) / 1e12,
                         "tensor": {"executed_tflops": tensor_flops / ((t_user + t_item) * 1e-3) / 1e12,
                                    "peak": float(peaks["bf16_tflops_sustained"]),
                                    "frac": tensor_flops / ((t_user + t_item) * 1e-3) / 1e12 / float(peaks["bf16_tflops_sustained"]),
                                    "what": "3 FP16 passes of the Gram (every row counted in its primal form) vs the sustained bf16 "
                                            "peak; the solves are conjugate gradients on the CUDA cores"
                                            + (" (+ 3 TF32 passes of the Gauss-Jordan updates: --algo tcgen05_direct)"
                                               if args.algo == "tcgen05_direct" else "")}},
            "eval_prec": {"ms": eval_ms, "gbs": eval_bytes / (eval_ms * 1e-3) / 1e9, "frac_of_hbm_peak": eval_bytes / (eval_ms * 1e-3) / 1e9 / peak,
                          "what": f"sddmm_loss over the {C.nnz} stored entries of this rank's rows (base_model.py:150-179), "
                                  f"algorithmic {eval_bytes} bytes"},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "nnz-updates/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": float(t_e2e.item()) * 1e3,
                    "ms_steps_rank0": [round(t * 1e3, 2) for t in times], "ms_mean_rank0": float(np.mean(times)) * 1e3,
                    "statistic": "median over the listed steps, max over ranks",
                    "host_marks_ms_per_step": marks,
                    "device_ms_last_step": {"half_steps": model.last_train_stats.get("half_step_ms"),
                                            "eval": model.last_train_stats.get("eval_ms")},
                    "what": "WMF.train(host CSR in " + ("pageable" if args.pageable else "pinned") + " host memory, iterations=1) "
                            "incl. upload, preprocess, transpose, epoch, eval_prec, factor read-back; 80/20 split so nnz = "
                            "train nnz"},
            "gpu_launches": int(launches_per_epoch * args.steps),
            "gpu_launches_note": f"{launches_per_epoch} kernel launches of libwmf_b200.so per epoch, counted by the library "
                                 "(wmf_launch_count) while the epoch was captured, x steps",
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
        if outputs:
            dump_outputs(args.dump_outputs, outputs)
    loop.graphs = None
    del loop
    finish(world, device)


def finish(world, device):
    import torch
    import torch.distributed as dist
    if world > 1:
        # Captured NCCL collectives keep the communicator busy at teardown (destroy_process_group was seen to
        # hang with live graphs): drain the device, meet once more and leave without it.
        torch.cuda.synchronize(device)
        dist.barrier()
        torch.cuda.synchronize(device)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="ml20m")
    ap.add_argument("--algo", choices=["auto", "simt", "tcgen05", "tcgen05_direct"], default="auto")
    ap.add_argument("--pageable", action="store_true",
                    help="e2e: hand WMF.train ordinary (pageable) NumPy arrays instead of pinned ones (adds the staging copy)")
    ap.add_argument("--cpu-frac", type=float, default=0.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="kernel tuning runs: skip the end-to-end leg (the line's e2e is NaN)")
    ap.add_argument("--no-graphs", action="store_true", help="launch the epoch from Python instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one computed as DIR/<name>.npy (float32, at most "
                         "64 MB in all; a fixed sample of rows where an output is larger): users.npy and items.npy, the "
                         "factors after the last epoch, or topk_ids.npy for --workload rank")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this package's CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
