"""Device-side operations of the WMF path: thin wrappers that hand torch CUDA tensors
(device memory + stream only) to the C-ABI kernels of libwmf_b200.so.

Nothing in this module computes on the host or with torch operators on the hot path; torch is
used for allocation, H2D/D2H copies, the current stream, and (in ``DeviceCSR.transpose``) a
stable device sort for the one-off CSR transpose.
"""
import os
import weakref

import numpy as np
import torch

from . import _lib

_workspaces = {}


def _stream(device=None):
    """Raw handle of torch's current stream ON THE DEVICE OF THE OPERANDS (not of the current device)."""
    return torch.cuda.current_stream(device).cuda_stream


def _on(device):
    """Context that makes ``device`` current: the C library launches on the current device, so every entry
    point below runs under the device of its operands (WMF(device='cuda:1') with cuda:0 current)."""
    return torch.cuda.device(device)


def _device_of(argpos):
    """Decorator: run the wrapped entry point with the device of its ``argpos``-th tensor argument current."""
    import functools

    def deco(fn):
        @functools.wraps(fn)
        def wrapped(*args, **kwargs):
            with torch.cuda.device(args[argpos].device):
                return fn(*args, **kwargs)
        return wrapped
    return deco


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def workspace(nbytes, device):
    """A cached, grow-only scratch buffer per device. Kernels launched back to back on one
    stream may share it (stream order serialises them)."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


def default_device():
    if not torch.cuda.is_available():
        raise _lib.WMFLibraryError("recmodel_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


_pinned = {}


def _host_copy(dst, src):
    """dst.copy_(src) for large CPU tensors with a fixed, moderate thread count. torch's CPU copy follows its intra-op
    thread count: torchrun pins it to 1 through OMP_NUM_THREADS (18 ms per rank for a 128 MB matrix instead of 2-4),
    and with one thread per logical CPU of a shared host a single descheduled thread stalls the whole copy (1.0 ms
    median, 11 ms worst for 64 MB with 16 threads; 1.6 / 1.9 ms with 8: scripts/dev/host_copy_noise.py)."""
    have = torch.get_num_threads()
    want = max(1, min(8, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
    if have == want or src.numel() < (1 << 20):
        dst.copy_(src)
        return
    torch.set_num_threads(want)
    try:
        dst.copy_(src)
    finally:
        torch.set_num_threads(have)


def _h2d(arr, dtype, device):
    """Host array -> device tensor. Large arrays go through a cached pinned staging buffer (filled by a
    multi-threaded host copy) so the transfer itself runs at PCIe rate instead of the pageable path's."""
    a = np.ascontiguousarray(arr, dtype=dtype)
    t = torch.from_numpy(a)
    n = t.numel()
    if a.nbytes < (4 << 20) or device.type != "cuda":
        return t.to(device, non_blocking=True)
    if t.is_pinned():
        # the caller's array already lives in page-locked memory (and needed no dtype conversion): DMA straight out
        # of it; the staging copy below exists only to give pageable arrays that property
        return t.to(device, non_blocking=True)
    key = (t.dtype, device.index)
    ent = _pinned.get(key)
    if ent is None or ent[0].numel() < n:
        ent = [torch.empty(max(n, 1 << 20), dtype=t.dtype, pin_memory=True), None]
        _pinned[key] = ent
    buf, busy = ent
    if busy is not None:
        busy.synchronize()  # the previous transfer out of this staging buffer has finished
    # chunk by chunk: the DMA of a chunk runs while the host copies the next one into the staging buffer
    out = torch.empty(n, dtype=t.dtype, device=device)
    flat = t.reshape(-1)
    chunk = 4 << 20
    for off in range(0, n, chunk):
        end = min(n, off + chunk)
        _host_copy(buf[off:end], flat[off:end])
        out[off:end].copy_(buf[off:end], non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(device))
    ent[1] = ev
    return out


def d2h(t):
    """Device tensor -> NumPy array backed by pinned host memory from torch's caching host allocator
    (a fresh pageable array costs tens of ms in first-touch page faults at 85 MB)."""
    if not t.is_cuda:
        return t.numpy()
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return h.numpy()


def _f32(t):
    assert t.dtype == torch.float32 and t.is_cuda and t.stride(-1) == 1, "expected a row-major float32 CUDA tensor"
    return t


class DeviceCSR:
    """CSR matrix resident in HBM: indptr int64[rows+1], indices int32[nnz], data float32[nnz],
    plus ``row_order`` (int32 permutation, longest rows first) used as the processing order of
    the half-step kernels."""

    def __init__(self, indptr, indices, data, shape):
        self.indptr, self.indices, self.data = indptr, indices, data
        self.shape = (int(shape[0]), int(shape[1]))
        self.nnz = int(indices.numel())
        self._row_order = None
        self._split_segments = None
        self._sorted = None

    @classmethod
    def from_scipy(cls, mat, device=None):
        device = device or default_device()
        mat = mat.tocsr()
        if mat.shape[1] >= 2 ** 31:
            raise ValueError("column count must fit int32")
        indptr = _h2d(mat.indptr, np.int64, device)
        indices = _h2d(mat.indices, np.int32, device)
        data = _h2d(mat.data, np.float32, device)
        return cls(indptr, indices, data, mat.shape)

    @property
    def device(self):
        return self.indptr.device

    @property
    def row_order(self):
        """Processing schedule for the half-step kernels (see include/wmf_b200.h): rows sorted
        longest first (one stable device sort) and dealt to the persistent CTAs in rounds, each
        round giving its heaviest row to the currently lightest CTA. int32, -1 = padding slot."""
        if self._row_order is None:
            self._row_order = device_schedule(self.indptr, _lib.require_device())
        return self._row_order

    @property
    def split_segments(self):
        """Upper bound of the segments the tcgen05 half-step cuts the long rows of this matrix into
        (include/wmf_b200.h: wmf_als_half_step_workspace_bytes_split)."""
        if self._split_segments is None:
            split = int(_lib.load().wmf_als_row_split_entries())
            counts = self.indptr[1:] - self.indptr[:-1]
            segs = torch.where(counts > split, (counts + (split - 1)) // split, torch.zeros_like(counts))
            self._split_segments = int(segs.sum().item())
        return self._split_segments

    def with_data(self, data):
        out = DeviceCSR(self.indptr, self.indices, data, self.shape)
        out._row_order = self._row_order
        out._split_segments = self._split_segments
        return out

    def row_ids(self):
        counts = self.indptr[1:] - self.indptr[:-1]
        return torch.repeat_interleave(torch.arange(self.shape[0], device=self.device, dtype=torch.int32), counts,
                                       output_size=self.nnz)

    def transpose(self):
        """CSR of the transpose with ascending row ids inside every output row: the ordering
        ``count_mat.T.tocsr()`` produces (wmf_model.py:128). The library's stable radix sort by column
        (wmf_csr_transpose); unsorted or duplicated input entries are fine."""
        lib = _lib.load()
        rows, cols = self.shape
        dev = self.device
        out_indptr = torch.empty(cols + 1, dtype=torch.int64, device=dev)
        out_indices = torch.empty(self.nnz, dtype=torch.int32, device=dev)
        out_data = torch.empty(self.nnz, dtype=torch.float32, device=dev)
        ws = workspace(lib.wmf_csr_transpose_workspace_bytes(rows, cols, self.nnz), dev)
        with _on(dev):
            _lib.check(lib.wmf_csr_transpose(_ptr(self.indptr), _ptr(self.indices), _ptr(self.data), rows, cols, self.nnz,
                                             _ptr(out_indptr), _ptr(out_indices), _ptr(out_data), _ptr(ws), ws.numel(),
                                             _stream(dev)), "wmf_csr_transpose")
        out = DeviceCSR(out_indptr, out_indices, out_data, (cols, rows))
        out._sorted = out
        return out

    def canonical(self):
        """The same matrix with sorted column indices inside every row (two transposes)."""
        return self.transpose().transpose()

    def sorted(self):
        """``canonical()``, computed once: ``self`` when its rows are known to be sorted (a transpose's are)."""
        if self._sorted is None:
            self._sorted = self.canonical()
        return self._sorted

    def row_slice(self, r0, r1):
        """Rows [r0, r1) as an independent DeviceCSR (used to shard rows across GPUs)."""
        lo, hi = int(self.indptr[r0].item()), int(self.indptr[r1].item())
        return DeviceCSR((self.indptr[r0:r1 + 1] - lo).contiguous(), self.indices[lo:hi], self.data[lo:hi],
                         (r1 - r0, self.shape[1]))

    def to_scipy(self):
        import scipy.sparse
        return scipy.sparse.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(), self.indptr.cpu().numpy()),
                                       shape=self.shape)


def device_schedule(indptr, n_cta, chunk=32, row_overhead=4, split=None):
    """``balanced_schedule`` with the O(rows log rows) part on the device: the rows are sorted by
    length there; when no row is heavy (the common case) the padded sorted order IS the schedule
    and nothing but two scalars crosses to the host. With a heavy head only the sorted costs go to
    the host for the greedy placement."""
    counts = indptr[1:] - indptr[:-1]
    rows = counts.numel()
    if rows == 0:
        return torch.full((n_cta,), -1, dtype=torch.int32, device=indptr.device)
    if split is None:
        split = int(_lib.load().wmf_als_row_split_entries())
    # the kernel cuts longer rows into segments and spreads the extra segments over all CTAs: a row never
    # costs its CTA more than one segment
    counts = torch.clamp(counts, max=split)
    sorted_counts, order = torch.sort(counts, descending=True, stable=True)
    cost = torch.where(sorted_counts > 0, (sorted_counts + (chunk - 1)) // chunk + row_overhead,
                       torch.zeros_like(sorted_counts))
    head = torch.stack((cost[0], cost.sum())).cpu()
    mean_load = float(head[1]) / n_cta
    if float(head[0]) < 0.05 * mean_load:  # no heavy head: round-robin over the sorted rows is balanced
        sched = torch.full((((rows + n_cta - 1) // n_cta) * n_cta,), -1, dtype=torch.int32, device=indptr.device)
        sched[:rows] = order.to(torch.int32)
        return sched
    sched = _schedule_from_sorted(order.cpu().numpy(), cost.cpu().numpy(), n_cta)
    return torch.from_numpy(sched).to(indptr.device)


def balanced_schedule(counts, n_cta, chunk=32, row_overhead=4):
    """Longest-processing-time schedule for the persistent CTAs (host version of
    ``device_schedule``). Cost of a row = its 32-entry chunks plus a fixed solve overhead. Returns
    int32[n_slots * n_cta]; slot k*n_cta + c is the k-th row of CTA c, -1 where that CTA has no
    k-th row (a CTA that owns a very long row takes fewer rows)."""
    counts = np.asarray(counts, dtype=np.int64)
    rows = len(counts)
    if rows == 0:
        return np.full(n_cta, -1, dtype=np.int32)
    order = np.argsort(-counts, kind="stable")
    cost = np.where(counts > 0, (counts + chunk - 1) // chunk + row_overhead, 0).astype(np.int64)[order]
    mean_load = cost.sum() / n_cta
    if cost[0] < 0.05 * mean_load:  # no heavy head: round-robin over the sorted rows is balanced
        sched = np.full(((rows + n_cta - 1) // n_cta) * n_cta, -1, dtype=np.int32)
        sched[:rows] = order
        return sched
    return _schedule_from_sorted(order, cost, n_cta)


def _schedule_from_sorted(order, cost, n_cta):
    """Heavy head: greedy LPT for the rows that matter, then rounds over the currently lightest
    CTAs. ``assign[k]`` = CTA of the k-th heaviest row; the schedule is built from it in one pass."""
    import heapq
    rows = len(order)
    order = np.asarray(order, dtype=np.int64)
    cost = np.asarray(cost, dtype=np.int64)
    mean_load = cost.sum() / n_cta
    assign = np.empty(rows, dtype=np.int64)
    n_head = int(np.searchsorted(-cost, -max(1, int(0.01 * mean_load)), side="right"))
    heap = [(0, c) for c in range(n_cta)]
    head_cost = cost[:n_head].tolist()
    for k in range(n_head):
        load, c = heapq.heappop(heap)
        assign[k] = c
        heapq.heappush(heap, (load + head_cost[k], c))
    load = np.zeros(n_cta)
    for l, c in heap:
        load[c] = l
    k = n_head
    remaining = float(cost[k:].sum())
    total = float(load.sum()) + remaining
    while k < rows:  # tail rows are small: hand them out in rounds to the currently lightest CTAs
        take = min(n_cta, rows - k)
        ctas = np.argsort(load, kind="stable")
        below = ctas[load[ctas] < total / n_cta][:take]
        ctas = below if len(below) else ctas[:take]
        n = len(ctas)
        assign[k:k + n] = ctas
        load[ctas] += cost[k:k + n]
        k += n
    by_cta = np.argsort(assign, kind="stable")           # rows grouped by CTA, heaviest first inside a CTA
    per_cta = np.bincount(assign, minlength=n_cta)
    starts = np.concatenate(([0], np.cumsum(per_cta)[:-1]))
    slot = np.arange(rows) - np.repeat(starts, per_cta)
    sched = np.full((int(per_cta.max()), n_cta), -1, dtype=np.int32)
    sched[slot, assign[by_cta]] = order[by_cta]
    return sched.reshape(-1)


def preprocess_(data, mode, alpha, beta):
    """In place d = alpha*log(1+beta*x) | alpha*x  (wmf_model.py:119-123)."""
    lib = _lib.load()
    codes = {"log": _lib.PREPROCESS_LOG, "linear": _lib.PREPROCESS_LINEAR}
    if mode not in codes:
        raise ValueError(f"Pre_process_count {mode} is not implement please use log or linear.")
    with _on(data.device):
        _lib.check(lib.wmf_preprocess(_ptr(_f32(data)), data.numel(), codes[mode], float(alpha), float(beta),
                                      _stream(data.device)), "wmf_preprocess")
    return data


def gram(Y, lam, ones_col0=False, ws=None, out=None):
    """G = Y^T Y + lam I (wmf_model.py:215 / :332 with the ones column). ``ws``: caller-owned scratch
    (captured CUDA graphs must not use the shared grow-only cache)."""
    lib = _lib.load()
    _f32(Y)
    n, f = Y.shape
    G = out if out is not None else torch.empty((f, f), dtype=torch.float32, device=Y.device)
    need = lib.wmf_gram_workspace_bytes(n, f)
    if ws is None:
        ws = workspace(need, Y.device)
    with _on(Y.device):
        _lib.check(lib.wmf_gram(_ptr(Y), n, f, Y.stride(0), float(lam), int(bool(ones_col0)), _ptr(G), _ptr(ws),
                                ws.numel(), _stream(Y.device)), "wmf_gram")
    return G


def gram_block_rows(n):
    """Rows per Gram block for a matrix of n rows (a function of n alone): shard boundaries of a
    row-sharded run are multiples of it, so every rank can compute the blocks of its own rows."""
    return int(_lib.load().wmf_gram_block_rows(int(n)))


def gram_blocks(n):
    """Number of Gram blocks of a matrix of n rows (a function of n alone)."""
    return int(_lib.load().wmf_gram_blocks(int(n)))


def gram_partials(Y_local, row0, n_total, ones_col0=False, out=None):
    """float64 [blocks, f, f] buffer holding the Gram partials of the blocks inside the local slice
    (global rows [row0, row0 + len(Y_local))) and zeros elsewhere; see include/wmf_b200.h. ``out``: an existing
    buffer of that shape (only the local blocks are written: the peer-memory exchange fills the others)."""
    lib = _lib.load()
    _f32(Y_local)
    nloc, f = Y_local.shape
    blocks = int(lib.wmf_gram_blocks(int(n_total)))
    buf = out if out is not None else torch.zeros((blocks, f, f), dtype=torch.float64, device=Y_local.device)
    with _on(Y_local.device):
        _lib.check(lib.wmf_gram_partials(_ptr(Y_local), int(row0), nloc, int(n_total), f, Y_local.stride(0),
                                         int(bool(ones_col0)), _ptr(buf), buf.numel() * 8, _stream(Y_local.device)),
                   "wmf_gram_partials")
    return buf


def peer_broadcast(src, peer_table, world, self_rank, dst_offset_bytes):
    """Write the contiguous tensor ``src`` to byte offset ``dst_offset_bytes`` of every peer's symmetric buffer
    (``peer_table``: int64 device tensor of peer-mapped base addresses); include/wmf_b200.h: wmf_peer_broadcast."""
    lib = _lib.load()
    assert src.is_contiguous()
    with _on(src.device):
        _lib.check(lib.wmf_peer_broadcast(_ptr(src), src.numel() * src.element_size(), _ptr(peer_table), int(world),
                                          int(self_rank), int(dst_offset_bytes), _stream(src.device)), "wmf_peer_broadcast")


def gram_from_partials(partials, n_total, lam, out=None):
    """G from the (exchanged) block partials: blocks added in block order, rounded once, + lam I."""
    lib = _lib.load()
    f = partials.shape[1]
    G = out if out is not None else torch.empty((f, f), dtype=torch.float32, device=partials.device)
    with _on(partials.device):
        _lib.check(lib.wmf_gram_reduce(_ptr(partials), int(n_total), f, float(lam), _ptr(G), _stream(partials.device)),
                   "wmf_gram_reduce")
    return G


def half_step_workspace_bytes(csr, f, algo=_lib.ALGO_AUTO):
    """Scratch bytes one ``half_step`` over ``csr`` needs (its long rows included)."""
    return int(_lib.load().wmf_als_half_step_workspace_bytes_split(csr.shape[0], csr.shape[1], f, int(algo),
                                                                   csr.split_segments))


def half_step(csr, Y, G, bias=False, algo=_lib.ALGO_AUTO, out=None, use_row_order=True, ws=None):
    """X = one ALS half-step over the rows of ``csr`` against fixed factors Y
    (wmf_model.py:213-240 / :311-351). ``ws``: caller-owned scratch of ``half_step_workspace_bytes`` bytes
    (a captured CUDA graph must own its scratch); by default the shared grow-only cache of the device."""
    lib = _lib.load()
    _f32(Y)
    _f32(G)
    rows = csr.shape[0]
    f = Y.shape[1]
    if csr.shape[1] != Y.shape[0]:
        raise ValueError(f"count matrix has {csr.shape[1]} columns but Y has {Y.shape[0]} rows")
    X = out if out is not None else torch.empty((rows, f), dtype=torch.float32, device=Y.device)
    if ws is None:
        ws = workspace(half_step_workspace_bytes(csr, f, algo), Y.device)
    order = csr.row_order if use_row_order else None
    with _on(Y.device):
        _lib.check(lib.wmf_als_half_step(_ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), rows, csr.shape[1],
                                         _ptr(order), 0 if order is None else order.numel(), _ptr(Y), Y.stride(0), f,
                                         _ptr(G), int(bool(bias)), _ptr(X), X.stride(0), int(algo), _ptr(ws), ws.numel(),
                                         _stream(Y.device)), "wmf_als_half_step")
    half_step.last_ws = weakref.ref(ws)
    return X


def half_step_status(ws=None):
    """(flags, fix-up rows) of the last tcgen05 half-step that used ``ws`` (synchronises its stream)."""
    import ctypes
    lib = _lib.load()
    if ws is None:
        ref = getattr(half_step, "last_ws", None)
        ws = ref() if ref is not None else None
    if ws is None:
        return 0, 0
    flags, fixed = ctypes.c_int(0), ctypes.c_int(0)
    with _on(ws.device):
        _lib.check(lib.wmf_als_half_step_status(_ptr(ws), ctypes.addressof(flags), ctypes.addressof(fixed),
                                                _stream(ws.device)), "wmf_als_half_step_status")
    return flags.value, fixed.value


def half_step_used_fallback(ws=None):
    """True if some row of the last tcgen05 half-step that used ``ws`` was factorised in tensor memory because its
    conjugate gradients did not converge within their product budget (synchronises the stream)."""
    import ctypes
    lib = _lib.load()
    if ws is None:
        ref = getattr(half_step, "last_ws", None)
        ws = ref() if ref is not None else None
    if ws is None:
        return False
    rows = ctypes.c_int(0)
    with _on(ws.device):
        _lib.check(lib.wmf_als_half_step_used_fallback(_ptr(ws), ctypes.addressof(rows), _stream(ws.device)),
                   "wmf_als_half_step_used_fallback")
    return rows.value != 0


@_device_of(1)
def sddmm_loss(csr, U, V, bias=False):
    """Device tensor [sum sq err, sum abs err, count] (float64) over the non-zero stored entries
    of ``csr`` (base_model.py:163-176 with predict, wmf_model.py:205-211)."""
    lib = _lib.load()
    _f32(U)
    _f32(V)
    out = torch.empty(3, dtype=torch.float64, device=U.device)
    need = lib.wmf_sddmm_loss_workspace_bytes(csr.nnz)
    ws = workspace(need, U.device)
    _lib.check(lib.wmf_sddmm_loss(_ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), csr.shape[0], csr.nnz, _ptr(U),
                                  U.stride(0), _ptr(V), V.stride(0), U.shape[1], int(bool(bias)), _ptr(out), _ptr(ws),
                                  ws.numel(), _stream()), "wmf_sddmm_loss")
    return out


@_device_of(2)
def predict_pairs(users, items, U, V, bias=False):
    """float32 scores of (users[k], items[k]); a single user broadcasts (wmf_model.py:191-211)."""
    lib = _lib.load()
    _f32(U)
    _f32(V)
    n = items.numel()
    stride = 1
    if users.numel() == 1 and n != 1:
        stride = 0
    elif users.numel() != n:
        raise ValueError("users and items need to have the same length or only one user / item needs to be provided.")
    out = torch.empty(n, dtype=torch.float32, device=U.device)
    _lib.check(lib.wmf_predict_pairs(_ptr(users), stride, _ptr(items), n, _ptr(U), U.stride(0), _ptr(V), V.stride(0),
                                     U.shape[1], int(bool(bias)), _ptr(out), _stream()), "wmf_predict_pairs")
    return out


@_device_of(0)
def rank_ahead(S, cand, slot, pair_user, pair_item, pair_score):
    """int32 [pairs]: how many candidates of its user's list WMF.rank puts ahead of each held-out item
    (include/wmf_b200.h: wmf_rank_ahead; base_model.py:84-95)."""
    lib = _lib.load()
    _f32(S)
    nu, L = S.shape
    n = pair_user.numel()
    out = torch.empty(n, dtype=torch.int32, device=S.device)
    assert cand.dtype == torch.int32 and slot.dtype == torch.int32 and pair_user.dtype == torch.int32
    assert pair_item.dtype == torch.int32 and pair_score.dtype == torch.float32 and cand.shape == S.shape
    _lib.check(lib.wmf_rank_ahead(_ptr(S), _ptr(cand), _ptr(slot), nu, L, _ptr(pair_user), _ptr(pair_item),
                                  _ptr(pair_score), n, _ptr(out), _stream()), "wmf_rank_ahead")
    return out


@_device_of(2)
def score_topk(users, cand, U, V, topn, bias=False, want_scores=False):
    """Top-``topn`` candidate ids [nu x topn] (int64), best first, for each user in ``users``
    over the shared candidate list ``cand`` (None = all items) (wmf_model.py:25-47)."""
    lib = _lib.load()
    _f32(U)
    _f32(V)
    nu = users.numel()
    ni = V.shape[0] if cand is None else cand.numel()
    ids = torch.empty((nu, topn), dtype=torch.int64, device=U.device)
    scores = torch.empty((nu, topn), dtype=torch.float32, device=U.device) if want_scores else None
    need = lib.wmf_score_topk_workspace_bytes(nu, ni, topn)
    ws = workspace(need, U.device)
    _lib.check(lib.wmf_score_topk(_ptr(users), nu, _ptr(cand), ni, _ptr(U), U.stride(0), _ptr(V), V.stride(0),
                                  U.shape[1], int(bool(bias)), int(topn), _ptr(ids), _ptr(scores), _ptr(ws), ws.numel(),
                                  _stream()), "wmf_score_topk")
    return (ids, scores) if want_scores else ids


@_device_of(2)
def score_topk_exclude(users, exclude, U, V, topn, bias=False, want_scores=False):
    """Top-``topn`` item ids [nu x topn] (int64) over all items minus the stored entries of row ``users[k]`` of
    ``exclude`` (a DeviceCSR with sorted rows, indexed by user id), -1 where a user has fewer unseen items
    (include/wmf_b200.h: wmf_score_topk_exclude). Returns (ids, scores or None, fixup_users): the last is a device
    int32 [1], the number of users whose candidate list made the exact kernels redo the call."""
    lib = _lib.load()
    _f32(U)
    _f32(V)
    nu, ni = users.numel(), V.shape[0]
    assert exclude.shape[1] == ni and exclude.indices.dtype == torch.int32 and exclude.indptr.dtype == torch.int64
    ids = torch.empty((nu, topn), dtype=torch.int64, device=U.device)
    scores = torch.empty((nu, topn), dtype=torch.float32, device=U.device) if want_scores else None
    fixup = torch.zeros(1, dtype=torch.int32, device=U.device)
    ws = workspace(lib.wmf_score_topk_exclude_workspace_bytes(nu, ni, topn), U.device)
    _lib.check(lib.wmf_score_topk_exclude(_ptr(users), nu, _ptr(exclude.indptr), _ptr(exclude.indices), ni, _ptr(U),
                                          U.stride(0), _ptr(V), V.stride(0), U.shape[1], int(bool(bias)), int(topn),
                                          _ptr(ids), _ptr(scores), _ptr(fixup), _ptr(ws), ws.numel(), _stream()),
               "wmf_score_topk_exclude")
    return ids, scores, fixup


TOPN_METRICS = ("Recall", "Precision", "NDCG", "MAP", "HitRate")  # the 5 values per cutoff, in buffer order


@_device_of(0)
def topn_metrics(ids, users, test_csr, ks, out=None):
    """float64 [nu x len(ks) x 5] (``TOPN_METRICS`` order): ranking quality of the lists ``ids`` [nu x K] (int64, -1
    padding) for the users ``users`` against the rows of ``test_csr`` (a DeviceCSR with sorted rows, indexed by user
    id), one row of NaN per user without a non-zero test entry (include/wmf_b200.h: wmf_topn_metrics). ``ks``: host
    sequence of at most 16 distinct cutoffs in [1, K]. ``out``: a contiguous buffer of that shape to write into."""
    lib = _lib.load()
    nu, K = ids.shape
    ks_h = np.ascontiguousarray(ks, dtype=np.int32)
    assert ids.dtype == torch.int64 and ids.is_contiguous() and users.dtype == torch.int64 and users.numel() == nu
    assert test_csr.indices.dtype == torch.int32 and test_csr.indptr.dtype == torch.int64
    if out is None:
        out = torch.empty((nu, len(ks_h), 5), dtype=torch.float64, device=ids.device)
    assert out.dtype == torch.float64 and out.is_contiguous() and tuple(out.shape) == (nu, len(ks_h), 5)
    _lib.check(lib.wmf_topn_metrics(_ptr(ids), nu, K, _ptr(users), _ptr(test_csr.indptr), _ptr(test_csr.indices),
                                    _ptr(test_csr.data), ks_h.ctypes.data, len(ks_h), _ptr(out), _stream()),
               "wmf_topn_metrics")
    return out


@_device_of(0)
def topn_metrics_reduce(per_user, nk):
    """float64 device [nk*5 + 1]: the sums of the per-user values of ``topn_metrics`` over the rows that are not NaN,
    then the number of those rows (include/wmf_b200.h: wmf_topn_metrics_reduce; bitwise reproducible)."""
    lib = _lib.load()
    nu = per_user.shape[0]
    assert per_user.dtype == torch.float64 and per_user.is_contiguous() and per_user.numel() == nu * nk * 5
    sums = torch.empty(nk * 5 + 1, dtype=torch.float64, device=per_user.device)
    ws = workspace(lib.wmf_topn_metrics_workspace_bytes(nu, nk), per_user.device)
    _lib.check(lib.wmf_topn_metrics_reduce(_ptr(per_user), nu, nk, _ptr(sums), _ptr(ws), ws.numel(), _stream()),
               "wmf_topn_metrics_reduce")
    return sums


@_device_of(1)
def unweighted_half_step(csr, Y, lam):
    """X = R (inv(Y^T Y + lam I) Y^T)^T  (wmf_model.py:85 / :88)."""
    lib = _lib.load()
    _f32(Y)
    n, f = Y.shape
    G = gram(Y, lam)
    Ginv = torch.empty_like(G)
    ws = workspace(lib.wmf_inverse_workspace_bytes(f), Y.device)
    _lib.check(lib.wmf_inverse(_ptr(G), f, _ptr(Ginv), _ptr(ws), ws.numel(), _stream()), "wmf_inverse")
    W = torch.empty((n, f), dtype=torch.float32, device=Y.device)
    _lib.check(lib.wmf_dense_right_multiply(_ptr(Y), n, Y.stride(0), _ptr(Ginv), f, _ptr(W), W.stride(0), _stream()),
               "wmf_dense_right_multiply")
    X = torch.empty((csr.shape[0], f), dtype=torch.float32, device=Y.device)
    _lib.check(lib.wmf_spmm(_ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), csr.shape[0], _ptr(W), W.stride(0), f,
                            _ptr(X), X.stride(0), _stream()), "wmf_spmm")
    return X


@_device_of(0)
def ease_train(csr, alpha):
    """W of the EASE model for the interaction matrix ``csr`` (ease_model.py:81-114): dense [items x items] float32."""
    lib = _lib.load()
    n = csr.shape[1]
    W = torch.empty((n, n), dtype=torch.float32, device=csr.device)
    ws = workspace(lib.wmf_ease_workspace_bytes(n), csr.device)
    _lib.check(lib.wmf_ease_train(_ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), csr.shape[0], n, float(alpha), _ptr(W),
                                  _ptr(ws), ws.numel(), _stream()), "wmf_ease_train")
    return W


@_device_of(1)
def ease_predict(csr, W, users, items):
    """float64 scores sum_j X[user, j] W[j, item] of (users[k], items[k]); one user broadcasts (ease_utils.pyx:15-30)."""
    lib = _lib.load()
    _f32(W)
    n = items.numel()
    stride = 1
    if users.numel() == 1 and n != 1:
        stride = 0
    elif users.numel() != n:
        raise ValueError("users and items need to have the same length or only one user needs to be provided.")
    out = torch.empty(n, dtype=torch.float64, device=W.device)
    _lib.check(lib.wmf_ease_predict(_ptr(csr.indptr), _ptr(csr.indices), _ptr(csr.data), _ptr(W), W.shape[0], _ptr(users), stride,
                                    _ptr(items), n, _ptr(out), _stream()), "wmf_ease_predict")
    return out


@_device_of(1)
def ease_score_topk(X_csr, W, users, topn, exclude=None, want_scores=False):
    """Top-``topn`` item ids [nu x topn] (int64) of the EASE scores sum_j X[user, j] W[j, item] (float64, bitwise those
    of ``ease_predict``) for each user in ``users`` over all items minus the stored entries of row ``users[k]`` of
    ``exclude`` (a DeviceCSR indexed by user id, any row order, or None), best first, ties to the lower item id, -1
    where a user has fewer unseen items (include/wmf_b200.h: wmf_ease_score_topk). With ``want_scores`` returns
    (ids, float64 scores, NaN at the -1 entries)."""
    lib = _lib.load()
    _f32(W)
    n = W.shape[0]
    nu = users.numel()
    assert users.dtype == torch.int64 and X_csr.shape[1] == n
    if exclude is not None:
        assert exclude.shape[1] == n and exclude.indices.dtype == torch.int32 and exclude.indptr.dtype == torch.int64
    ids = torch.empty((nu, topn), dtype=torch.int64, device=W.device)
    scores = torch.empty((nu, topn), dtype=torch.float64, device=W.device) if want_scores else None
    ws = workspace(lib.wmf_ease_score_topk_workspace_bytes(nu, n, topn), W.device)
    _lib.check(lib.wmf_ease_score_topk(_ptr(X_csr.indptr), _ptr(X_csr.indices), _ptr(X_csr.data), _ptr(W), n,
                                       _ptr(users), nu, _ptr(None if exclude is None else exclude.indptr),
                                       _ptr(None if exclude is None else exclude.indices), int(topn), _ptr(ids),
                                       _ptr(scores), _ptr(ws), ws.numel(), _stream()), "wmf_ease_score_topk")
    return (ids, scores) if want_scores else ids


@_device_of(0)
def knn_train(X_csr, XT_csr, k, similarity, shrink):
    """The ItemKNN neighbours of the canonical interaction matrix ``X_csr`` (sorted rows, no duplicates, no explicit
    zeros; ``XT_csr`` its transpose): (indptr int64 [n+1], indices int32, data float64) of the n x n CSR W, rows
    sorted by id (include/wmf_b200.h: wmf_knn_train). ``similarity``: a key of ``_lib.KNN_SIMILARITIES``. Called as
    ``knn_train(X.transpose(), X, ...)`` it returns the UserKNN neighbours of X (n = the number of users)."""
    lib = _lib.load()
    n = X_csr.shape[1]
    dev = X_csr.device
    kk = min(int(k), n)
    indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    indices = torch.empty(n * kk, dtype=torch.int32, device=dev)
    data = torch.empty(n * kk, dtype=torch.float64, device=dev)
    ws = workspace(lib.wmf_knn_train_workspace_bytes(n, int(k)), dev)
    _lib.check(lib.wmf_knn_train(_ptr(X_csr.indptr), _ptr(X_csr.indices), X_csr.shape[0], _ptr(XT_csr.indptr),
                                 _ptr(XT_csr.indices), n, int(k), _lib.KNN_SIMILARITIES[similarity], float(shrink),
                                 _ptr(indptr), _ptr(indices), _ptr(data), _ptr(ws), ws.numel(), _stream()),
               "wmf_knn_train")
    nnz = int(indptr[-1])
    if nnz < n * kk:
        indices, data = indices[:nnz].clone(), data[:nnz].clone()
    return indptr, indices, data


@_device_of(0)
def rp3beta_train(P_csr, PT_csr, du, ra, cb, k):
    """The RP3beta weights of the binary pattern ``P_csr`` of a canonical interaction matrix (``PT_csr`` its
    transpose) from the float64 device scales du [users], ra [items] and cb [items] (include/wmf_b200.h:
    wmf_rp3beta_train): (indptr int64 [n+1], indices int32, data float64) of the n x n CSR W, rows sorted by id, the
    layout ``knn_predict`` and ``knn_score_topk`` take."""
    lib = _lib.load()
    n = P_csr.shape[1]
    dev = P_csr.device
    assert du.dtype == ra.dtype == cb.dtype == torch.float64 and du.numel() == P_csr.shape[0]
    assert ra.numel() == cb.numel() == n and PT_csr.nnz == P_csr.nnz
    kk = min(int(k), n)
    indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    indices = torch.empty(n * kk, dtype=torch.int32, device=dev)
    data = torch.empty(n * kk, dtype=torch.float64, device=dev)
    ws = workspace(lib.wmf_rp3beta_train_workspace_bytes(n, P_csr.nnz, int(k)), dev)
    _lib.check(lib.wmf_rp3beta_train(_ptr(P_csr.indptr), _ptr(P_csr.indices), P_csr.shape[0], _ptr(PT_csr.indptr),
                                     _ptr(PT_csr.indices), n, P_csr.nnz, _ptr(du), _ptr(ra), _ptr(cb), int(k),
                                     _ptr(indptr), _ptr(indices), _ptr(data), _ptr(ws), ws.numel(), _stream()),
               "wmf_rp3beta_train")
    nnz = int(indptr[-1])
    if nnz < n * kk:
        indices, data = indices[:nnz].clone(), data[:nnz].clone()
    return indptr, indices, data


@_device_of(0)
def knn_predict(X_csr, W, users, items):
    """float64 ItemKNN scores s(users[k], items[k]) (include/wmf_b200.h: wmf_knn_predict) for the canonical ``X_csr``
    and W = (indptr, indices, data) as ``knn_train`` returns it; one user broadcasts."""
    lib = _lib.load()
    w_indptr, w_indices, w_data = W
    n = items.numel()
    stride = 1
    if users.numel() == 1 and n != 1:
        stride = 0
    elif users.numel() != n:
        raise ValueError("users and items need to have the same length or only one user needs to be provided.")
    out = torch.empty(n, dtype=torch.float64, device=w_indptr.device)
    _lib.check(lib.wmf_knn_predict(_ptr(X_csr.indptr), _ptr(X_csr.indices), _ptr(X_csr.data), _ptr(w_indptr),
                                   _ptr(w_indices), _ptr(w_data), _ptr(users), stride, _ptr(items), n, _ptr(out),
                                   _stream()), "wmf_knn_predict")
    return out


@_device_of(0)
def knn_score_topk(X_csr, W, users, topn, exclude=None, want_scores=False):
    """``ease_score_topk`` for the ItemKNN scores of ``knn_predict`` (bitwise): top-``topn`` item ids [nu x topn]
    (int64) over all items minus the stored entries of row ``users[k]`` of ``exclude``, best first, ties to the lower
    item id, -1 padding (include/wmf_b200.h: wmf_knn_score_topk); with ``want_scores`` (ids, float64 scores)."""
    lib = _lib.load()
    w_indptr, w_indices, w_data = W
    n = w_indptr.numel() - 1
    nu = users.numel()
    dev = w_indptr.device
    assert users.dtype == torch.int64 and X_csr.shape[1] == n
    if exclude is not None:
        assert exclude.shape[1] == n and exclude.indices.dtype == torch.int32 and exclude.indptr.dtype == torch.int64
    ids = torch.empty((nu, topn), dtype=torch.int64, device=dev)
    scores = torch.empty((nu, topn), dtype=torch.float64, device=dev) if want_scores else None
    ws = workspace(lib.wmf_knn_score_topk_workspace_bytes(nu, n, topn), dev)
    _lib.check(lib.wmf_knn_score_topk(_ptr(X_csr.indptr), _ptr(X_csr.indices), _ptr(X_csr.data), _ptr(w_indptr),
                                      _ptr(w_indices), _ptr(w_data), n, _ptr(users), nu,
                                      _ptr(None if exclude is None else exclude.indptr),
                                      _ptr(None if exclude is None else exclude.indices), int(topn), _ptr(ids),
                                      _ptr(scores), _ptr(ws), ws.numel(), _stream()), "wmf_knn_score_topk")
    return (ids, scores) if want_scores else ids


@_device_of(0)
def userknn_predict(X_csr, N, users, items):
    """float64 UserKNN scores s(users[k], items[k]) (include/wmf_b200.h: wmf_userknn_predict) for the canonical
    ``X_csr`` and the user-user neighbours N = (indptr, indices, data) as ``knn_train(X_csr.transpose(), X_csr, ...)``
    returns them; one user broadcasts."""
    lib = _lib.load()
    nb_indptr, nb_indices, nb_data = N
    n = items.numel()
    stride = 1
    if users.numel() == 1 and n != 1:
        stride = 0
    elif users.numel() != n:
        raise ValueError("users and items need to have the same length or only one user needs to be provided.")
    out = torch.empty(n, dtype=torch.float64, device=nb_indptr.device)
    _lib.check(lib.wmf_userknn_predict(_ptr(X_csr.indptr), _ptr(X_csr.indices), _ptr(X_csr.data), _ptr(nb_indptr),
                                       _ptr(nb_indices), _ptr(nb_data), _ptr(users), stride, _ptr(items), n, _ptr(out),
                                       _stream()), "wmf_userknn_predict")
    return out


@_device_of(0)
def userknn_score_topk(X_csr, N, users, topn, exclude=None, want_scores=False):
    """``knn_score_topk`` for the UserKNN scores of ``userknn_predict`` (bitwise): top-``topn`` item ids [nu x topn]
    (int64) over all items minus the stored entries of row ``users[k]`` of ``exclude``, best first, ties to the lower
    item id, -1 padding (include/wmf_b200.h: wmf_userknn_score_topk); with ``want_scores`` (ids, float64 scores).
    ``users`` index the rows of N and N's column ids the rows of ``X_csr``: N is the training neighbours or the
    ``userknn_fold_in`` rows of new histories."""
    lib = _lib.load()
    nb_indptr, nb_indices, nb_data = N
    n = X_csr.shape[1]
    nu = users.numel()
    dev = nb_indptr.device
    assert users.dtype == torch.int64
    if exclude is not None:
        assert exclude.shape[1] == n and exclude.indices.dtype == torch.int32 and exclude.indptr.dtype == torch.int64
    ids = torch.empty((nu, topn), dtype=torch.int64, device=dev)
    scores = torch.empty((nu, topn), dtype=torch.float64, device=dev) if want_scores else None
    ws = workspace(lib.wmf_userknn_score_topk_workspace_bytes(nu, n, topn), dev)
    _lib.check(lib.wmf_userknn_score_topk(_ptr(X_csr.indptr), _ptr(X_csr.indices), _ptr(X_csr.data), _ptr(nb_indptr),
                                          _ptr(nb_indices), _ptr(nb_data), n, _ptr(users), nu,
                                          _ptr(None if exclude is None else exclude.indptr),
                                          _ptr(None if exclude is None else exclude.indices), int(topn), _ptr(ids),
                                          _ptr(scores), _ptr(ws), ws.numel(), _stream()), "wmf_userknn_score_topk")
    return (ids, scores) if want_scores else ids


@_device_of(1)
def userknn_fold_in(Q_csr, XT_csr, X_csr, k, similarity, shrink):
    """The UserKNN neighbours N' among the training users of the rows of ``Q_csr`` (new histories, canonical like X)
    for the canonical training ``X_csr`` (``XT_csr`` its transpose): (indptr int64 [nq+1], indices int32, data float64)
    of the nq x m CSR, rows sorted by user id (include/wmf_b200.h: wmf_userknn_fold_in), the layout
    ``userknn_predict`` and ``userknn_score_topk`` take with user ids = rows of ``Q_csr``."""
    lib = _lib.load()
    nq, m = Q_csr.shape[0], X_csr.shape[0]
    dev = XT_csr.device
    assert Q_csr.shape[1] == XT_csr.shape[0] == X_csr.shape[1] and XT_csr.shape[1] == m
    kk = min(int(k), m)
    indptr = torch.zeros(nq + 1, dtype=torch.int64, device=dev)
    indices = torch.empty(nq * kk, dtype=torch.int32, device=dev)
    data = torch.empty(nq * kk, dtype=torch.float64, device=dev)
    if nq == 0:
        return indptr, indices, data
    ws = workspace(lib.wmf_userknn_fold_in_workspace_bytes(nq, m, int(k)), dev)
    _lib.check(lib.wmf_userknn_fold_in(_ptr(Q_csr.indptr), _ptr(Q_csr.indices), nq, _ptr(XT_csr.indptr),
                                       _ptr(XT_csr.indices), XT_csr.shape[0], _ptr(X_csr.indptr), m, int(k),
                                       _lib.KNN_SIMILARITIES[similarity], float(shrink), _ptr(indptr), _ptr(indices),
                                       _ptr(data), _ptr(ws), ws.numel(), _stream()), "wmf_userknn_fold_in")
    nnz = int(indptr[-1])
    if nnz < nq * kk:
        indices, data = indices[:nnz].clone(), data[:nnz].clone()
    return indptr, indices, data


@_device_of(0)
def slim_train(X_csr, XT_csr, k, l1, l2, max_iter, tol):
    """The SLIM weights of the canonical interaction matrix ``X_csr`` (``XT_csr`` its transpose): the candidates are
    the ``knn_train`` cosine neighbours (shrink 0) of each item, then ``wmf_slim_train`` solves every column (include/
    wmf_b200.h). Returns (W, sweeps): W = (indptr int64 [n+1], indices int32, data float64), the n x n CSR with W[a, j]
    in row a, ascending ids (the layout ``knn_predict`` and ``knn_score_topk`` take), and sweeps int32 [n]."""
    lib = _lib.load()
    n = X_csr.shape[1]
    dev = X_csr.device
    kk = min(int(k), n)
    cand_indptr, cand_indices, _ = knn_train(X_csr, XT_csr, k, "cosine", 0.0)
    wt_indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    wt_indices = torch.empty(n * kk, dtype=torch.int32, device=dev)
    wt_data = torch.empty(n * kk, dtype=torch.float64, device=dev)
    sweeps = torch.empty(n, dtype=torch.int32, device=dev)
    nbytes = lib.wmf_slim_train_workspace_bytes(n, int(k))
    if nbytes == 0:
        raise ValueError(f"SLIM takes 1..{_lib.SLIM_K_MAX} candidates and at most 2^30 items, got k={k}, n={n}")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)   # the dense n x n G: not kept in the shared workspace
    _lib.check(lib.wmf_slim_train(_ptr(X_csr.indptr), _ptr(X_csr.indices), X_csr.shape[0], _ptr(XT_csr.indptr),
                                  _ptr(XT_csr.indices), n, _ptr(cand_indptr), _ptr(cand_indices), int(k), float(l1),
                                  float(l2), int(max_iter), float(tol), _ptr(wt_indptr), _ptr(wt_indices),
                                  _ptr(wt_data), _ptr(sweeps), _ptr(ws), ws.numel(), _stream()), "wmf_slim_train")
    del ws
    nnz = int(wt_indptr[-1])
    cols = torch.repeat_interleave(torch.arange(n, device=dev, dtype=torch.int64), wt_indptr[1:] - wt_indptr[:-1],
                                   output_size=nnz)
    rows = wt_indices[:nnz].to(torch.int64)
    keys, order = torch.sort(rows * n + cols, stable=True)   # W^T -> W: by (a, j)
    indptr = torch.searchsorted(keys, torch.arange(n + 1, device=dev, dtype=torch.int64) * n)
    return (indptr, cols[order].to(torch.int32), wt_data[:nnz][order]), sweeps
