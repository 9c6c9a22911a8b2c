"""Model-independent parts of ``recommend`` and ``eval_ranking``, shared by WMF and Ease: the exact-score sort path for
lists longer than the selection kernels take, and the full-ranking evaluation around a model's device ranking."""
import numpy as np
import torch

from . import engine
from .engine import DeviceCSR

EVAL_CHUNK_IDS = 1 << 25  # eval_ranking ranks users in chunks of at most this many list entries (32 M ids, 256 MB)


def sort_path_ids(users_d, ni, k, ex, scores):
    """Device int64 [len(users_d) x k]: each user's items 0..ni-1 in descending order of ``scores(chunk, items_d)``
    (a device [len(chunk) x ni] tensor of exact scores), ties to the lower item id, with the stored entries of row
    ``users_d[r]`` of ``ex`` (a DeviceCSR indexed by user id, or None) moved behind every unseen item and reported as
    -1. The users are scored in chunks of at most ~16 M (user, item) pairs."""
    dev = users_d.device
    rows = []
    per = max(1, (1 << 24) // ni)
    items_d = torch.arange(ni, dtype=torch.int64, device=dev)
    for u0 in range(0, users_d.numel(), per):
        chunk = users_d[u0:u0 + per]
        n = chunk.numel()
        order = torch.sort(scores(chunk, items_d), dim=1, descending=True, stable=True).indices
        if ex is None:
            rows.append(order[:, :k])
            continue
        lo, cnt = ex.indptr[chunk], ex.indptr[chunk + 1] - ex.indptr[chunk]
        total = int(cnt.sum())
        row = torch.repeat_interleave(torch.arange(n, device=dev), cnt, output_size=total)
        entry = torch.arange(total, device=dev) + torch.repeat_interleave(lo - (torch.cumsum(cnt, 0) - cnt),
                                                                         cnt, output_size=total)
        seen = torch.zeros((n, ni), dtype=torch.bool, device=dev)
        seen[row, ex.indices[entry].long()] = True
        # unseen first, each group in score order (a seen item never displaces an unseen one, whatever the scores)
        seen_sorted = seen.gather(1, order)
        regroup = torch.sort(seen_sorted.to(torch.uint8), dim=1, stable=True).indices[:, :k]
        rows.append(torch.where(seen_sorted.gather(1, regroup), -1, order.gather(1, regroup)))
    return torch.cat(rows) if rows else torch.empty((0, k), dtype=torch.int64, device=dev)


def eval_ranking(rank_ids, dims, users_what, device, test_mat, topn, exclude, users, chunk_ids=EVAL_CHUNK_IDS):
    """The full-ranking evaluation of ``WMF.eval_ranking`` / ``Ease.eval_ranking`` (see their docstrings) for a model
    whose ``rank_ids(users_d, k, ex)`` returns the device int64 [len(users_d) x k] lists of ``recommend`` (k <= the
    number of items; ex: the exclusion DeviceCSR, or None). ``dims()`` returns (items, users) of the model, read once
    ``topn`` is valid: user ids must lie below that number of users and the rows of ``test_mat``; ``users_what`` names
    what bounds them in the error message. The users are ranked in chunks of at most
    ``chunk_ids`` list entries (``eval_ranking_sums``)."""
    ks = np.asarray(topn)
    if ks.ndim == 0:
        ks = ks.reshape(1)
    if (ks.ndim != 1 or not 1 <= len(ks) <= 16 or not np.issubdtype(ks.dtype, np.integer) or ks.min() < 1
            or len(np.unique(ks)) != len(ks)):
        raise ValueError("topn must be an int or a 1-D sequence of at most 16 distinct positive ints")
    ks = ks.astype(np.int64)
    ni, n_users = dims()
    if test_mat.shape[1] != ni:
        raise ValueError(f"test_mat has {test_mat.shape[1]} columns but the model has {ni} items")
    if exclude is not None and tuple(exclude.shape) != tuple(test_mat.shape):
        raise ValueError(f"exclude has shape {tuple(exclude.shape)}, test_mat {tuple(test_mat.shape)}")
    n_ok = min(test_mat.shape[0], n_users)
    bad_users = ValueError(f"user ids must lie in [0, {n_ok}) ({users_what})")
    if users is not None:
        users = np.ascontiguousarray(users, dtype=np.int64).reshape(-1)
        if len(users) and (users.min() < 0 or users.max() >= n_ok):
            raise bad_users
    T = (test_mat if isinstance(test_mat, DeviceCSR) else DeviceCSR.from_scipy(test_mat, device)).sorted()
    ex = None
    if exclude is not None:
        ex = exclude if isinstance(exclude, DeviceCSR) else DeviceCSR.from_scipy(exclude, device)
    if users is None:
        users_d = torch.nonzero(T.indptr[1:] > T.indptr[:-1]).squeeze(1)
        if users_d.numel() and int(users_d[-1]) >= n_ok:
            raise bad_users
    else:
        users_d = torch.from_numpy(users).to(device)
    sums = eval_ranking_sums(rank_ids, ni, T, ex, users_d, ks, chunk_ids).cpu().numpy()
    count = int(sums[-1])
    out = {}
    for j, kk in enumerate(ks.tolist()):
        for m, name in enumerate(engine.TOPN_METRICS):
            out[f"{name}@{kk}"] = float(sums[j * 5 + m] / count) if count else float("nan")
    out["users"] = count
    return out


def eval_ranking_sums(rank_ids, ni, T, ex, users_d, ks, chunk_ids=EVAL_CHUNK_IDS):
    """The device part of ``eval_ranking`` (T: the test DeviceCSR with sorted rows; ex: the exclusion DeviceCSR or
    None; ks: int64 cutoffs): the users are ranked in chunks of at most ``chunk_ids`` list entries, each chunk's
    per-user metrics land in one buffer, and one reduce returns the device float64 [len(ks)*5 + 1] sums and the
    evaluated-user count, summed in a fixed order (bitwise reproducible). No ids leave the device."""
    device = users_d.device
    K = int(max(ks))
    k = min(K, ni)
    n = users_d.numel()
    per_user = torch.empty((n, len(ks), 5), dtype=torch.float64, device=device)
    chunk = max(1, chunk_ids // K)
    for u0 in range(0, n, chunk):
        part = users_d[u0:u0 + chunk]
        ids = rank_ids(part, k, ex)
        if k < K:  # cutoffs past the number of items: -1 padding, as recommend returns it
            ids = torch.cat((ids, torch.full((part.numel(), K - k), -1, dtype=torch.int64, device=device)), dim=1)
        engine.topn_metrics(ids, part, T, ks, out=per_user[u0:u0 + chunk])
    return engine.topn_metrics_reduce(per_user, len(ks))
