"""B200-native WMF (implicit-feedback ALS) with the reference's Python surface.

Mirror of /root/reference/RecModel/wmf_model.py:8-351: same constructor, ``train``, ``predict``,
``rank``, ``recompute_factors*`` and inherited ``eval_prec`` / ``eval_topn`` signatures, argument
meaning, return types and error behaviour, so a script written against ``RecModel.WMF`` runs
unchanged. All arithmetic runs in hand-written sm_100a kernels behind the C ABI of
libwmf_b200.so (include/wmf_b200.h); this file only orchestrates. There is no CPU fallback.

Deliberate differences (documented, none changes results beyond rounding):
 * ``dtype`` must be float32 (the reference default); the device path computes in fp32.
 * ``cores`` is validated like the reference (ValueError below 1) and otherwise ignored: the
   reference's Pool paths compute the same numbers as the serial loop (SURVEY.md R6).
 * under ``torch.distributed`` (world size N > 1) rows are partitioned across the ranks and
   factor shards are all-gathered after every half-step (SURVEY.md §8e).
"""
import time

import numpy as np
import scipy.sparse
import torch

from . import _lib, engine, ranking, sharding
from .base_model import RecModel
from .engine import DeviceCSR

_ALGOS = {"auto": _lib.ALGO_AUTO, "simt": _lib.ALGO_SIMT, "tcgen05": _lib.ALGO_TCGEN05,
          "tcgen05_direct": _lib.ALGO_TCGEN05_DIRECT}


class WMF(RecModel):

    def __init__(self, num_items, num_users, dim, gamma, weighted=None, bias=False, seed=1993, dtype="float32",
                 device=None, algo="auto"):
        if np.dtype(dtype) != np.float32:
            raise ValueError(f"recmodel_b200.WMF computes in float32 on the device; dtype={dtype} is not supported")
        # wmf_model.py:11-17: global RNG seeded, float64 U[0,1) draw cast to dtype. Bit-reproduced on
        # the host with NumPy (MT19937 is not re-implemented on the GPU).
        np.random.seed(seed)
        self.bias = bias
        self.gamma = gamma
        self._device = device
        self._users_d = None
        self._items_d = None
        self._users_h = None
        self._items_h = None
        if self.bias is False:
            self._items_h = np.random.random((num_items, dim)).astype(dtype=dtype)
        elif self.bias is True:
            self._items_h = np.random.random((num_items, (dim + 1))).astype(dtype=dtype)
        self.num_users = num_users
        self.num_items = num_items
        self.dim = dim
        self.weighted = weighted
        self.dtype = dtype
        if algo not in _ALGOS:
            raise ValueError(f"algo must be one of {sorted(_ALGOS)}")
        self.algo = algo
        self.last_train_stats = {}
        # the confidence transform of the last train: (pre_process_count, alpha, beta, preprocess_mat), train's defaults
        # until then, so that a model with assigned factors folds in like a freshly trained one
        self._transform = ("log", 10, 1, False)

    # ---------------------------------------------------------------- factor storage (T2)
    @property
    def device(self):
        if self._device is None:
            self._device = engine.default_device()
        return torch.device(self._device)

    def _to_device(self, arr):
        return torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)).to(self.device)

    # ``users`` / ``items`` are plain ndarrays in the reference (wmf_model.py:15-18). Here the device tensor is the
    # source of truth and the getters hand out a cached host copy, marked READ-ONLY so that an in-place edit cannot be
    # silently ignored: assign a whole array (``m.items = new``) to change the factors.
    @property
    def items(self):
        if self._items_h is None and self._items_d is not None:
            self._items_h = engine.d2h(self._items_d)
            self._items_h.setflags(write=False)
        return self._items_h

    @items.setter
    def items(self, value):
        self._items_h = None if value is None else np.asarray(value)
        self._items_d = None

    @property
    def users(self):
        if self._users_h is None and self._users_d is not None:
            pre = getattr(self, "_users_prefetch", None)
            if pre is not None and pre[0] is self._users_d:  # read back while the item half-step was running
                pre[2].synchronize()
                self._users_h = pre[1].numpy()
            else:
                self._users_h = engine.d2h(self._users_d)
            self._users_h.setflags(write=False)
            self._users_prefetch = None
        return self._users_h

    @users.setter
    def users(self, value):
        self._users_h = None if value is None else np.asarray(value)
        self._users_d = None

    @property
    def items_device(self):
        if self._items_d is None and self._items_h is not None:
            self._items_d = self._to_device(self._items_h)
        return self._items_d

    @property
    def users_device(self):
        if self._users_d is None and self._users_h is not None:
            self._users_d = self._to_device(self._users_h)
        return self._users_d

    def _set_device_factors(self, users=None, items=None):
        if users is not None:
            self._users_d, self._users_h = users, None
        if items is not None:
            self._items_d, self._items_h = items, None

    # ---------------------------------------------------------------- rank (R10)
    def rank(self, items, users, topn=None):
        """Top-``topn`` of the candidate ``items`` for one user (or a list of users), best first
        (wmf_model.py:25-47). Index sets equal the reference's; ties are ordered by candidate
        position (the reference leaves tie order to argpartition/argsort)."""
        if topn is None:
            topn = len(items)
        if isinstance(users, list):
            ranked = self.rank_batch(items, np.asarray(users, dtype=np.int64), topn)
            return [ranked[k] for k in range(len(users))]
        if not type(items) == np.ndarray:
            items = np.array(items)
        return self.rank_batch(items, np.asarray([users], dtype=np.int64), topn)[0]

    def rank_batch(self, items, users, topn, distributed=False):
        """[len(users) x topn] ranked candidate ids for many users over one shared candidate list
        in a single device pass (the batched form of ``rank``). Like the reference's ``rank`` this is a LOCAL
        call by default, also under ``torch.distributed``. ``distributed=True`` is a COLLECTIVE: every rank of
        the default group must call it with the same arguments; each scores an equal slice of the users and the
        id lists are all-gathered (SURVEY.md 8e: users are independent, item factors replicated)."""
        items = np.asarray(items)
        ni = len(items)
        k = int(min(topn, ni))
        users_d = torch.from_numpy(np.ascontiguousarray(users, dtype=np.int64)).to(self.device)
        if ni == 0 or k == 0:
            return np.empty((len(users), 0), dtype=items.dtype)
        cand_d = torch.from_numpy(np.ascontiguousarray(items, dtype=np.int64)).to(self.device)
        ids = self._rank_ids(self.users_device, users_d, cand_d, k, None, distributed)
        return ids.cpu().numpy().astype(items.dtype, copy=False)

    def recommend(self, users, topn, exclude=None, distributed=False):
        """int64 [len(users) x topn]: the top-``topn`` of all items for each user, best first, leaving out the stored
        entries of row ``users[k]`` of ``exclude`` (users x items, any SciPy format or a DeviceCSR; every stored entry
        excludes its item whatever its value). Row k is ``rank(np.delete(np.arange(num_items), seen), users[k],
        topn)`` followed by -1 where the user has fewer than ``topn`` unseen items; ties go to the lower item id.
        ``exclude=None`` is ``rank_batch(np.arange(num_items), users, topn)``. ``distributed=True`` is a collective
        like in ``rank_batch``: each rank scores an equal slice of the users and the id lists are all-gathered."""
        V = self.items_device
        ni = V.shape[0]
        if exclude is None:
            return self.rank_batch(np.arange(ni, dtype=np.int64), users, topn, distributed=distributed)
        users = np.ascontiguousarray(users, dtype=np.int64).reshape(-1)
        if exclude.shape[1] != ni:
            raise ValueError(f"exclude has {exclude.shape[1]} columns but the model has {ni} items")
        if len(users) and (users.min() < 0 or users.max() >= exclude.shape[0]):
            raise ValueError(f"user ids must lie in [0, {exclude.shape[0]}) (the rows of exclude)")
        topn = int(topn)
        k = min(topn, ni)
        out = np.full((len(users), topn), -1, dtype=np.int64)
        if k <= 0 or len(users) == 0:
            return out
        ex = exclude if isinstance(exclude, DeviceCSR) else DeviceCSR.from_scipy(exclude, self.device)
        ids = self._recommend_ids(torch.from_numpy(users).to(self.device), k, ex.sorted(), distributed)
        out[:, :k] = ids.cpu().numpy()
        return out

    def _recommend_ids(self, users_d, k, ex, distributed=False):
        """Device int64 [len(users_d) x k], k <= num_items: the device part of ``recommend`` (``ex``: a DeviceCSR with
        sorted rows, or None to exclude nothing, where the lists are those of ``rank_batch`` over all items)."""
        return self._rank_ids(self.users_device, users_d, None, k, ex, distributed)

    def _rank_ids(self, U, users_d, cand_d, k, ex, distributed):
        """Device int64 [len(users_d) x k]: the lists of ``rank_batch`` for the rows ``users_d`` of the user factors U
        over the device candidate ids ``cand_d`` (None: all items), or, with ``ex`` (a DeviceCSR with sorted rows; needs
        ``cand_d`` None), those of ``recommend``. ``distributed`` as in ``rank_batch``; lists longer than TOPK_MAX are
        ranked locally."""
        V, bias = self.items_device, self.bias is True
        if k > _lib.TOPK_MAX:  # very long lists: exact device scores, then stable device sorts, many users per pass
            ni = V.shape[0] if cand_d is None else cand_d.numel()
            return ranking.sort_path_ids(users_d, ni, k, ex, lambda chunk, items_d: engine.predict_pairs(
                chunk.repeat_interleave(ni), items_d.repeat(chunk.numel()), U, V, bias=bias).view(chunk.numel(), ni),
                cand_d)

        def topk(u):
            if ex is None:
                return engine.score_topk(u, cand_d, U, V, k, bias=bias)
            return engine.score_topk_exclude(u, ex, U, V, k, bias=bias)[0]

        rank_id, world = sharding.dist_info()
        if not (distributed and world > 1):
            return topk(users_d)
        per = -(-users_d.numel() // world)
        mine = users_d[rank_id * per:(rank_id + 1) * per]
        local = torch.full((per, k), -1, dtype=torch.int64, device=self.device)
        if mine.numel():
            local[:mine.numel()] = topk(mine)
        ids = torch.empty((world * per, k), dtype=torch.int64, device=self.device)
        torch.distributed.all_gather_into_tensor(ids, local)
        return ids[:users_d.numel()]

    def eval_ranking(self, test_mat, topn=np.array([10]), exclude=None, users=None, distributed=False):
        """Full-ranking quality of ``recommend``: for each cutoff k of ``topn`` (an int or at most 16 distinct positive
        ints) a dict with "Recall@k", "Precision@k", "NDCG@k", "MAP@k" and "HitRate@k" (Python floats, means over the
        evaluated users) and "users" (their number). Unlike ``eval_topn``, which ranks each held-out item against
        ``rand_sampled`` random items and divides the hits by nnz(test), this ranks ALL items and averages per user.

        The list of user u is ``recommend(users, K, exclude)`` with K = max(topn) (ties to the lower item id, -1
        padding never a hit). T_u is the set of distinct columns of row u of ``test_mat`` with a stored non-zero value
        (duplicates count once; unsorted rows and explicit zeros are fine), h_i the hits among the first i items:
        Precision@k = h_k / k (k also when the list is padded), Recall@k = h_k / |T_u|, NDCG@k = the sum of
        1/log2(i+1) over the hits at i <= k over the same sum over i <= min(k, |T_u|) (binary gains), MAP@k = the sum
        of h_i / i over the hits at i <= k over min(k, |T_u|), HitRate@k = [h_k > 0]. Users with T_u empty are ranked
        but not counted; an item both in ``exclude`` and in T_u counts in |T_u| and can never be hit.

        ``test_mat`` and ``exclude`` (None: nothing excluded) are users x items SciPy matrices or DeviceCSRs, uploaded
        once. ``users`` defaults to the rows of ``test_mat`` with stored entries; repeated entries count each time.
        Lists, metrics and their sums stay on the device (the per-user rows are reduced once, in a fixed order: the
        result is bitwise reproducible). ``distributed=True`` is a collective like in ``recommend``: every rank gets
        the same result, bitwise equal to the local call."""
        return ranking.eval_ranking(
            lambda users_d, k, ex: self._recommend_ids(users_d, k, None if ex is None else ex.sorted(), distributed),
            lambda: (self.items_device.shape[0], self.users_device.shape[0]),
            "the rows of test_mat and of the user factors", self.device, test_mat, topn, exclude, users)

    # ---------------------------------------------------------------- fold-in (DESIGN.md 4.10)
    def _confidence(self, rows_d, counts):
        """The uploaded users x items DeviceCSR ``rows_d`` with the transform of the last ``train`` applied to its
        values: ``counts`` True for the count matrix of weighted training (always transformed), False for the
        utility matrix (transformed only with ``preprocess_mat``)."""
        mode, alpha, beta, preprocess_mat = self._transform
        if counts:
            return rows_d.with_data(engine.preprocess_(rows_d.data, mode, alpha, beta))
        if preprocess_mat == True and mode in ("log", "linear"):  # noqa: E712  (wmf_model.py:65-70)
            return rows_d.with_data(engine.preprocess_(rows_d.data.clone(), mode, alpha, beta))
        return rows_d

    def _fold_in_device(self, count_rows):
        """Device float32 [rows x f]: the user half-step of ``train`` for the rows of ``count_rows`` (new users x items
        SciPy, counts for weighted models, utilities otherwise) against the fixed item factors."""
        V = self.items_device
        if V is None:
            raise ValueError("the model has no item factors")
        if not scipy.sparse.issparse(count_rows) or count_rows.shape[1] != V.shape[0]:
            raise ValueError(f"count_rows must be a SciPy sparse matrix with {V.shape[0]} columns (the items), got "
                             f"{getattr(count_rows, 'shape', type(count_rows).__name__)}")
        if count_rows.shape[0] == 0:
            return torch.empty((0, V.shape[1]), dtype=torch.float32, device=self.device)
        weighted = self.weighted is True
        C = self._confidence(DeviceCSR.from_scipy(count_rows, self.device), counts=weighted)
        if not weighted:
            return engine.unweighted_half_step(C, V, self.gamma)                      # :85
        bias = self.bias is True
        G = engine.gram(V, self.gamma, ones_col0=bias)                                 # epoch.ResidentEpoch, stage 0
        return engine.half_step(C, V, G, bias=bias, algo=_ALGOS[self.algo])

    def fold_in(self, count_rows):
        """float32 [rows x f] (a new ndarray): the user factors of the new users whose histories are the rows of
        ``count_rows`` (new users x items, any SciPy format, in the form ``train`` takes: ``count_mat`` when weighted,
        ``utility_mat`` otherwise; not modified), solved against the fixed item factors. This is the user half-step of
        ``train`` with its confidence transform (pre_process_count, alpha, beta, preprocess_mat of the last ``train``,
        its defaults before one): a row's factors are bitwise those ``train`` gives the same row, whatever other rows
        share the call."""
        return self._fold_in_device(count_rows).cpu().numpy()

    def recommend_for(self, user_items, topn, exclude=True):
        """int64 [user_items.shape[0] x topn]: ``recommend`` for users that are not rows of the user factors. Row r is
        the top-``topn`` of all items for the user whose factors ``fold_in`` solves from row r of ``user_items``, best
        first, ties to the lower item id, -1 padding. ``exclude``: True leaves out each row's own stored entries
        (whatever their value), None nothing, a SciPy matrix or DeviceCSR of the shape of ``user_items`` its stored
        entries. A local call (no ``distributed``)."""
        return ranking.recommend_for(self._fold_in_device, self._fold_in_rank_ids, self.items_device.shape[0],
                                     self.device, user_items, topn, exclude)

    def eval_ranking_for(self, user_items, test_mat, topn=np.array([10]), exclude=True, users=None):
        """``eval_ranking`` (the same metrics and definitions) over the lists of ``recommend_for(user_items, K,
        exclude)``, K = max(topn): the strong-generalisation protocol, where the evaluated users are not rows of the
        user factors. ``test_mat`` has the shape of ``user_items``; ``users`` (ids into its rows) defaults to the rows of
        ``test_mat`` with stored entries. The factors are folded in once per call; no list leaves the device and the
        result is bitwise reproducible."""
        return ranking.eval_ranking_for(self._fold_in_device, self._fold_in_rank_ids, self.items_device.shape[0],
                                        self.device, user_items, test_mat, topn, exclude, users)

    def _fold_in_rank_ids(self, U, users_d, k, ex):
        return self._rank_ids(U, users_d, None, k, None if ex is None else ex.sorted(), False)

    # ---------------------------------------------------------------- train (R2, R7, R11)
    def train(self, utility_mat, iterations, verbose=0, eval_mat=None, count_mat=None, alpha=10,
              cores=4, stopping_rounds=3, dtype="float64", min_improvement=0.0001,
              pre_process_count="log", beta=1, preprocess_mat=False):
        """Same contract as wmf_model.py:49-189; returns the 0-based index of the last epoch run.
        Inputs are never mutated (the reference copies them, :54-56; here they are uploaded)."""
        if self.bias is True and self.weighted is False:
            print("Bias computation is only implemented for weighted matrix factorization.")
        if eval_mat is None and verbose > 1:
            print("Since no explicit evaluation was provided the train matrix is used for evaluation.")
            eval_mat = utility_mat
        rank_id, world = sharding.dist_info()
        dev = self.device
        t_start = self._t_train_start = time.perf_counter()

        self._transform = (pre_process_count, alpha, beta, preprocess_mat)
        util_d = None
        if preprocess_mat == True or verbose > 1 or self.weighted is not True:  # noqa: E712
            util_d = self._confidence(DeviceCSR.from_scipy(utility_mat, dev), counts=False)

        stats = {"half_step_ms": [], "eval_ms": [], "setup_ms": 0.0}
        if self.weighted is not True:
            it = self._train_unweighted(util_d, iterations, verbose, eval_mat, stopping_rounds, min_improvement, stats)
        else:
            if count_mat is None:
                raise AttributeError("'NoneType' object has no attribute 'data' (weighted training needs count_mat)")
            if pre_process_count not in ("log", "linear"):
                raise ValueError(f"Pre_process_count {pre_process_count} is not implement please use log or linear.")
            # Row-sharded runs: every rank uploads the whole matrix over its own PCIe link (in parallel, so no slower
            # than one GPU) and builds the transpose locally; only the epoch itself is sharded. Exchanging slices of
            # the matrix between the GPUs instead cost more than it saved (31 ms against 22 ms at 2 GPUs, round 1).
            C_full = DeviceCSR.from_scipy(count_mat, dev)
            stats["host_marks_ms"] = [("upload issued", (time.perf_counter() - t_start) * 1e3)]
            C_full = self._confidence(C_full, counts=True)
            CT_full = C_full.transpose()  # count_mat.T.tocsr()  (:128)
            stats["host_marks_ms"].append(("transpose issued", (time.perf_counter() - t_start) * 1e3))
            it = self._train_weighted(C_full, CT_full, util_d, iterations, verbose, eval_mat, cores, stopping_rounds,
                                      min_improvement, stats, rank_id, world)
        torch.cuda.synchronize(dev)
        stats["total_ms"] = (time.perf_counter() - t_start) * 1e3
        self.last_train_stats = stats
        return it

    def _eval_csr(self, mat, bounds=None, rank_id=0):
        if mat is None:
            raise AttributeError("'NoneType' object has no attribute 'nonzero' (train() needs eval_mat, as in the "
                                 "reference when verbose <= 1)")
        if isinstance(mat, DeviceCSR):
            return mat
        mat = mat.tocsr()
        if bounds is not None:
            mat = mat[int(bounds[rank_id]):int(bounds[rank_id + 1])]
        return DeviceCSR.from_scipy(mat, self.device)

    def _mse_device(self, eval_d, users_rows, distributed):
        sums = engine.sddmm_loss(eval_d, users_rows, self.items_device, bias=self.bias is True)
        if distributed:
            sharding.all_reduce_sum_(sums)
        s = sums.cpu().numpy()
        return np.float32(s[0] / s[2]) if s[2] > 0 else np.float32(np.nan)

    def _train_unweighted(self, R, iterations, verbose, eval_mat, stopping_rounds, min_improvement, stats):
        if self.items.shape[1] != self.dim:  # np.eye(self.dim) vs dim+1 columns (wmf_model.py:85)
            raise ValueError(f"operands could not be broadcast together with shapes ({self.items.shape[1]},"
                             f"{self.items.shape[1]}) ({self.dim},{self.dim})")
        RT = R.transpose()
        eval_d = self._eval_csr(eval_mat)
        last_mse, count_improvement = -np.inf, 0
        it = None
        for it in range(iterations):
            if verbose > 0:
                print(f"Starting fitting iteration {it}")
            users = engine.unweighted_half_step(R, self.items_device, self.gamma)      # :85
            self._set_device_factors(users=users)
            items = engine.unweighted_half_step(RT, users, self.gamma)                 # :88
            self._set_device_factors(items=items)
            mse_eval = self._mse_device(eval_d, self.users_device, False)
            if verbose > 0:
                print(f"Current eval mse is {mse_eval}")
            if verbose > 1:
                print(f"\tMSE Eval: {mse_eval}")
                print(f"\tMSE Train: {self.eval_prec(R)}")
            if mse_eval * (1 + min_improvement) > last_mse:
                count_improvement += 1
            else:
                count_improvement = 0
            last_mse = mse_eval
            if count_improvement >= stopping_rounds:
                break
        if it is None:
            raise UnboundLocalError("cannot access local variable 'iter' where it is not associated with a value")
        if verbose > 0:
            print("Training was completed.")
        if verbose > 1:
            print(f"MSE Eval at iteration {it}: {self.eval_prec(eval_d)}")
            print(f"MSE Train at iteration {it}: {self.eval_prec(R)}")
        return it

    def _train_weighted(self, C_full, CT_full, util_d, iterations, verbose, eval_mat, cores, stopping_rounds,
                        min_improvement, stats, rank_id, world):
        from .epoch import ResidentEpoch
        bias = self.bias is True
        algo = _ALGOS[self.algo]
        f = self.items.shape[1] if self.items is not None else self.dim
        distributed = world > 1
        if distributed:
            ucounts = (C_full.indptr[1:] - C_full.indptr[:-1]).cpu().numpy()
            icounts = (CT_full.indptr[1:] - CT_full.indptr[:-1]).cpu().numpy()
            ub = sharding.balanced_row_partition(ucounts, world, f, align=engine.gram_block_rows(len(ucounts)))
            ib = sharding.balanced_row_partition(icounts, world, f, align=engine.gram_block_rows(len(icounts)))
            C = C_full.row_slice(int(ub[rank_id]), int(ub[rank_id + 1]))
            CT = CT_full.row_slice(int(ib[rank_id]), int(ib[rank_id + 1]))
            u_lo, u_hi = int(ub[rank_id]), int(ub[rank_id + 1])
        else:
            C, CT, ub, ib = C_full, CT_full, None, None
            u_lo, u_hi = 0, C_full.shape[0]
        # the epoch's stages (half-step | exchange / Gram | half-step | exchange / Gram), launched eagerly:
        # wmf_model.py:140-156. Row-sharded, the exchange runs over peer memory when it is available.
        t_mark = time.perf_counter()
        stats.setdefault("host_marks_ms", []).append(("partition done", (t_mark - self._t_train_start) * 1e3))
        loop = ResidentEpoch(C, CT, self.items_device, self.gamma, bias=bias, algo=algo, ub=ub, ib=ib, graphs=False,
                             count_launches=False, shared_ws=True)
        stats.setdefault("host_marks_ms", []).append(("epoch object ready (+ms)", (time.perf_counter() - t_mark) * 1e3))
        eval_d = None  # uploaded on a side stream so a bad eval_mat fails where the reference fails (:163)
        stats["setup_ms"] = 0.0
        stats["exchange"] = loop.exchange_mode
        last_mse, count_improvement = -np.inf, 0
        it = None
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        side = getattr(self, "_side_stream", None)
        if side is None:
            side = self._side_stream = torch.cuda.Stream(device=self.device)
        eval_ready = None
        self._users_prefetch = None
        for it in range(iterations):
            if verbose > 0:
                print(f"Starting fitting iteration {it}")
            if cores < 1:
                raise ValueError(f"Values of cores has to be positive not {cores}")
            if self.bias is not True and self.bias is not False:
                raise ValueError(f"self.bias = {self.bias} is unknown. Only True / False are allowed.")
            start = time.time()
            ev[0].record()
            loop.run_stage(0)           # users from items (:143 / :151)
            loop.run_stage(1)           # Gram of the new users (+ exchange of the shards)
            users = loop.users
            self._set_device_factors(users=users)
            ev[1].record()
            if it == iterations - 1:
                # last epoch: the user factors are final, read them back while the item half-step runs
                side.wait_event(ev[1])
                with torch.cuda.stream(side):
                    host = torch.empty(users.shape, dtype=users.dtype, pin_memory=True)
                    host.copy_(users, non_blocking=True)
                    done = torch.cuda.Event()
                    done.record(side)
                users.record_stream(side)
                self._users_prefetch = (users, host, done)
            loop.run_stage(2)           # items from users (:144 / :152)
            loop.run_stage(3)           # Gram of the new items for the next epoch (+ exchange of the shards)
            self._set_device_factors(items=loop.items)
            ev[2].record()
            if eval_d is None and eval_mat is not None:
                # the evaluation matrix goes up on a side stream while the epoch issued above runs (its host-side
                # slicing and staging copy would otherwise sit between two stages and leave the GPU idle; a missing
                # matrix still fails below, where the reference fails, :163)
                with torch.cuda.stream(side):
                    eval_d = self._eval_csr(eval_mat, ub, rank_id)
                    eval_ready = torch.cuda.Event()
                    eval_ready.record(side)
            if eval_d is None:
                eval_d = self._eval_csr(eval_mat, ub, rank_id)
            if eval_ready is not None:
                cur = torch.cuda.current_stream(self.device)
                cur.wait_event(eval_ready)
                for t in (eval_d.indptr, eval_d.indices, eval_d.data):
                    t.record_stream(cur)
                eval_ready = None
            stats["host_marks_ms"].append((f"epoch {it} issued (+ms)", (time.perf_counter() - t_mark) * 1e3))
            mse_eval = self._mse_device(eval_d, self.users_device[u_lo:u_hi], distributed)
            ev[3].record()
            torch.cuda.synchronize(self.device)
            stats["host_marks_ms"].append((f"epoch {it} done (+ms)", (time.perf_counter() - t_mark) * 1e3))
            stats["half_step_ms"].append((ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])))
            stats["eval_ms"].append(ev[2].elapsed_time(ev[3]))
            if bias and cores == 1:
                print(f"Iteration {it} took {round(time.time() - start, 4)} seconds.")  # :153
            if mse_eval * (1 + min_improvement) > last_mse:
                count_improvement += 1
            else:
                count_improvement = 0
            last_mse = mse_eval
            if verbose > 0:
                print(f"Current eval mse is {mse_eval}")
            if verbose > 1:
                print(f"\tMSE Eval: {mse_eval}")
                print(f"\tMSE Train: {self.eval_prec(util_d)}")
            if count_improvement >= stopping_rounds:
                break
        if it is None:
            raise UnboundLocalError("cannot access local variable 'iter' where it is not associated with a value")
        if loop.px is not None:
            # the symmetric buffers are shared with the next training of the same shape: the model keeps its own copy
            # (the read-back of the users already in flight reads the buffer, which nothing overwrites before the
            # synchronisation at the end of train())
            self._items_d = loop.items.clone()
            if self._users_prefetch is None:
                self._users_d = loop.users.clone()
            else:
                keep = loop.users.clone()
                self._users_prefetch = (keep, self._users_prefetch[1], self._users_prefetch[2])
                self._users_d = keep
        if verbose > 0:
            print("Training was completed.")
        if verbose > 1:
            print(f"MSE Eval at iteration {it}: {self.eval_prec(eval_mat)}")
            print(f"MSE Train at iteration {it}: {self.eval_prec(util_d)}")
        return it

    # ---------------------------------------------------------------- eval_prec (R9)
    def eval_prec(self, utility_mat, metric="mse"):
        """MSE / RMSE / MAE over the non-zero stored entries (base_model.py:150-179), one fused
        device pass; returns a float32 scalar like the reference."""
        metric = metric.upper()
        if metric not in ("MSE", "RMSE", "MAE"):
            raise ValueError("Metric {metric} is not implemented.")
        csr = self._eval_csr(utility_mat)
        s = engine.sddmm_loss(csr, self.users_device, self.items_device, bias=self.bias is True).cpu().numpy()
        if s[2] == 0:
            return np.float32(np.nan)
        if metric == "MAE":
            return np.float32(s[1] / s[2])
        mse = s[0] / s[2]
        return np.float32(np.sqrt(mse)) if metric == "RMSE" else np.float32(mse)

    # ---------------------------------------------------------------- eval_topn (R12, SURVEY.md 8f N2)
    def eval_topn(self, test_mat, train_mat=None, eval_mat=None, topn=[10], rand_sampled=1000, cores=1,
                  random_state=None, dtype="float32"):
        """Sampled Recall@N with the reference's protocol and RNG draw order (base_model.py:51-148), all
        held-out interactions ranked in one device pass instead of one ``rank`` call each: per user the
        candidate list and the slot are drawn on the host exactly as ``compute_hit`` does (:79-80), the
        list is scored once (bit-exact ``predict`` scores), and ``item in top[:k]`` becomes "fewer than k
        candidates are ranked ahead of it" (``wmf_rank_ahead``; ties by position like ``rank``).
        ``RecModel.eval_topn(self, ...)`` is the per-interaction host loop with the same results. This is the
        reference's sampled protocol (hits / nnz(test)); ``eval_ranking`` ranks all unseen items and averages per user."""
        for other in (train_mat, eval_mat):
            if other is not None and other.shape != test_mat.shape:
                raise ValueError("inconsistent shapes")  # what `test_mat + other` raises (:115-120)
        if random_state is not None:
            np.random.seed(random_state)
        if not isinstance(topn, np.ndarray):
            raise ValueError("Topn has to be a np.array")
        test_mat = test_mat.tocsr()
        indptr = np.asarray(test_mat.indptr, dtype=np.int64)
        counts = np.diff(indptr)
        with_test = np.flatnonzero(counts > 0)
        L = int(rand_sampled) + 1
        kmax = int(topn.max())
        cand = np.empty((len(with_test), L), dtype=np.int32)
        slot = np.empty(len(with_test), dtype=np.int32)
        for k in range(len(with_test)):  # the reference's draw order: users in row order, list then slot
            cand[k] = np.random.randint(0, self.num_items, size=(rand_sampled + 1))
            slot[k] = np.random.randint(0, rand_sampled - (2 * kmax))
        hits = np.zeros(topn.shape, dtype=np.int64)
        dev = self.device
        U, V, bias = self.users_device, self.items_device, self.bias is True
        topn_d = torch.from_numpy(np.ascontiguousarray(topn, dtype=np.int32)).to(dev)
        step = max(1, (1 << 25) // L)  # users per pass: at most 32 M list scores resident
        for k0 in range(0, len(with_test), step):
            k1 = min(k0 + step, len(with_test))
            users = torch.from_numpy(with_test[k0:k1]).to(dev)
            cand_d = torch.from_numpy(cand[k0:k1]).to(dev)
            slot_d = torch.from_numpy(slot[k0:k1]).to(dev)
            S = engine.predict_pairs(users.repeat_interleave(L), cand_d.reshape(-1).to(torch.int64), U, V,
                                     bias=bias).reshape(k1 - k0, L)
            lo, hi = int(indptr[with_test[k0]]), int(indptr[with_test[k1 - 1] + 1])
            n_per = torch.from_numpy(counts[with_test[k0:k1]]).to(dev)
            pair_user = torch.arange(k1 - k0, device=dev, dtype=torch.int32).repeat_interleave(n_per)
            pair_item = torch.from_numpy(np.ascontiguousarray(test_mat.indices[lo:hi], dtype=np.int32)).to(dev)
            pair_score = engine.predict_pairs(users[pair_user.long()], pair_item.to(torch.int64), U, V, bias=bias)
            ahead = engine.rank_ahead(S, cand_d, slot_d, pair_user, pair_item, pair_score)
            hits += (ahead[:, None] < topn_d[None, :]).sum(0).cpu().numpy()
        recall = hits.astype(dtype) / len(test_mat.nonzero()[0])
        return {f"Recall@{topn[pos]}": recall[pos] for pos in range(len(topn))}

    # ---------------------------------------------------------------- predict (R8)
    def predict(self, users, items):
        """Scores f(user_k, item_k); one user against many items broadcasts (wmf_model.py:191-211).
        Bit-exact with the reference: products rounded to fp32, NumPy's pairwise sum order, then
        + user bias + item bias."""
        if (type(users) == list or type(users) == np.ndarray) and (type(items) == list or type(items) == np.ndarray):
            if len(users) != len(items):
                if not (len(users) == 1 or len(items) == 0):
                    raise ValueError("users and items need to have the same length or only one user / item "
                                     "needs to be provided.")
        u = torch.from_numpy(np.atleast_1d(np.asarray(users)).astype(np.int64)).to(self.device)
        i = torch.from_numpy(np.atleast_1d(np.asarray(items)).astype(np.int64)).to(self.device)
        if i.numel() == 0:
            return np.empty(0, dtype=np.float32)
        if i.numel() == 1 and u.numel() > 1:
            i = i.expand(u.numel()).contiguous()
        return engine.predict_pairs(u, i, self.users_device, self.items_device, bias=self.bias is True).cpu().numpy()

    # ---------------------------------------------------------------- half-steps (R4, R5, R6)
    def _half_step_host(self, Y, C, lambda_reg, bias):
        Yd = self._to_device(Y)
        Cd = C if isinstance(C, DeviceCSR) else DeviceCSR.from_scipy(C, self.device)
        G = engine.gram(Yd, lambda_reg, ones_col0=bias)
        return engine.half_step(Cd, Yd, G, bias=bias, algo=_ALGOS[self.algo]).cpu().numpy()

    def recompute_factors(self, Y, C, lambda_reg):
        """X from Y for the count matrix C, no biases (wmf_model.py:213-240)."""
        return self._half_step_host(Y, C, lambda_reg, False)

    def recompute_factors_par(self, Y, C, lambda_reg, cores=4):
        """Pool variant (wmf_model.py:242-250): same numbers, so same kernel."""
        return self._half_step_host(Y, C, lambda_reg, False)

    def recompute_factors_bias(self, Y, C, lambda_reg, cores=1):
        """Bias formula (wmf_model.py:311-351). Like the reference (:331) the caller's Y has its
        column 0 set to 1 afterwards; the kernel itself reads the bias from the unmodified copy."""
        X = self._half_step_host(Y, C, lambda_reg, True)
        if isinstance(Y, np.ndarray) and Y.flags.writeable:
            Y[:, 0] = 1
        return X

    def recompute_factors_bias_par(self, Y, C, lambda_reg, cores=3):
        """Pool variant of the bias half-step (wmf_model.py:252-265)."""
        return self.recompute_factors_bias(Y, C, lambda_reg)


WMFModel = WMF  # BASELINE.json's name for the class (SURVEY.md D1)
