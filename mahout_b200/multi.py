"""One process, all GPUs of the box: the item-similarity phase behind one C call (csrc/job.cu).

Mirror of what a JVM does through JNI for `--numGpus`: `MultiGpu(n)` is `mb200_create_multi`, `item_similarity`
is `mb200_job_item_similarity` = phase 1 of ItemSimilarityJob.run (ItemSimilarityJob.java:146-162).  The
one-process-per-GPU path over torch.distributed (similarity.sharded_item_similarity) computes the same thing for
callers that already run one rank per GPU.

`sized_bank` is CosineCM with a CountMinSketchConfig on every GPU of the handle (csrc/sized_multi.cu): one
replica of the sized bank per GPU, query users split t mod G, results bit-identical to `SizedBank`'s.

`item_based` is RecommenderJob's aggregate-and-recommend phase on every GPU of the handle (csrc/itembased_multi.cu):
one replica of the item top-k lists and the user vectors per GPU, query users split t mod G, results byte-identical
to `itembased.recommend` on one context.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from . import sketch as sk
from .sketch import _DTYPES, _PRECISIONS, HashFunctionBuilder, IdentityHashBuilder


class MultiGpu:
    def __init__(self, n_gpus: int = 0, devices=None):
        h = C.c_void_p()
        dv = None
        if devices is not None:
            dv = np.ascontiguousarray(devices, np.int32)
            n_gpus = int(dv.shape[0])
        N.check(N.lib().mb200_create_multi(int(n_gpus), dv.ctypes.data_as(C.c_void_p) if dv is not None else None,
                                           C.byref(h)))
        self._h = h
        n = C.c_int32()
        N.lib().mb200_multi_gpus(h, C.byref(n))
        self.n_gpus = n.value
        self.devices = dv.tolist() if dv is not None else list(range(self.n_gpus))

    def close(self):
        if getattr(self, "_h", None) is not None:
            try:
                N.lib().mb200_multi_destroy(self._h)
            except Exception:
                pass
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc == N.OK:
            return
        s = N.lib().mb200_multi_last_error(self._h)
        msg = s.decode("utf-8", "replace") if s else ""
        if rc == N.ERR_BAD_ARG:
            raise ValueError(msg)
        if rc == N.ERR_OOM:
            raise MemoryError(msg)
        if rc in (N.ERR_INEXACT, N.ERR_RANGE):
            raise N.InexactError(rc, msg)
        raise N.NativeError(rc, msg)

    def item_similarity(self, row, key, pref, num_items: int, k: int = 100, threshold: float | None = None,
                        width: int = 4096, depth: int = 4, seed: int = 42, frac_bits: int = 1, dtype: str = "f16",
                        precision: str = "rescored", hash_params=None):
        """(idx [N,k] int64, sim [N,k] float64, cnt [N] int32, stats dict) for host arrays of prepared events
        (dense item rows, user keys, preferences).  hash_params = (a, b) replaces the seeded hash family
        (a = 1, b = 0, width = number of users: the exact measure)."""
        row = np.ascontiguousarray(row, np.int64)
        key = np.ascontiguousarray(key, np.int64)
        pref = np.ascontiguousarray(pref, np.float32)
        if not (row.shape == key.shape == pref.shape):
            raise ValueError("row, key and pref must have the same length")
        p = N.JobParams()
        p.k, p.threshold, p.width, p.depth, p.seed = int(k), float(threshold or 0.0), int(width), int(depth), int(seed)
        keep = None
        if hash_params is not None:
            keep = (np.ascontiguousarray(hash_params[0], np.int64), np.ascontiguousarray(hash_params[1], np.int64))
            p.hash_a, p.hash_b = keep[0].ctypes.data, keep[1].ctypes.data
        p.frac_bits, p.dtype, p.precision = int(frac_bits), _DTYPES[dtype], _PRECISIONS[precision]
        idx = np.empty((num_items, k), np.int64)
        sim = np.empty((num_items, k), np.float64)
        cnt = np.empty(num_items, np.int32)
        st = N.JobStats()
        self._check(N.lib().mb200_job_item_similarity(
            self._h, row.ctypes.data_as(C.c_void_p), key.ctypes.data_as(C.c_void_p), pref.ctypes.data_as(C.c_void_p),
            row.shape[0], int(num_items), C.byref(p), idx.ctypes.data_as(C.c_void_p), sim.ctypes.data_as(C.c_void_p),
            cnt.ctypes.data_as(C.c_void_p), C.byref(st)))
        del keep
        return idx, sim, cnt, {f: getattr(st, f) for f, _ in N.JobStats._fields_}

    def sized_bank(self, width, depth, hfBuilder, user_ptr, item, pref, frac_bits: int = 1) -> "MultiSizedBank":
        """SizedBank's inputs (host arrays): one replica of the sized bank on every GPU of this handle"""
        return MultiSizedBank(self, width, depth, hfBuilder, user_ptr, item, pref, frac_bits)

    def item_based(self, lists, uv, item_id) -> "MultiItemBased":
        """itembased.recommend's data -- the lists (idx [I, k], sim [I, k], cnt [I]) as cosine_topk or
        item_similarity return them, a UserVectors and item_id [I], host or device memory: one replica per GPU"""
        return MultiItemBased(self, lists, uv, item_id)

    def context(self, g: int = 0) -> sk.Context:
        """GPU g's context as a Context that the handle owns (close() on it does not destroy it)"""
        h = C.c_void_p()
        self._check(N.lib().mb200_multi_ctx(self._h, int(g), C.byref(h)))
        return _BorrowedContext(h, self.devices[g], self)

    def contexts(self):
        """the raw mb200_ctx handles of the GPUs, in order (launch counts, stats)"""
        out = []
        for g in range(self.n_gpus):
            h = C.c_void_p()
            N.lib().mb200_multi_ctx(self._h, g, C.byref(h))
            out.append(h)
        return out


class _BorrowedContext(sk.Context):
    """one of a MultiGpu's contexts; it lives as long as the handle, and reads as closed once the handle is"""

    def __init__(self, handle, device: int, owner: MultiGpu):
        self._handle, self.device, self.stream_ptr, self._owner = handle, int(device), None, owner

    @property
    def _h(self):
        return self._handle if getattr(self._owner, "_h", None) is not None else None

    def close(self):
        self._handle = None

    __del__ = close


def _host(a, dtype):
    if hasattr(a, "cpu"):
        a = a.cpu().numpy()
    return np.ascontiguousarray(np.atleast_1d(np.asarray(a)), dtype)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class MultiSizedBank:
    """CosineCM's per-user-sized sketches replicated on every GPU of a MultiGpu (mb200_sized_multi_*).  Each call
    splits its users between the GPUs -- query position t to GPU t mod G; estimates by distinct user -- and returns
    numpy arrays in the caller's order, bit-identical to the same SizedBank calls on one GPU."""

    def __init__(self, multi: MultiGpu, width, depth, hfBuilder, user_ptr, item, pref, frac_bits: int = 1):
        self.multi = multi
        if not isinstance(hfBuilder, (HashFunctionBuilder, IdentityHashBuilder)):
            hfBuilder = HashFunctionBuilder(int(hfBuilder))
        self.width = _host(width, np.int32)
        self.depth = _host(depth, np.int32)
        if self.width.shape != self.depth.shape:
            raise ValueError("width and depth must be 1-d arrays of one entry per user")
        dmax = int(self.depth.max()) if self.depth.size else 1
        if not (0 < dmax <= N.MAX_DEPTH):
            raise ValueError(f"depth must be in (0, {N.MAX_DEPTH}] (got {dmax})")
        self.a, self.b = hfBuilder.params(dmax)
        ptr, it, pr = _host(user_ptr, np.int64), _host(item, np.int64), _host(pref, np.float32)
        if ptr.shape[0] != self.width.shape[0] + 1 or it.shape != pr.shape:
            raise ValueError("user_ptr must have users + 1 entries; item and pref the same length")
        self.U, self.frac_bits = int(self.width.shape[0]), int(frac_bits)
        h = C.c_void_p()
        self._h = None
        multi._check(N.lib().mb200_sized_multi_create(multi._h, self.U, _p(self.width), _p(self.depth), _p(self.a),
                                                      _p(self.b), self.frac_bits, _p(ptr), _p(it), _p(pr), C.byref(h)))
        self._h = h

    @property
    def handle(self):
        if self._h is None:
            raise ValueError("bank is closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None and getattr(self.multi, "_h", None) is not None:
            try:
                N.lib().mb200_sized_multi_destroy(self._h)
            except Exception:   # interpreter shutdown
                pass
        self._h = None

    __del__ = close

    def neighborhood(self, query_rows, n: int, min_similarity: float = -np.inf):
        """SizedBank.neighborhood over all GPUs: (idx [q, n] int64, sim [q, n] float64, cnt [q] int32)"""
        q = _host(query_rows, np.int64)
        n = int(n)
        idx = np.empty((q.shape[0], max(n, 0)), np.int64)
        sim = np.empty((q.shape[0], max(n, 0)), np.float64)
        cnt = np.empty(q.shape[0], np.int32)
        self.multi._check(N.lib().mb200_sized_multi_neighborhood(self.handle, _p(q), q.shape[0], n,
                                                                 float(min_similarity), _p(idx), _p(sim), _p(cnt)))
        return idx, sim, cnt

    def recommend_users(self, users, n: int, min_similarity: float, item_ptr, item_col, item_ids, how_many: int,
                        include_known: bool = False):
        """each user's neighbourhood(n, min_similarity), then SizedBank.recommend over it, on the GPU that computed
        it: (items [m, how_many] int64, values [m, how_many] float32, counts [m] int32), unused slots -1 / 0"""
        us = _host(users, np.int64)
        ip, ic, ii = _host(item_ptr, np.int64), _host(item_col, np.int32), _host(item_ids, np.int64)
        if ip.shape[0] != self.U + 1:
            raise ValueError("item_ptr must be [U + 1] for the bank's U rows")
        m, h = us.shape[0], int(how_many)
        items = np.empty((m, max(h, 0)), np.int64)
        vals = np.empty((m, max(h, 0)), np.float32)
        cnt = np.empty(m, np.int32)
        self.multi._check(N.lib().mb200_sized_multi_recommend(
            self.handle, _p(us), m, int(n), float(min_similarity), _p(ip), _p(ic), ic.shape[0], _p(ii), ii.shape[0], h,
            int(bool(include_known)), _p(items), _p(vals), _p(cnt)))
        return items, vals, cnt

    def estimate_prefs(self, user, item_id, n: int, min_similarity: float = -np.inf):
        """doEstimatePreference for the pairs (user[t], item_id[t]) over each user's neighbourhood(n,
        min_similarity); float32 [q], NaN where there is no estimate"""
        u, it = _host(user, np.int64), _host(item_id, np.int64)
        if u.shape != it.shape:
            raise ValueError("user and item_id must have the same length")
        out = np.empty(u.shape[0], np.float32)
        self.multi._check(N.lib().mb200_sized_multi_estimate_prefs(self.handle, _p(u), _p(it), u.shape[0], int(n),
                                                                   float(min_similarity), _p(out)))
        return out

    def stats(self) -> dict:
        """the last call: {"work": queries (pairs for estimates) per GPU, "seconds": each GPU's worker wall clock,
        "wall_s": the call's wall clock}"""
        G = self.multi.n_gpus
        work = np.zeros(G, np.int64)
        secs = np.zeros(G, np.float64)
        wall = C.c_double()
        self.multi._check(N.lib().mb200_sized_multi_last_stats(self.handle, _p(work), _p(secs), C.byref(wall)))
        return {"work": work.tolist(), "seconds": secs.tolist(), "wall_s": wall.value}


class MultiItemBased:
    """The item top-k lists, the user vectors and the itemIDs replicated on every GPU of a MultiGpu
    (mb200_itembased_multi_*).  recommend splits its users between the GPUs -- query position t to GPU t mod G -- and
    returns numpy arrays in the caller's order, byte-identical to itembased.recommend on one GPU."""

    def __init__(self, multi: MultiGpu, lists, uv, item_id):
        self.multi = multi
        self._h = None
        idx, sim, cnt = (_host(x, t) for x, t in zip(lists, (np.int64, np.float64, np.int32)))
        ptr, prow, pval = _host(uv.user_ptr, np.int64), _host(uv.pref_row, np.int32), _host(uv.pref_val, np.float32)
        ids = _host(item_id, np.int64)
        n_items = cnt.shape[0]
        ld = idx.size // n_items if n_items else 1
        if idx.size != n_items * ld or sim.size != idx.size or ids.shape[0] != n_items or prow.shape != pval.shape \
                or ptr.shape[0] < 1:
            raise ValueError("lists must be idx / sim [I, k] and cnt [I], item_id [I]; pref_row and pref_val the same "
                             "length")
        self.num_items, self.num_users = n_items, ptr.shape[0] - 1
        h = C.c_void_p()
        multi._check(N.lib().mb200_itembased_multi_create(
            multi._h, _p(idx), _p(sim), _p(cnt), n_items, max(ld, 1), _p(ptr), _p(prow), _p(pval), self.num_users,
            prow.shape[0], _p(ids), C.byref(h)))
        self._h = h

    @property
    def handle(self):
        if self._h is None:
            raise ValueError("item-based recommender is closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None and getattr(self.multi, "_h", None) is not None:
            try:
                N.lib().mb200_itembased_multi_destroy(self._h)
            except Exception:   # interpreter shutdown
                pass
        self._h = None

    __del__ = close

    def recommend(self, users=None, how_many: int = 10, max_prefs_per_user: int = 10, boolean_data: bool = False,
                  allowed=None):
        """itembased.recommend for the user rows `users` (None: every user row) over all GPUs.  allowed: optional
        bit mask over item rows (itembased.allowed_mask).  Returns numpy (items [m, how_many] int64 itemIDs, values
        [m, how_many] float32, counts [m] int32); unused slots are -1 / 0."""
        us = np.arange(self.num_users, dtype=np.int64) if users is None else _host(users, np.int64)
        al = None
        if allowed is not None:
            al = np.ascontiguousarray(allowed.cpu().numpy() if hasattr(allowed, "cpu") else allowed).reshape(-1)
            if al.dtype.kind not in "iu" or al.dtype.itemsize != 4:
                raise ValueError("allowed must be 32-bit words")
            al = al.view(np.uint32)
            if al.shape[0] != (self.num_items + 31) // 32:
                raise ValueError(f"allowed must hold {(self.num_items + 31) // 32} words for {self.num_items} items")
        m, n = us.shape[0], int(how_many)
        items = np.empty((m, max(n, 0)), np.int64)
        vals = np.empty((m, max(n, 0)), np.float32)
        cnt = np.empty(m, np.int32)
        self.multi._check(N.lib().mb200_itembased_multi_recommend(
            self.handle, _p(us), m, n, int(max_prefs_per_user), int(bool(boolean_data)),
            _p(al) if al is not None else None, _p(items), _p(vals), _p(cnt)))
        return items, vals, cnt

    def stats(self) -> dict:
        """the last call: {"work": users per GPU (every user for create), "seconds": each GPU's worker wall clock,
        "wall_s": the call's wall clock}"""
        G = self.multi.n_gpus
        work = np.zeros(G, np.int64)
        secs = np.zeros(G, np.float64)
        wall = C.c_double()
        self.multi._check(N.lib().mb200_itembased_multi_last_stats(self.handle, _p(work), _p(secs), C.byref(wall)))
        return {"work": work.tolist(), "seconds": secs.tolist(), "wall_s": wall.value}
