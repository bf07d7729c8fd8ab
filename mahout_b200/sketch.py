"""Host-side mirror of the reference's sketch operator API over the C ABI.

Same names, argument meaning and error behaviour as the fork's Java classes
(mr/src/main/java/org/apache/mahout/cf/taste/impl/common/):

  HashFunctionBuilder(seed)                      HashFunctionBuilder.java:23-60
  HashFunction.hash(key)                         HashFunction.java:31-34
  DoubleCountMinSketch(w, d, hfb) / (delta, eps, hfb)
      .update(key, inc) .get(key) .cosine(a, b)  DoubleCountMinSketch.java:32-149
  SketchBank: E sketches sharing one builder     CosineCM.java:41-67 (one sketch per entity)

Everything computes on the GPU through libmahout_b200.so; nothing here has a CPU path.
Array arguments may be numpy arrays (host memory) or torch CUDA tensors (device memory).
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _native as N

_tls = threading.local()


class Context:
    """One mb200_ctx (one GPU, one stream set).  Calls on a context are serialised by the library."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        rc = N.lib().mb200_create(int(device), C.byref(h))
        if rc != N.OK:
            N.check(rc, None)
        self._h = h
        self.device = int(device)
        self.stream_ptr = None       # the caller's stream when set_stream was used

    @property
    def handle(self):
        if self._h is None:
            raise ValueError("context is closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None:
            try:
                N.lib().mb200_destroy(self._h)
            except Exception:   # interpreter shutdown: module globals are already gone
                pass
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def sync(self):
        N.check(N.lib().mb200_sync(self.handle), self.handle)

    def set_stream(self, cuda_stream: int | None):
        N.check(N.lib().mb200_set_stream(self.handle, C.c_void_p(cuda_stream or 0)), self.handle)
        self.stream_ptr = cuda_stream or None

    def set_option(self, option: int, value: int):
        """mb200_set_option (e.g. N.OPT_GROUP_MIN_EVENTS: bank-mode updates of at least that many events are
        grouped by entity on the device before K1)"""
        N.check(N.lib().mb200_set_option(self.handle, int(option), int(value)), self.handle)

    def set_profiling(self, on: bool):
        N.check(N.lib().mb200_set_profiling(self.handle, int(on)), self.handle)

    def reset_profile(self):
        N.check(N.lib().mb200_reset_profile(self.handle), self.handle)

    def kernel_time(self, kernel_id: int):
        ms, n = C.c_double(), C.c_int64()
        N.check(N.lib().mb200_kernel_time(self.handle, kernel_id, C.byref(ms), C.byref(n)), self.handle)
        return ms.value, n.value

    def stats(self) -> dict:
        """mb200_get_stats: device, SMs, kernels launched, workspace / staging bytes held, last fallback rows"""
        st = N.Stats()
        N.check(N.lib().mb200_get_stats(self.handle, C.byref(st)), self.handle)
        return {f: (getattr(st, f).decode() if f == "device_name" else getattr(st, f)) for f, _ in N.Stats._fields_}

    def launch_count(self) -> int:
        n = C.c_int64()
        N.check(N.lib().mb200_launch_count(self.handle, C.byref(n)), self.handle)
        return n.value


def bind_host_thread_to_gpu(device: int) -> bool:
    """Pin the calling process to the CPU cores local to `device` (NVML's affinity mask, intersected with
    what the process may use) so that the pinned host buffers it allocates afterwards are first-touched on
    the GPU's own NUMA node: with 8 ranks on a two-socket box, buffers on the wrong socket make the H2D
    copies of mb200_bank_update(MEM_HOST) cross the inter-socket link.  Returns False if nothing was done."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[device]) if vis else device
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        local = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        target = local & allowed
        if not target or target == allowed:
            return False
        os.sched_setaffinity(0, target)
        return True
    except Exception:
        return False


def default_context() -> Context:
    ctx = getattr(_tls, "ctx", None)
    if ctx is None or ctx._h is None:
        dev = 0
        try:
            import torch
            if torch.cuda.is_available():
                dev = torch.cuda.current_device()
        except Exception:
            pass
        ctx = Context(dev)
        _tls.ctx = ctx
    return ctx


# --------------------------------------------------------------------------------------------
# argument marshalling: numpy (host) or torch.cuda (device)
# --------------------------------------------------------------------------------------------
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


class _Arg:
    """Pointer + memory space of one array argument; keeps the converted array alive."""

    def __init__(self, x, np_dtype, torch_dtype_name, allow_none=False):
        self.keep = None
        self.ptr = None
        self.mem = None
        self.n = 0
        if x is None:
            if not allow_none:
                raise ValueError("array argument is None")
            return
        if _is_torch(x):
            import torch
            want = getattr(torch, torch_dtype_name)
            if not x.is_cuda:
                x = x.numpy()
            else:
                if x.dtype != want:
                    x = x.to(want)
                x = x.contiguous()
                self.keep, self.ptr, self.mem, self.n = x, C.c_void_p(x.data_ptr()), N.MEM_DEVICE, x.numel()
                return
        a = np.ascontiguousarray(x, dtype=np_dtype)
        self.keep, self.ptr, self.mem, self.n = a, C.c_void_p(a.ctypes.data), N.MEM_HOST, a.size


def _same_mem(*args):
    mems = {a.mem for a in args if a.mem is not None}
    if len(mems) > 1:
        raise ValueError("array arguments must all be host (numpy) or all device (torch.cuda)")
    return mems.pop() if mems else N.MEM_HOST


def _out(shape, np_dtype, torch_dtype_name, mem, device):
    if mem == N.MEM_DEVICE:
        import torch
        t = torch.empty(shape, dtype=getattr(torch, torch_dtype_name), device=f"cuda:{device}")
        return t, C.c_void_p(t.data_ptr())
    a = np.empty(shape, dtype=np_dtype)
    return a, C.c_void_p(a.ctypes.data)


# --------------------------------------------------------------------------------------------
# hash family
# --------------------------------------------------------------------------------------------
BIG_PRIME = 9223372036854775783  # HashFunctionBuilder.java:24


class HashFunctionBuilder:
    """`new HashFunctionBuilder(seed)`: parameters a_i, b_i = abs(nextLong()), abs(nextLong())
    drawn lazily, in iteration order, from one java.util.Random(seed)."""

    def __init__(self, seed: int):
        self.seed = int(seed)
        self._a = np.zeros(0, np.int64)
        self._b = np.zeros(0, np.int64)

    def params(self, depth: int):
        if depth > self._a.shape[0]:
            # the parameter stream is a pure function of (seed, index): regenerate the prefix
            a = np.zeros(depth, np.int64)
            b = np.zeros(depth, np.int64)
            N.check(N.lib().mb200_hash_params(self.seed, depth, a.ctypes.data_as(C.c_void_p),
                                              b.ctypes.data_as(C.c_void_p)))
            self._a, self._b = a, b
        return self._a[:depth].copy(), self._b[:depth].copy()

    def getHashFunction(self, iteration: int, size: int) -> "HashFunction":
        a, b = self.params(iteration + 1)
        return HashFunction(int(a[iteration]), int(b[iteration]), int(size))


class HashFunction:
    """h(key) = ((a*key + b) mod (2^63-25)) mod w, evaluated on the GPU."""

    def __init__(self, a: int, b: int, w: int, ctx: Context | None = None):
        self.a, self.b, self.w = int(a), int(b), int(w)
        self._ctx = ctx

    def hash(self, key):
        ctx = self._ctx or default_context()
        scalar = np.isscalar(key)
        k = _Arg(np.atleast_1d(key) if not _is_torch(key) else key, np.int64, "int64")
        out, optr = _out((k.n,), np.int32, "int32", k.mem, ctx.device)
        N.check(N.lib().mb200_hash_keys(ctx.handle, self.a, self.b, self.w, k.ptr, k.n, optr, k.mem),
                ctx.handle)
        return int(out[0]) if scalar else out


class IdentityHashBuilder:
    """a_i = 1, b_i = 0: h(key) = key mod w.  With keys renumbered 0..U-1 and w >= U every key owns its
    column, so a depth-1 "sketch" holds the exact vector (RowSimilarityJob's exact cosine on K1-K5)."""
    seed = None

    def params(self, depth: int):
        return np.ones(depth, np.int64), np.zeros(depth, np.int64)

    def getHashFunction(self, iteration: int, size: int) -> "HashFunction":
        return HashFunction(1, 0, int(size))


def cm_dims(delta: float, epsilon: float):
    """(w, d) of AbstractCountMinSketch(delta, epsilon); raises CMException on the rejected ranges."""
    w, d = C.c_int32(), C.c_int32()
    N.check(N.lib().mb200_cm_dims(float(delta), float(epsilon), C.byref(w), C.byref(d)))
    return w.value, d.value


# --------------------------------------------------------------------------------------------
# sketch bank
# --------------------------------------------------------------------------------------------
class SketchBank:
    """E count-min sketches of d x W counters sharing one HashFunctionBuilder, HBM-resident.

    frac_bits: counters are exact multiples of 2^-frac_bits (1 covers MovieLens-style
    half-star prefs); increments that are not raise InexactError at the next check."""

    def __init__(self, entities: int, width: int, depth: int, hfBuilder: HashFunctionBuilder | int = 42,
                 frac_bits: int = 1, ctx: Context | None = None):
        self.ctx = ctx or default_context()
        if not isinstance(hfBuilder, (HashFunctionBuilder, IdentityHashBuilder)):
            hfBuilder = HashFunctionBuilder(int(hfBuilder))
        self.hfBuilder = hfBuilder
        if not (0 < int(depth) <= N.MAX_DEPTH):
            raise ValueError(f"depth must be in (0, {N.MAX_DEPTH}] (got {depth})")
        a, b = hfBuilder.params(int(depth))
        self.a, self.b = a, b
        h = C.c_void_p()
        N.check(N.lib().mb200_bank_create_params(
            self.ctx.handle, int(entities), int(depth), int(width), a.ctypes.data_as(C.c_void_p),
            b.ctypes.data_as(C.c_void_p), int(frac_bits), C.byref(h)), self.ctx.handle)
        self._h = h
        self.E, self.w, self.d, self.frac_bits = int(entities), int(width), int(depth), int(frac_bits)

    @property
    def handle(self):
        if self._h is None:
            raise ValueError("bank is closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None and self.ctx._h is not None:
            try:
                N.lib().mb200_bank_destroy(self._h)
            except Exception:   # interpreter shutdown
                pass
        self._h = None

    __del__ = close

    def clear(self):
        N.check(N.lib().mb200_bank_clear(self.handle), self.ctx.handle)

    def dump(self, path: str):
        """checkpoint: shape, quantum, hash parameters and the raw counters (mb200_bank_dump)"""
        N.check(N.lib().mb200_bank_dump(self.handle, str(path).encode()), self.ctx.handle)

    @classmethod
    def load(cls, path: str, ctx: "Context | None" = None) -> "SketchBank":
        """a new bank with exactly the dumped state (mb200_bank_load)"""
        ctx = ctx or default_context()
        h = C.c_void_p()
        N.check(N.lib().mb200_bank_load(ctx.handle, str(path).encode(), C.byref(h)), ctx.handle)
        self = cls.__new__(cls)
        self.ctx, self._h, self.hfBuilder = ctx, h, None
        import struct
        with open(path, "rb") as f:
            head = f.read(8 + 8 + 16 + 8 + 16 * N.MAX_DEPTH)
        self.E, self.d, self.w, self.frac_bits, _ = struct.unpack_from("<qiiii", head, 8)
        self.a = np.frombuffer(head, np.int64, self.d, 40).copy()
        self.b = np.frombuffer(head, np.int64, self.d, 40 + 8 * N.MAX_DEPTH).copy()
        return self

    def update(self, entity, key, inc):
        """C[entity[t]][i][h_i(key[t])] += inc[t]; entity may be None when E == 1."""
        k = _Arg(key, np.int64, "int64")
        e = _Arg(entity, np.int64, "int64", allow_none=True)
        f64 = (inc.dtype == np.float64) if isinstance(inc, np.ndarray) else (
            _is_torch(inc) and str(inc.dtype) == "torch.float64")
        v = _Arg(inc, np.float64 if f64 else np.float32, "float64" if f64 else "float32")
        if v.n != k.n or (e.ptr is not None and e.n != k.n):
            raise ValueError("entity, key and inc must have the same length")
        mem = _same_mem(k, e, v)
        fn = N.lib().mb200_bank_update_f64 if f64 else N.lib().mb200_bank_update
        N.check(fn(self.handle, e.ptr, k.ptr, v.ptr, k.n, mem), self.ctx.handle)

    def update_u8(self, entity, key, quanta):
        """The update in the narrow wire format: uint32 entity / key, one byte of quanta per event
        (increment = quanta * 2^-frac_bits).  Same counters as update(), bit for bit."""
        k = _Arg(key, np.uint32, "int32")
        e = _Arg(entity, np.uint32, "int32", allow_none=True)
        v = _Arg(quanta, np.uint8, "uint8")
        if v.n != k.n or (e.ptr is not None and e.n != k.n):
            raise ValueError("entity, key and quanta must have the same length")
        mem = _same_mem(k, e, v)
        N.check(N.lib().mb200_bank_update_u8(self.handle, e.ptr, k.ptr, v.ptr, k.n, mem), self.ctx.handle)

    def read_i32(self, e0: int = 0, e1: int | None = None, device: bool = False):
        """counters of entities [e0, e1) as int32 quanta, shape [e1-e0, d, w]"""
        e1 = self.E if e1 is None else e1
        mem = N.MEM_DEVICE if device else N.MEM_HOST
        out, optr = _out((e1 - e0, self.d, self.w), np.int32, "int32", mem, self.ctx.device)
        N.check(N.lib().mb200_bank_read_i32(self.handle, e0, e1, optr, mem), self.ctx.handle)
        return out

    def update_grouped(self, row_ptr, key, inc):
        """The update for events already grouped by entity (CSR: entity e owns [row_ptr[e], row_ptr[e+1])) --
        one PreferenceArray per entity, as CosineCM.exportProfile walks them (CosineCM.java:41-58)."""
        r = _Arg(row_ptr, np.int64, "int64")
        k = _Arg(key, np.int64, "int64")
        v = _Arg(inc, np.float32, "float32")
        if r.n != self.E + 1 or v.n != k.n:
            raise ValueError("row_ptr must have entities + 1 entries; key and inc the same length")
        mem = _same_mem(r, k, v)
        N.check(N.lib().mb200_bank_update_grouped(self.handle, r.ptr, k.ptr, v.ptr, k.n, mem), self.ctx.handle)

    def check(self):
        N.check(N.lib().mb200_bank_check(self.handle), self.ctx.handle)

    def read(self, e0: int = 0, e1: int | None = None, device: bool = False):
        """Counters of entities [e0, e1) as the reference's doubles, shape [e1-e0, d, w]."""
        e1 = self.E if e1 is None else e1
        if not (0 <= e0 <= e1 <= self.E):
            raise ValueError(f"bad entity range [{e0},{e1}) of {self.E}")
        out, optr = _out((e1 - e0, self.d, self.w), np.float64, "float64",
                         N.MEM_DEVICE if device else N.MEM_HOST, self.ctx.device)
        N.check(N.lib().mb200_bank_read(self.handle, e0, e1, optr,
                                        N.MEM_DEVICE if device else N.MEM_HOST), self.ctx.handle)
        return out

    def query(self, entity, key):
        """DoubleCountMinSketch.get for n (entity, key) pairs."""
        k = _Arg(key, np.int64, "int64")
        e = _Arg(entity, np.int64, "int64", allow_none=True)
        mem = _same_mem(k, e)
        out, optr = _out((k.n,), np.float64, "float64", mem, self.ctx.device)
        N.check(N.lib().mb200_bank_query(self.handle, e.ptr, k.ptr, k.n, optr, mem), self.ctx.handle)
        return out

    def pair_cosine(self, ea, eb):
        """DoubleCountMinSketch.cosine(sketch[ea[t]], sketch[eb[t]]) in FP64."""
        a = _Arg(ea, np.int64, "int64")
        b = _Arg(eb, np.int64, "int64")
        if a.n != b.n:
            raise ValueError("ea and eb must have the same length")
        mem = _same_mem(a, b)
        out, optr = _out((a.n,), np.float64, "float64", mem, self.ctx.device)
        N.check(N.lib().mb200_bank_pair_cosine(self.handle, a.ptr, b.ptr, a.n, optr, mem),
                self.ctx.handle)
        return out

    # ---- all-pairs cosine + top-k (RowSimilarityJob / ItemSimilarityJob semantics) --------------
    def cosine_topk(self, k: int, threshold: float | None = None, exclude_self: bool = True,
                    dtype: str = "f16", precision: str = "rescored", device: bool = False):
        """Per entity, the k most similar entities under sketch cosine (min over depth rows).

        Returns (idx [E,k] int64, sim [E,k] float64, cnt [E] int32); unused slots are -1 / 0.
        threshold None == RowSimilarityJob.NO_THRESHOLD."""
        mem = N.MEM_DEVICE if device else N.MEM_HOST
        idx, pi = _out((self.E, k), np.int64, "int64", mem, self.ctx.device)
        sim, ps = _out((self.E, k), np.float64, "float64", mem, self.ctx.device)
        cnt, pc = _out((self.E,), np.int32, "int32", mem, self.ctx.device)
        N.check(N.lib().mb200_bank_cosine_topk(
            self.handle, int(k), float(threshold) if threshold is not None else 0.0, int(exclude_self),
            _DTYPES[dtype], _PRECISIONS[precision], pi, ps, pc, mem), self.ctx.handle)
        return idx, sim, cnt

    def normalize(self, dtype: str = "f16"):
        """K2: unit-norm 16-bit rows [d, E, ld] and validity words [d, valid_words(E)] (torch, device)."""
        import torch
        ld = int(N.lib().mb200_row_ld(self.w))
        vw = int(N.lib().mb200_valid_words(self.E))
        dev = f"cuda:{self.ctx.device}"
        rows = torch.empty((self.d, self.E, ld), dtype=torch.float16 if dtype == "f16" else torch.bfloat16,
                           device=dev)
        valid = torch.empty((self.d, vw), dtype=torch.int32, device=dev)
        torch.cuda.synchronize(self.ctx.device)
        N.check(N.lib().mb200_bank_normalize(self.handle, _DTYPES[dtype], C.c_void_p(rows.data_ptr()),
                                             C.c_void_p(valid.data_ptr())), self.ctx.handle)
        self.ctx.sync()
        return rows, valid

    def sign_info(self) -> bool:
        """after normalize(): did K2 see a negative counter (or a row norm >= 2^36 quanta)?  The exact-set
        precisions then work with absolute error bounds (mb200_cosine_args.mixed_sign)."""
        m = C.c_int32()
        N.check(N.lib().mb200_bank_sign_info(self.handle, C.byref(m)), self.ctx.handle)
        return bool(m.value)

    def counters_tensor(self):
        """The raw int64 fixed-point counters [E, d, w] as a torch view (plumbing: collectives)."""
        p, n = self.counters_ptr()
        return _as_tensor(p, n, self.ctx.device).view(self.E, self.d, self.w)

    def counters_ptr(self):
        p, n = C.c_void_p(), C.c_int64()
        N.check(N.lib().mb200_bank_counters(self.handle, C.byref(p), C.byref(n)), self.ctx.handle)
        return p.value, n.value


_DTYPES = {"f16": N.DTYPE_F16, "bf16": N.DTYPE_BF16}
_PRECISIONS = {"tensor": N.PRECISION_TENSOR, "rescored": N.PRECISION_RESCORED, "certified": N.PRECISION_CERTIFIED}


def cosine_topk_blocks(ctx: Context, a_rows, a_valid, b_rows, b_valid, depth: int, width: int, k: int,
                       a_id=(1, 0), b_id=(1, 0), threshold: float | None = None, exclude_self: bool = True,
                       dtype: str = "f16", precision: str = "tensor", a_counters=None, b_counters=None,
                       block_n: int = 0, want_dense: bool = False, out=None, mixed_sign: bool = False):
    """mb200_cosine_topk over device tensors: A rows [d, a_count, ld] against b_blocks gathered blocks
    B [blocks, d, b_count, ld].  Returns torch device tensors (idx, sim, cnt[, dense])."""
    import torch
    dev = f"cuda:{ctx.device}"
    a_count = a_rows.shape[1]
    blocks, b_count = b_rows.shape[0], b_rows.shape[2]
    if out is not None:
        idx, sim, cnt = out
    else:
        idx = torch.empty((a_count, k), dtype=torch.int64, device=dev)
        sim = torch.empty((a_count, k), dtype=torch.float64, device=dev)
        cnt = torch.empty((a_count,), dtype=torch.int32, device=dev)
    args = N.CosineArgs()
    args.a_rows, args.a_valid, args.a_count = a_rows.data_ptr(), a_valid.data_ptr(), a_count
    args.a_id_mul, args.a_id_off = a_id
    args.b_rows, args.b_valid, args.b_count, args.b_blocks = b_rows.data_ptr(), b_valid.data_ptr(), b_count, blocks
    args.b_id_mul, args.b_id_add = b_id
    args.depth, args.width, args.dtype, args.precision = depth, width, _DTYPES[dtype], _PRECISIONS[precision]
    args.k, args.threshold, args.exclude_self, args.block_n = k, (threshold or 0.0), int(exclude_self), block_n
    args.a_counters = a_counters.data_ptr() if a_counters is not None else None
    args.b_counters = b_counters.data_ptr() if b_counters is not None else None
    args.out_idx, args.out_sim, args.out_cnt = idx.data_ptr(), sim.data_ptr(), cnt.data_ptr()
    args.mixed_sign = int(bool(mixed_sign))
    dense = None
    if want_dense:
        bn = block_n or 256
        ldc = blocks * ((b_count + bn - 1) // bn) * bn
        dense = torch.full((a_count, ldc), float("nan"), dtype=torch.float32, device=dev)
        args.dense_out, args.dense_ld = dense.data_ptr(), ldc
        torch.cuda.synchronize(ctx.device)   # the fill runs on torch's stream, K3 writes on the context's

    import os
    import time
    dbg = os.environ.get("MB200_BENCH_DEBUG") is not None
    t0 = time.perf_counter()
    if dbg:
        torch.cuda.synchronize(ctx.device)
    t1 = time.perf_counter()
    N.check(N.lib().mb200_cosine_topk(ctx.handle, C.byref(args)), ctx.handle)   # complete on return
    t2 = time.perf_counter()
    if dbg:
        import sys
        ctx.sync()
        print(f"[bench debug] cosine_topk_blocks {precision}: sync before {1e3 * (t1 - t0):.2f} ms, call "
              f"{1e3 * (t2 - t1):.2f} ms, sync after {1e3 * (time.perf_counter() - t2):.2f} ms", file=sys.stderr)
    return (idx, sim, cnt, dense) if want_dense else (idx, sim, cnt)


class CosineJob:
    """mb200_cosine_begin / push / finish: the B side arrives in pieces (row chunks of an all-gather in
    flight, or peer blocks streamed through a ring).  All tensors are torch CUDA tensors; push only
    queues work on the context's stream."""

    def __init__(self, ctx: Context, a_rows, a_valid, depth: int, width: int, k: int, a_id=(1, 0),
                 threshold: float | None = None, exclude_self: bool = True, dtype: str = "f16",
                 precision: str = "tensor", block_n: int = 0, mixed_sign: bool = False):
        self.ctx, self.k, self.a_count = ctx, int(k), int(a_rows.shape[1])
        self._keep = [a_rows, a_valid]              # the job borrows these until finish
        args = N.CosineArgs()
        args.a_rows, args.a_valid, args.a_count = a_rows.data_ptr(), a_valid.data_ptr(), self.a_count
        args.a_id_mul, args.a_id_off = a_id
        args.depth, args.width, args.dtype, args.precision = depth, width, _DTYPES[dtype], _PRECISIONS[precision]
        args.k, args.threshold, args.exclude_self, args.block_n = k, (threshold or 0.0), int(exclude_self), block_n
        args.mixed_sign = int(bool(mixed_sign))
        self._args = args
        h = C.c_void_p()
        N.check(N.lib().mb200_cosine_begin(ctx.handle, C.byref(args), C.byref(h)), ctx.handle)
        self._h = h

    def push(self, b_rows, b_valid, id_mul: int = 1, id_add: int = 0, id_base: int = 0, ready=None,
             first_block: int = 0):
        """b_rows [blocks, d, b_count, ld], b_valid [blocks, d, valid_words(b_count)];
        global index of row l of block g = l * id_mul + g * id_add + id_base.
        ready = (flags_ptr, epoch) from mb200_gather_pull: K3 waits for every block's arrival flag and
        sweeps the blocks starting with first_block."""
        pc = N.CosinePiece()
        pc.b_rows, pc.b_valid = b_rows.data_ptr(), b_valid.data_ptr()
        pc.b_blocks, pc.b_count = int(b_rows.shape[0]), int(b_rows.shape[2])
        pc.b_id_mul, pc.b_id_add, pc.b_id_base = int(id_mul), int(id_add), int(id_base)
        if ready is not None:
            pc.ready_flags, pc.ready_epoch, pc.first_block = ready[0], int(ready[1]), int(first_block)
        self._keep += [b_rows, b_valid]
        N.check(N.lib().mb200_cosine_push(self._h, C.byref(pc)), self.ctx.handle)

    def finish(self, a_counters=None, b_counters=None, b_id=(1, 0), out=None, counter_blocks=None, b_count=None,
               counter_blocks32=None, resident_b=None, defer_uncertified: bool = False):
        """Returns (idx, sim, cnt) device tensors.  precision="rescored" / "certified" need the resident
        counters: a_counters [a_count, d, w], b_counters [blocks, b_count, d, w] with b_id = (id_mul, id_add);
        "certified" alternatively takes counter_blocks, a ctypes array of one device pointer per block
        (peer-mapped banks of b_count rows each) instead of the gathered b_counters."""
        import torch
        dev = f"cuda:{self.ctx.device}"
        if out is None:
            out = (torch.empty((self.a_count, self.k), dtype=torch.int64, device=dev),
                   torch.empty((self.a_count, self.k), dtype=torch.float64, device=dev),
                   torch.empty((self.a_count,), dtype=torch.int32, device=dev))
        idx, sim, cnt = out
        fin = N.CosineArgs()
        fin.out_idx, fin.out_sim, fin.out_cnt = idx.data_ptr(), sim.data_ptr(), cnt.data_ptr()
        if resident_b is not None:
            # the (single) pushed piece is still where the push found it: uncertified rows may take the band pass
            fin.b_rows, fin.b_valid = resident_b[0].data_ptr(), resident_b[1].data_ptr()
        if a_counters is not None:
            fin.a_counters = a_counters.data_ptr()
            if counter_blocks is not None:
                fin.b_counter_blocks = C.cast(counter_blocks, C.c_void_p)
                if counter_blocks32 is not None:
                    fin.b_counter_blocks32 = C.cast(counter_blocks32, C.c_void_p)
                fin.b_blocks, fin.b_count = len(counter_blocks), int(b_count)
            else:
                fin.b_counters = b_counters.data_ptr()
                fin.b_blocks, fin.b_count = int(b_counters.shape[0]), int(b_counters.shape[1])
            fin.b_id_mul, fin.b_id_add = b_id
        if getattr(self, "_band_pending", None) is not None:
            # second finish of a deferred job: completes the band pass, writes the rows that were waiting
            idx, sim, cnt = self._band_pending
            h, self._h, self._band_pending = self._h, None, None
            N.check(N.lib().mb200_cosine_finish(h, C.byref(fin)), self.ctx.handle)
            self._keep = []
            return idx, sim, cnt
        fin.defer_uncertified = int(bool(defer_uncertified))
        rc = N.lib().mb200_cosine_finish(self._h, C.byref(fin))
        if rc == N.BAND_PENDING:
            # uncertified rows wait for a second round of pushes (the same pieces) and a second finish()
            self._band_pending = (idx, sim, cnt)
            self._keep += [a_counters, b_counters]
            return None
        h, self._h = self._h, None
        N.check(rc, self.ctx.handle)
        self._keep = []
        return idx, sim, cnt

    def abort(self):
        if getattr(self, "_h", None) is not None:
            N.lib().mb200_cosine_abort(self._h)
            self._h = None
            self._keep = []

    __del__ = abort


def last_band_rows(ctx: Context) -> int:
    n = C.c_int64()
    N.check(N.lib().mb200_cosine_last_band_rows(ctx.handle, C.byref(n)), ctx.handle)
    return n.value


def last_fallback_rows(ctx: Context) -> int:
    n = C.c_int64()
    N.check(N.lib().mb200_cosine_last_fallback_rows(ctx.handle, C.byref(n)), ctx.handle)
    return n.value


class DoubleCountMinSketch:
    """One sketch: `new DoubleCountMinSketch(w, d, hfBuilder)` or `(delta, epsilon, hfBuilder)`."""

    def __init__(self, width_or_delta, depth_or_epsilon, hfBuilder: HashFunctionBuilder,
                 frac_bits: int = 1, ctx: Context | None = None):
        if isinstance(width_or_delta, float) or isinstance(depth_or_epsilon, float):
            w, d = cm_dims(float(width_or_delta), float(depth_or_epsilon))
        else:
            w, d = int(width_or_delta), int(depth_or_epsilon)
        self.w, self.d = w, d
        self._bank = SketchBank(1, w, d, hfBuilder, frac_bits, ctx)
        self.hashFunctions = [hfBuilder.getHashFunction(i, w) for i in range(d)]

    def update(self, key, increment):
        k = np.atleast_1d(np.asarray(key, dtype=np.int64))
        v = np.atleast_1d(np.asarray(increment, dtype=np.float64))
        self._bank.update(None, k, np.broadcast_to(v, k.shape))

    def get(self, key):
        scalar = np.isscalar(key)
        out = self._bank.query(None, np.atleast_1d(np.asarray(key, dtype=np.int64)))
        return float(out[0]) if scalar else out

    def counts(self) -> np.ndarray:
        return self._bank.read()[0]

    @staticmethod
    def cosine(a: "DoubleCountMinSketch", b: "DoubleCountMinSketch") -> float:
        z = np.zeros(1, np.int64)
        out = np.empty(1, np.float64)
        N.check(N.lib().mb200_bank_cross_cosine(
            a._bank.handle, z.ctypes.data_as(C.c_void_p), b._bank.handle, z.ctypes.data_as(C.c_void_p),
            1, out.ctypes.data_as(C.c_void_p), N.MEM_HOST), a._bank.ctx.handle)
        return float(out[0])


def _as_tensor(ptr: int, n: int, device: int):
    """View n int64 device words at `ptr` as a torch tensor (plumbing only)."""
    import torch

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 3}
    return torch.as_tensor(h, device=f"cuda:{device}")
