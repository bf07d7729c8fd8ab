"""Host side of the item-similarity path over the C ABI: what ItemSimilarityJob / RowSimilarityJob
do around the hot loop, with the hot loop (sketch build + all-pairs cosine + top-k) on the GPU.

Reference call stack being mirrored (SURVEY.md 3a):
  ItemSimilarityJob.run                       cf/taste/hadoop/similarity/item/ItemSimilarityJob.java:97-179
    PreparePreferenceMatrixJob                cf/taste/hadoop/preparation/PreparePreferenceMatrixJob.java:54-114
      ToEntityPrefsMapper  (text -> long,long,float)     cf/taste/hadoop/ToEntityPrefsMapper.java:56-76
      ItemIDIndexMapper / Reducer (idToIndex, min ID)     cf/taste/hadoop/item/ItemIDIndex*.java
      ToUserVectorsReducer (set(index, pref): last wins; minPrefsPerUser)
    RowSimilarityJob (cosine)                 math/hadoop/similarity/cooccurrence/RowSimilarityJob.java
    MostSimilarItemPairsMapper / Reducer      ItemSimilarityJob.java:181-232  ((minID,maxID) keys, dedup)

Single GPU: `item_similarity`.  One process per GPU (torch.distributed): `sharded_item_similarity`
-- items are sharded by index % G, every rank builds the sketches of its own items, the
normalised 16-bit rows are all-gathered (NCCL over NVLink) and each rank computes its block row of
the similarity matrix; no merge across GPUs is needed because a row's candidates all live on its
owner (SURVEY.md 8e).
"""
from __future__ import annotations

import numpy as np

from . import sketch as sk

LOCAL_COUNTERS_MAX_BYTES = 64 << 30      # PeerRows: local copies of the peers' int32 banks are held up to this size ...
LOCAL_COUNTERS_MIN_ROWS = 16384          # ... for shards of at least this many rows (below, the copies outlast K3) ...
LOCAL_COUNTERS_KEEP_FREE = 40 << 30      # ... and only if this much device memory stays free for the cosine workspaces
FUSED_RETRIES = [0]                      # fused_gather_cosine: sweeps repeated after a pull-gather time-out (this process)
NO_THRESHOLD = 4.9e-324          # RowSimilarityJob.NO_THRESHOLD = Double.MIN_VALUE (RowSimilarityJob.java:56)
DEFAULT_MAX_SIMILAR_ITEMS_PER_ITEM = 100   # ItemSimilarityJob.java:88
DEFAULT_MIN_PREFS_PER_USER = 1


# ------------------------------------------------------------------------------------------------
# ingest: PreparePreferenceMatrixJob runs on the GPU (mahout_b200/ingest.py over csrc/ingest.cu)
# ------------------------------------------------------------------------------------------------
def java_double_to_string(v: float) -> str:
    """Double.toString: the shortest digits that round-trip, decimal notation for 1e-3 <= |v| < 1e7, otherwise
    computerised scientific notation (`9.765625E-4`); what TextOutputFormat writes for the similarity."""
    import decimal
    import math
    if math.isnan(v):
        return "NaN"
    if math.isinf(v):
        return "Infinity" if v > 0 else "-Infinity"
    if v == 0.0:
        return "-0.0" if math.copysign(1.0, v) < 0 else "0.0"
    sign, digits, exp = decimal.Decimal(repr(float(v))).as_tuple()
    return _java_notation(sign, "".join(map(str, digits)), exp)


def java_float_to_string(v: float) -> str:
    """Float.toString: the shortest digits that round-trip through float32, with Double.toString's notation rules
    (`0.70710677`, `1.0E-4`, `9999999.0`, `1.0E7`); what RecommenderJob's text output writes for a value."""
    import math
    v = float(np.float32(v))
    if math.isnan(v) or math.isinf(v) or v == 0.0:
        return java_double_to_string(v)
    mant, e = np.format_float_scientific(np.float32(v), unique=True, trim="-").split("e")
    if len(mant.lstrip("-")) == 1 and abs(v) < 1.1754943508222875e-38:
        # a subnormal whose shortest form has one digit: Java prints d.d, the closest two digits (1.4E-45)
        mant, e = np.format_float_scientific(np.float32(v), precision=1, unique=False).split("e")
    sign = mant.startswith("-")
    digits = mant.lstrip("-").replace(".", "")
    return _java_notation(sign, digits, int(e) - len(digits) + 1)


def _java_notation(sign, digits: str, exp: int) -> str:
    """digits x 10^exp in Java's notation: decimal for 1e-3 <= |v| < 1e7, else computerised scientific"""
    stripped = digits.rstrip("0") or "0"
    exp += len(digits) - len(stripped)
    digits = stripped
    exp10 = len(digits) + exp - 1
    if -3 <= exp10 < 7:
        if exp10 >= 0:
            digits = digits.ljust(exp10 + 1, "0")
            out = digits[:exp10 + 1] + "." + (digits[exp10 + 1:] or "0")
        else:
            out = "0." + "0" * (-exp10 - 1) + digits
    else:
        out = digits[0] + "." + (digits[1:] or "0") + "E" + str(exp10)
    return ("-" if sign else "") + out


def most_similar_item_pairs(idx, sim, cnt, item_id=None):
    """MostSimilarItemPairsMapper / Reducer: per-row top-k entries -> (minID, maxID) keys, the
    duplicate of a symmetric pair collapses to one value; ordered by (a, b)
    (EntityEntityWritable.java:64-71)."""
    pairs = {}
    for r in range(idx.shape[0]):
        rid = int(item_id[r]) if item_id is not None else r
        for t in range(int(cnt[r])):
            c = int(idx[r, t])
            cid = int(item_id[c]) if item_id is not None else c
            key = (rid, cid) if rid < cid else (cid, rid)
            pairs.setdefault(key, float(sim[r, t]))
    return sorted((a, b, s) for (a, b), s in pairs.items())


# ------------------------------------------------------------------------------------------------
# single GPU
# ------------------------------------------------------------------------------------------------
def item_similarity(row, user, pref, num_items: int, k: int = DEFAULT_MAX_SIMILAR_ITEMS_PER_ITEM,
                    threshold: float | None = None, width: int = 4096, depth: int = 4, seed: int = 42,
                    frac_bits: int = 1, dtype: str = "f16", precision: str = "rescored", ctx=None,
                    device: bool = False):
    """Sketch build + all-pairs cosine + per-item top-k on one GPU.
    entity = item row, key = userID, increment = pref (SURVEY.md 8a5, item-similarity mode).
    device=True returns the lists as torch CUDA tensors (they stay in HBM for the item-based recommender)."""
    ctx = ctx or sk.default_context()
    bank = sk.SketchBank(num_items, width, depth, seed, frac_bits, ctx)
    try:
        bank.update(row, user, pref)
        bank.check()
        return bank.cosine_topk(k, threshold, True, dtype, precision, device=device)
    finally:
        bank.close()


def exact_item_similarity(row, user, pref, num_items: int, k: int = DEFAULT_MAX_SIMILAR_ITEMS_PER_ITEM,
                          threshold: float | None = None, frac_bits: int = 1, dtype: str = "f16",
                          precision: str = "rescored", ctx=None, ucol=None, num_users: int | None = None,
                          device: bool = False):
    """RowSimilarityJob with CosineSimilarity, exactly (RowSimilarityJob.java:478-559; no sketch, no
    --maxPrefs down-sampling): the users are renumbered 0..U-1 and every user owns one counter column
    (depth 1, width U, identity hash), so K1 writes the item x user matrix, K3 computes all pairs on the
    tensor cores and K5 re-scores the kept candidates in exact integer / FP64 arithmetic.
    The events must be de-duplicated (one pref per (user, item): `Events.prepare`).  device=True: as in
    item_similarity."""
    import torch
    ctx = ctx or sk.default_context()
    dev = f"cuda:{ctx.device}"
    if ucol is not None:
        col, width = ucol, max(int(num_users), 1)                     # dense user numbers from Events.prepare
    else:
        users, col = torch.unique(torch.as_tensor(user).to(dev), return_inverse=True)      # plumbing
        width = max(int(users.numel()), 1)
    bank = sk.SketchBank(num_items, width, 1, sk.IdentityHashBuilder(), frac_bits, ctx)
    try:
        bank.update(torch.as_tensor(row).to(dev), col, torch.as_tensor(pref).to(dev))
        bank.check()
        return bank.cosine_topk(k, threshold, True, dtype, precision, device=device)
    finally:
        bank.close()


# ------------------------------------------------------------------------------------------------
# item-hash sharding (one process per GPU)
# ------------------------------------------------------------------------------------------------
class ShardPlan:
    """owner(index) = index % G; local row = index // G; every shard is padded to the same size."""

    def __init__(self, num_items: int, world: int, rank: int):
        self.N, self.G, self.rank = int(num_items), int(world), int(rank)
        self.rows_per_shard = (self.N + self.G - 1) // self.G

    def owner(self, row):
        return np.asarray(row) % self.G

    def local_row(self, row):
        return np.asarray(row) // self.G

    def global_row(self, local, shard=None):
        shard = self.rank if shard is None else shard
        return np.asarray(local) * self.G + shard

    def my_events(self, row, *cols):
        """the events whose item this rank owns, with rows renumbered locally"""
        m = self.owner(row) == self.rank
        return (self.local_row(row[m]),) + tuple(c[m] for c in cols)

    def local_count(self, shard=None):
        shard = self.rank if shard is None else shard
        return max(0, (self.N - shard + self.G - 1) // self.G)

    def assemble(self, parts):
        """per-shard [rows_per_shard, ...] results (shard order) -> global row order [N, ...]"""
        first = np.asarray(parts[0])
        out = np.zeros((self.N,) + first.shape[1:], first.dtype)
        for g, part in enumerate(parts):
            n = self.local_count(g)
            out[g::self.G] = np.asarray(part)[:n]
        return out


class GpuShardBackend:
    """The product backend: every step is a C-ABI call on this rank's GPU."""

    def __init__(self, ctx=None):
        self.ctx = ctx or sk.default_context()
        self.device = f"cuda:{self.ctx.device}"

    def build(self, plan, local_row, key, inc, width, depth, seed, frac_bits):
        self.bank = sk.SketchBank(plan.rows_per_shard, width, depth, seed, frac_bits, self.ctx)
        self.bank.update(local_row, key, inc)
        self.bank.check()

    def normalized(self, dtype):
        return self.bank.normalize(dtype)            # rows [d, E_loc, ld], valid [d, vw] (torch, device)

    def counters(self):
        return self.bank.counters_tensor()

    def mixed_sign(self, precision, group=None) -> bool:
        """OR over all ranks of mb200_bank_sign_info (after K2); only the exact-set precisions need it"""
        if precision == "tensor":
            return False
        m = self.bank.sign_info()
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            import torch
            t = torch.tensor([int(m)], dtype=torch.int32, device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
            m = bool(t.item())
        return m

    def cosine(self, plan, a_rows, a_valid, b_rows, b_valid, k, threshold, dtype, precision,
               a_counters=None, b_counters=None, mixed_sign=False):
        idx, sim, cnt = sk.cosine_topk_blocks(
            self.ctx, a_rows, a_valid, b_rows, b_valid, self.bank.d, self.bank.w, k,
            a_id=(plan.G, plan.rank), b_id=(plan.G, 1) if plan.G > 1 else (1, plan.rows_per_shard),
            threshold=threshold, exclude_self=True, dtype=dtype, precision=precision,
            a_counters=a_counters, b_counters=b_counters, mixed_sign=mixed_sign)
        return idx, sim, cnt

    def begin(self, plan, a_rows, a_valid, k, threshold, dtype, precision, mixed_sign=False):
        """incremental form of `cosine` (mb200_cosine_begin / push / finish)"""
        return sk.CosineJob(self.ctx, a_rows, a_valid, self.bank.d, self.bank.w, k, a_id=(plan.G, plan.rank),
                            threshold=threshold, exclude_self=True, dtype=dtype, precision=precision,
                            mixed_sign=mixed_sign)

    def close(self):
        self.bank.close()


def _all_gather(t, world, group):
    """all_gather_into_tensor of equally shaped shards -> [world, *t.shape] (NCCL and gloo)."""
    import torch
    import torch.distributed as dist
    t = t.contiguous()
    flat = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(flat, t, group=group)
    return flat.view((world,) + tuple(t.shape))


class EventRouter:
    """The exchange step of the sharded ingest on the GPUs (csrc/route.cu): every rank owns receive columns
    (row, key, inc) of `capacity` events in peer-accessible memory, mapped by all the others (CUDA IPC over
    NVLink).  `route` = count by owner, exchange of the G x G count matrix (the only collective: G int64 per
    rank), one kernel that partitions this rank's events by owner in shared memory and stores every run
    straight into its owner's columns, one stream-ordered barrier.  Collective; set up once, reused."""

    def __init__(self, ctx, plan, capacity: int, group=None):
        import ctypes as C
        import torch
        import torch.distributed as dist
        from . import _native as N
        from .ingest import _view
        self.ctx, self.plan, self.group, self.capacity = ctx, plan, group, int(max(capacity, 1))
        G = plan.G
        dev = f"cuda:{ctx.device}"
        self._own, handles = [], b""
        for width in (8, 8, 4):
            p, h = C.c_void_p(), (C.c_char * 64)()
            N.check(N.lib().mb200_peer_alloc(ctx.handle, self.capacity * width, C.byref(p), C.cast(h, C.c_void_p)), ctx.handle)
            self._own.append(p)
            handles += bytes(h)
        self.recv_row = _view(self._own[0].value, self.capacity, ctx.device, "<i8")
        self.recv_key = _view(self._own[1].value, self.capacity, ctx.device, "<i8")
        self.recv_inc = _view(self._own[2].value, self.capacity, ctx.device, "<f4")
        mine = torch.frombuffer(bytearray(handles), dtype=torch.uint8).to(dev)
        allh = torch.empty(G * 192, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, mine, group=group)
        allh = allh.cpu().numpy().tobytes()
        self._opened = []
        self.dst = [(C.c_void_p * G)() for _ in range(3)]
        for g in range(G):
            for j in range(3):
                if g == plan.rank:
                    self.dst[j][g] = self._own[j].value
                    continue
                q = C.c_void_p()
                hb = (C.c_char * 64).from_buffer_copy(allh[g * 192 + j * 64:g * 192 + (j + 1) * 64])
                N.check(N.lib().mb200_peer_open(ctx.handle, C.cast(hb, C.c_void_p), C.byref(q)), ctx.handle)
                self._opened.append(q)
                self.dst[j][g] = q.value
        self.token = torch.zeros(1, dtype=torch.int32, device=dev)

    def counts(self, row):
        """events of `row` per owner (host int64 [G]) and the all-gathered G x G matrix M[src][dst]"""
        import ctypes as C
        import torch
        import torch.distributed as dist
        from . import _native as N
        G = self.plan.G
        c = np.zeros(G, np.int64)
        N.check(N.lib().mb200_route_count(self.ctx.handle, C.c_void_p(row.data_ptr()), row.numel(), G,
                                          c.ctypes.data_as(C.c_void_p)), self.ctx.handle)
        mine = torch.from_numpy(c).to(row.device)
        allc = torch.empty(G * G, dtype=torch.int64, device=row.device)
        dist.all_gather_into_tensor(allc, mine, group=self.group)
        return c, allc.cpu().numpy().reshape(G, G)

    def route(self, row, user, pref, matrix=None):
        """-> this rank's (local_row, user, pref): views of the receive columns, valid until the next route()"""
        import ctypes as C
        import torch.distributed as dist
        from . import _native as N
        G, me = self.plan.G, self.plan.rank
        row, user, pref = row.contiguous(), user.contiguous(), pref.contiguous()
        if matrix is None:
            _, matrix = self.counts(row)
        total = int(matrix[:, me].sum())
        if int(matrix.sum(axis=0).max()) > self.capacity:
            raise ValueError(f"EventRouter: a shard receives {int(matrix.sum(axis=0).max())} events, capacity {self.capacity}")
        off = matrix[:me].sum(axis=0).astype(np.int64) if me > 0 else np.zeros(G, np.int64)
        off = np.ascontiguousarray(off)
        # the all-gather of the counts already ordered every rank's previous use of its columns before this
        N.check(N.lib().mb200_route_scatter(
            self.ctx.handle, C.c_void_p(row.data_ptr()), C.c_void_p(user.data_ptr()), C.c_void_p(pref.data_ptr()),
            row.numel(), G, C.cast(self.dst[0], C.c_void_p), C.cast(self.dst[1], C.c_void_p),
            C.cast(self.dst[2], C.c_void_p), off.ctypes.data_as(C.c_void_p)), self.ctx.handle)
        dist.all_reduce(self.token, group=self.group)          # every source has delivered
        return self.recv_row[:total], self.recv_key[:total], self.recv_inc[:total]

    def close(self):
        import torch
        import torch.distributed as dist
        from . import _native as N
        if getattr(self, "_own", None) is None:
            return
        torch.cuda.synchronize(self.ctx.device)
        dist.all_reduce(self.token, group=self.group)          # nobody is still writing into my columns
        torch.cuda.synchronize(self.ctx.device)
        self.recv_row = self.recv_key = self.recv_inc = None
        for q in self._opened:
            N.lib().mb200_peer_close(self.ctx.handle, q)
        for p in self._own:
            N.lib().mb200_peer_free(self.ctx.handle, p)
        self._own = None


def route_events_device(ctx, plan, row, user, pref, group=None, router: EventRouter | None = None):
    """route_events on the GPUs through an EventRouter (created, sized by the exchanged counts, when none is
    passed).  The context's stream must be the current torch stream (the NCCL barrier is ordered with the
    scatter kernel through it).  Returns (local_row, user, pref, router): the tensors alias the router's
    receive columns."""
    import torch
    dev = torch.device(f"cuda:{ctx.device}")
    row = torch.as_tensor(row).to(dev)
    user, pref = torch.as_tensor(user).to(dev), torch.as_tensor(pref).to(dev)
    matrix = None
    if router is None:
        # size the receive columns by what the largest shard receives
        probe = EventRouter.__new__(EventRouter)
        probe.ctx, probe.plan, probe.group = ctx, plan, group
        _, matrix = EventRouter.counts(probe, row.contiguous())
        router = EventRouter(ctx, plan, int(matrix.sum(axis=0).max()), group)
    lrow, luser, lpref = router.route(row, user, pref, matrix)
    return lrow, luser, lpref, router


def route_events(plan, row, user, pref, group=None):
    """The exchange step of a sharded ingest (SURVEY.md 8e) for HOST tensors (gloo; the CPU-side tests of the
    sharding logic): events travel to the owner of their item (owner = row % G) with one all-to-all of the
    20-byte events.  On GPUs the product path is `route_events_device` (csrc/route.cu).  Returns this rank's
    (local_row, user, pref) as torch tensors on the inputs' device; order within a source is kept."""
    import torch
    import torch.distributed as dist
    G = plan.G
    row = torch.as_tensor(row)
    dev = row.device
    user, pref = torch.as_tensor(user).to(dev), torch.as_tensor(pref).to(dev)
    if G == 1:
        return row // 1, user, pref
    owner = row % G
    order = torch.sort(owner, stable=True).indices
    send_counts = torch.bincount(owner, minlength=G)
    recv_counts = torch.empty_like(send_counts)
    dist.all_to_all_single(recv_counts, send_counts, group=group)
    sc, rc = send_counts.tolist(), recv_counts.tolist()
    out = []
    for t in (row, user, pref):
        src = t[order].contiguous()
        dst = torch.empty(sum(rc), dtype=t.dtype, device=dev)
        dist.all_to_all_single(dst, src, rc, sc, group=group)
        out.append(dst)
    return out[0] // G, out[1], out[2]


def pipelined_cosine(backend, plan, a_rows, a_valid, k, threshold, dtype, precision, group=None,
                     chunk_rows: int = 2048, a_counters=None, mixed_sign: bool = False, counter_blocks=None,
                     counter_blocks32=None):
    """C1 overlapped with K3 (SURVEY.md 8e): the all-gather of the normalised rows runs in row chunks on
    a communication stream, two chunks ahead of the compute stream, and every gathered chunk
    [G, d, rows_c, ld] is pushed into one incremental cosine job as soon as it has landed.  Only two
    chunk buffers are resident, so the gathered operand never exists as a whole (config 5).
    Chunk c covers local rows [c0, c1) of every shard: global index of (shard g, row l) = (c0 + l) * G + g.
    Returns this rank's (idx, sim, cnt)."""
    import torch
    import torch.distributed as dist
    G, E_loc = plan.G, plan.rows_per_shard
    d, ld = int(a_rows.shape[0]), int(a_rows.shape[2])
    chunk_rows = max(256, (int(chunk_rows) + 255) // 256 * 256)
    cuda = a_rows.is_cuda
    nbuf = 2
    rows_max = min(chunk_rows, (E_loc + 255) // 256 * 256)
    vw_of = lambda n: (n + 255) // 256 * 8                                  # mb200_valid_words
    bufs = [torch.empty(G * d * rows_max * ld, dtype=a_rows.dtype, device=a_rows.device) for _ in range(nbuf)]
    vbufs = [torch.empty(G * d * vw_of(rows_max), dtype=a_valid.dtype, device=a_valid.device) for _ in range(nbuf)]
    job = backend.begin(plan, a_rows, a_valid, k, threshold, dtype, precision, **({"mixed_sign": True} if mixed_sign else {}))
    if cuda:
        ctx = backend.ctx
        prev = ctx.stream_ptr
        comp = torch.cuda.Stream(a_rows.device) if prev is None else torch.cuda.ExternalStream(prev, a_rows.device)
        if prev is None:
            ctx.set_stream(comp.cuda_stream)
        comm = torch.cuda.Stream(a_rows.device)
        comm.wait_stream(torch.cuda.current_stream(a_rows.device))
        comm.wait_stream(comp)
        free = [None] * nbuf
    b_cnt = None
    import os
    import sys
    import time
    debug = os.environ.get("MB200_BENCH_DEBUG") is not None
    t_start = time.perf_counter()

    def note(what):
        if debug:
            if cuda:
                torch.cuda.synchronize(a_rows.device)
            print(f"[pipelined_cosine rank {plan.rank} +{time.perf_counter() - t_start:8.3f}s] {what}", file=sys.stderr, flush=True)

    def stream_pass(do_push: bool):
        """one sweep over the B side: chunk c of every shard is gathered while chunk c-1 is consumed"""
        for ci, c0 in enumerate(range(0, E_loc, chunk_rows)):
            c1 = min(E_loc, c0 + chunk_rows)
            n, vw = c1 - c0, vw_of(c1 - c0)
            b = ci % nbuf
            out = bufs[b][:G * d * n * ld].view(G, d, n, ld)
            vout = vbufs[b][:G * d * vw].view(G, d, vw)

            def gather():
                src = a_rows[:, c0:c1].contiguous()
                vsrc = torch.zeros((d, vw), dtype=a_valid.dtype, device=a_valid.device)
                words = a_valid[:, c0 // 32:(c1 + 31) // 32]
                vsrc[:, :words.shape[1]] = words
                dist.all_gather_into_tensor(out.view(G * d, n, ld), src, group=group)
                dist.all_gather_into_tensor(vout.view(G * d, vw), vsrc, group=group)

            if cuda:
                with torch.cuda.stream(comm):
                    if free[b] is not None:
                        comm.wait_event(free[b])                 # the push that read this buffer is done
                    gather()
                    landed = torch.cuda.Event()
                    landed.record(comm)
                comp.wait_event(landed)
                if do_push:
                    job.push(out, vout, id_mul=G, id_add=1, id_base=c0 * G)
                free[b] = torch.cuda.Event()
                free[b].record(comp)
            else:
                gather()
                if do_push:
                    job.push(out.clone(), vout.clone(), id_mul=G, id_add=1, id_base=c0 * G)

    try:
        stream_pass(True)
        note("first sweep queued and done")
        if precision != "tensor" and counter_blocks is not None:
            # the undecided candidates are read from their owners' banks through peer mappings
            # (PeerRows.map_counters): no counter is ever gathered -- what makes exact sets possible when the
            # bank of all shards (config 5: 10^7 x 4096 x 8 B) could not exist on one GPU.  Rows the candidate
            # lists cannot certify are deferred: the B side is streamed a second time for those rows only (band
            # pass) -- on every rank if any rank has such rows, because the all-gathers are collective.
            err = None
            try:
                res = job.finish(a_counters=a_counters, b_id=(G, 1), counter_blocks=counter_blocks,
                                 b_count=plan.rows_per_shard, counter_blocks32=counter_blocks32, defer_uncertified=True)
            except Exception as ex:          # e.g. MB200_OPT_MAX_FALLBACK_ROWS: every rank must learn of it
                err, res = ex, ()
            pending = torch.tensor([2 if err is not None else (1 if res is None else 0)], dtype=torch.int32,
                                   device=a_rows.device)
            if cuda:
                comp.synchronize()
                with torch.cuda.stream(comp):
                    dist.all_reduce(pending, op=dist.ReduceOp.MAX, group=group)
            else:
                dist.all_reduce(pending, op=dist.ReduceOp.MAX, group=group)
            state = int(pending.item())
            note(f"first finish: state {state} (0 done, 1 band pass pending somewhere, 2 failed), "
                 f"band rows here {sk.last_band_rows(backend.ctx) if cuda else 0}")
            if state == 2:
                raise err if err is not None else RuntimeError("pipelined_cosine: the certified finish failed on another rank")
            if state == 1:
                if cuda:
                    comm.wait_stream(comp)
                    free = [None] * nbuf
                stream_pass(res is None)
                note("band sweep done")
                err = None
                if res is None:
                    try:
                        res = job.finish()
                    except Exception as ex:
                        err = ex
                note(f"band finish done ({'ok' if err is None else repr(err)[:200]})")
                if not all_ranks_ok(err is None, a_rows.device, group):
                    raise err if err is not None else RuntimeError("pipelined_cosine: the band pass failed on another rank")
        elif precision != "tensor":
            # the exact re-score reads the counters of arbitrary peers: gathered whole, behind the rows
            if cuda:
                with torch.cuda.stream(comm):
                    b_cnt = _all_gather(a_counters, G, group)
                    done = torch.cuda.Event()
                    done.record(comm)
                comp.wait_event(done)
            else:
                b_cnt = _all_gather(a_counters, G, group)
            res = job.finish(a_counters=a_counters, b_counters=b_cnt, b_id=(G, 1))
        else:
            res = job.finish()
        if cuda:
            torch.cuda.current_stream(a_rows.device).wait_stream(comp)
            torch.cuda.current_stream(a_rows.device).wait_stream(comm)
        return res
    except BaseException:
        job.abort()
        raise
    finally:
        if cuda and prev is None:
            backend.ctx.sync()
            backend.ctx.set_stream(None)


class PeerRows:
    """This rank's normalised rows and validity words in peer-accessible device memory, the mapped
    buffers of every other rank (CUDA IPC over NVLink) and the local staging operand of the fused
    pull-gather (mb200_gather_pull).  Set up once per (shape, group); collective."""

    def __init__(self, ctx, plan, depth: int, width: int, dtype: str = "f16", group=None, staging: bool = True):
        import ctypes as C
        import torch
        import torch.distributed as dist
        from . import _native as N
        from .ingest import _view
        self.ctx, self.plan, self.group = ctx, plan, group
        G, E_loc = plan.G, plan.rows_per_shard
        ld = int(N.lib().mb200_row_ld(width))
        vw = int(N.lib().mb200_valid_words(E_loc))
        self.rows_bytes, self.valid_bytes = depth * E_loc * ld * 2, depth * vw * 4
        dev = f"cuda:{ctx.device}"
        self._own, handles = [], []
        for nbytes in (self.rows_bytes, self.valid_bytes):
            p, h = C.c_void_p(), (C.c_char * 64)()
            N.check(N.lib().mb200_peer_alloc(ctx.handle, nbytes, C.byref(p), C.cast(h, C.c_void_p)), ctx.handle)
            self._own.append(p)
            handles.append(bytes(h))
        tdt = torch.float16 if dtype == "f16" else torch.bfloat16
        self.rows = _view(self._own[0].value, self.rows_bytes // 2, ctx.device, "<i2").view(tdt).view(depth, E_loc, ld)
        self.valid = _view(self._own[1].value, self.valid_bytes // 4, ctx.device, "<i4").view(depth, vw)
        mine = torch.frombuffer(bytearray(handles[0] + handles[1]), dtype=torch.uint8).to(dev)
        allh = torch.empty(G * 128, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, mine, group=group)
        allh = allh.cpu().numpy().tobytes()
        self._opened = []
        self.peer_rows = (C.c_void_p * G)()
        self.peer_valid = (C.c_void_p * G)()
        for g in range(G):
            if g == plan.rank:
                self.peer_rows[g], self.peer_valid[g] = self._own[0].value, self._own[1].value
                continue
            for j, arr in enumerate((self.peer_rows, self.peer_valid)):
                q = C.c_void_p()
                hb = (C.c_char * 64).from_buffer_copy(allh[g * 128 + j * 64:g * 128 + (j + 1) * 64])
                N.check(N.lib().mb200_peer_open(ctx.handle, C.cast(hb, C.c_void_p), C.byref(q)), ctx.handle)
                self._opened.append(q)
                arr[g] = q.value
        # the local copy of every shard's rows the fused pull-gather sweeps; the streamed form (pipelined_cosine)
        # never holds the gathered operand and does without it
        self.staging_rows = torch.empty((G, depth, E_loc, ld), dtype=tdt, device=dev) if staging else None
        self.staging_valid = torch.empty((G, depth, vw), dtype=torch.int32, device=dev) if staging else None
        self.token = torch.zeros(1, dtype=torch.int32, device=dev)

    def map_counters(self, bank):
        """Map every rank's counter bank (CUDA IPC): `counter_blocks[g]` then points at shard g's counters
        [E_loc][d][w] -- MB200_PRECISION_CERTIFIED reads the few undecided candidates through them, so
        the counters are never gathered.  Collective; call after the banks are built."""
        import ctypes as C
        import torch
        import torch.distributed as dist
        from . import _native as N
        G, ctx = self.plan.G, self.ctx
        h = (C.c_char * 64)()
        N.check(N.lib().mb200_bank_ipc_handle(bank.handle, C.cast(h, C.c_void_p)), ctx.handle)
        dev = f"cuda:{ctx.device}"
        mine = torch.frombuffer(bytearray(bytes(h)), dtype=torch.uint8).to(dev)
        allh = torch.empty(G * 64, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, mine, group=self.group)
        allh = allh.cpu().numpy().tobytes()
        own, _ = bank.counters_ptr()
        self.counter_blocks = (C.c_void_p * G)()
        for g in range(G):
            if g == self.plan.rank:
                self.counter_blocks[g] = own
                continue
            q = C.c_void_p()
            hb = (C.c_char * 64).from_buffer_copy(allh[g * 64:(g + 1) * 64])
            N.check(N.lib().mb200_peer_open(ctx.handle, C.cast(hb, C.c_void_p), C.byref(q)), ctx.handle)
            self._opened.append(q)
            self.counter_blocks[g] = q.value
        # int32 copies in peer-accessible memory: what the undecided candidates are actually read from
        E, d, w = bank.E, bank.d, bank.w
        p32, h32 = C.c_void_p(), (C.c_char * 64)()
        N.check(N.lib().mb200_peer_alloc(ctx.handle, E * d * w * 4, C.byref(p32), C.cast(h32, C.c_void_p)), ctx.handle)
        self._own.append(p32)
        self._narrow_of = (bank, p32)
        mine = torch.frombuffer(bytearray(bytes(h32)), dtype=torch.uint8).to(dev)
        dist.all_gather_into_tensor(allh_t := torch.empty(G * 64, dtype=torch.uint8, device=dev), mine, group=self.group)
        allh = allh_t.cpu().numpy().tobytes()
        self.counter_blocks32 = (C.c_void_p * G)()
        for g in range(G):
            if g == self.plan.rank:
                self.counter_blocks32[g] = p32.value
                continue
            q = C.c_void_p()
            hb = (C.c_char * 64).from_buffer_copy(allh[g * 64:(g + 1) * 64])
            N.check(N.lib().mb200_peer_open(ctx.handle, C.cast(hb, C.c_void_p), C.byref(q)), ctx.handle)
            self._opened.append(q)
            self.counter_blocks32[g] = q.value
        # Local copies of the peers' int32 banks, when they fit beside everything else (the fused form only: the
        # streamed form exists for shapes whose gathered operands do not fit): the undecided candidates are then
        # read from local HBM -- the same peer rows are wanted by thousands of local rows, and every read through
        # a peer mapping is an NVLink round trip.  Filled per step by pull_counters().
        self.local32, self.local_blocks32 = None, None
        nbytes = E * d * w * 4
        free, _ = torch.cuda.mem_get_info(ctx.device)
        want = (G - 1) * nbytes
        # (worth it only when K3 is long enough to hide the copies: K3 time / copy time ~ 2.3e-4 * rows per shard)
        fits = torch.tensor([1 if (self.staging_rows is not None and G > 1 and E >= LOCAL_COUNTERS_MIN_ROWS
                                   and want <= LOCAL_COUNTERS_MAX_BYTES
                                   and free - want >= LOCAL_COUNTERS_KEEP_FREE) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(fits, op=dist.ReduceOp.MIN, group=self.group)      # the same path on every rank
        if int(fits.item()) == 1:
            self.local32 = [None if g == self.plan.rank else torch.empty(E * d * w, dtype=torch.int32, device=dev)
                            for g in range(G)]
            self.local_blocks32 = (C.c_void_p * G)()
            for g in range(G):
                self.local_blocks32[g] = p32.value if g == self.plan.rank else self.local32[g].data_ptr()
            self._counter_bytes = nbytes
        return self.counter_blocks

    def pull_counters(self):
        """queue the copies of the peers' int32 banks behind the row pulls (no-op when they are read in place)"""
        import ctypes as C
        from . import _native as N
        if self.local_blocks32 is None:
            return
        N.check(N.lib().mb200_gather_pull_counters(self.ctx.handle, C.cast(self.local_blocks32, C.c_void_p),
                                                   C.cast(self.counter_blocks32, C.c_void_p), self.plan.G, self.plan.rank,
                                                   self._counter_bytes), self.ctx.handle)

    def fence(self):
        """the compute stream waits for the copies queued so far"""
        from . import _native as N
        N.check(N.lib().mb200_gather_fence(self.ctx.handle), self.ctx.handle)

    @property
    def blocks32(self):
        """where k_certify reads the int32 counters of every block: local copies if held, else the peer mappings"""
        return self.local_blocks32 if getattr(self, "local_blocks32", None) is not None else getattr(self, "counter_blocks32", None)

    def refresh_narrow(self):
        """bring this rank's int32 copy up to date with its bank (before the step's first barrier)"""
        from . import _native as N
        if getattr(self, "_narrow_of", None) is not None:
            bank, p32 = self._narrow_of
            N.check(N.lib().mb200_bank_narrow32(bank.handle, p32), self.ctx.handle)

    def barrier(self):
        """stream-ordered cross-rank barrier (a one-word all-reduce on the current stream)"""
        import torch.distributed as dist
        dist.all_reduce(self.token, group=self.group)

    def pull(self):
        """queue the DMA pulls of every shard + their arrival flags; returns (flags_ptr, epoch)"""
        import ctypes as C
        from . import _native as N
        flags, epoch = C.c_void_p(), C.c_uint32()
        N.check(N.lib().mb200_gather_pull(
            self.ctx.handle, C.c_void_p(self.staging_rows.data_ptr()), C.c_void_p(self.staging_valid.data_ptr()),
            C.cast(self.peer_rows, C.c_void_p), C.cast(self.peer_valid, C.c_void_p), self.plan.G, self.plan.rank,
            self.rows_bytes, self.valid_bytes, C.byref(flags), C.byref(epoch)), self.ctx.handle)
        return flags.value, epoch.value

    def close(self):
        from . import _native as N
        import torch
        if getattr(self, "_own", None) is None:
            return
        torch.cuda.synchronize(self.ctx.device)
        self.barrier()                       # nobody is still reading my buffers
        torch.cuda.synchronize(self.ctx.device)
        self.rows = self.valid = None
        self.local32 = self.local_blocks32 = None
        for q in self._opened:
            N.lib().mb200_peer_close(self.ctx.handle, q)
        for p in self._own:
            N.lib().mb200_peer_free(self.ctx.handle, p)
        self._own = None


def fused_gather_cosine(backend, plan, peers: PeerRows, k, threshold=None, dtype: str = "f16",
                        precision: str = "tensor", a_counters=None, b_counters=None, out=None, counter_blocks=None,
                        mixed_sign: bool = False):
    """C1 fused into K3: `peers.rows` / `peers.valid` hold this rank's normalised rows (K2 output).  One
    stream-ordered barrier makes every rank's rows final, the copy engines then pull the shards over
    NVLink while K3 -- launched immediately, once, over all blocks -- waits block by block on the arrival
    flags; a second barrier keeps every rank's rows alive until all peers have read them.  The context's
    stream must be the current torch stream (the NCCL barriers are ordered with K2 / K3 through it)."""
    G = plan.G
    if counter_blocks is not None:
        peers.refresh_narrow()
    peers.barrier()
    ready = peers.pull()
    if counter_blocks is not None and precision != "tensor":
        peers.pull_counters()

    def attempt(flags):
        job = backend.begin(plan, peers.rows, peers.valid, k, threshold, dtype, precision,
                            **({"mixed_sign": True} if mixed_sign else {}))
        try:
            job.push(peers.staging_rows, peers.staging_valid, id_mul=G, id_add=1, ready=flags, first_block=plan.rank)
            if precision != "tensor":
                if counter_blocks is not None:
                    peers.fence()
                return job.finish(a_counters=a_counters, b_counters=b_counters, b_id=(G, 1), out=out,
                                  resident_b=(peers.staging_rows, peers.staging_valid),
                                  counter_blocks=counter_blocks, b_count=plan.rows_per_shard,
                                  counter_blocks32=peers.blocks32 if counter_blocks is not None else None)
            return job.finish(out=out)
        except BaseException:
            job.abort()
            raise

    try:
        try:
            res = attempt(ready)
        except sk.N.NativeError as ex:
            if getattr(ex, "code", None) != sk.N.ERR_PULL_TIMEOUT:
                raise
            # A pull had not landed when K3 gave up (~4 s).  The peers keep their rows until the closing barrier, so
            # this rank can recover on its own: wait for the copy stream, then sweep the fully staged operand
            # without flags.
            import warnings
            warnings.warn(f"fused pull-gather: {ex}; repeating the sweep over the staged operand")
            FUSED_RETRIES[0] += 1
            sk.N.check(sk.N.lib().mb200_gather_wait(backend.ctx.handle), backend.ctx.handle)
            res = attempt(None)
    except BaseException:
        # the peers are waiting at the closing barrier: meet them before the error leaves this rank, or the step
        # deadlocks (the caller is expected to fail on every rank -- see `all_ranks_ok`)
        peers.barrier()
        raise
    peers.barrier()
    return res


def all_ranks_ok(ok: bool, device, group=None) -> bool:
    """collective AND of a per-rank status: a step that failed on one rank (e.g. too many rows for the exact path)
    must be abandoned by all of them together, or the next collective hangs"""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return bool(ok)
    t = torch.tensor([0 if ok else 1], dtype=torch.int32, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return int(t.item()) == 0


def _fused_path(backend, plan, k, threshold, dtype, precision, group, gather_result, num_items):
    """sharded_item_similarity over fused_gather_cosine: K2 writes straight into the peer-accessible rows"""
    import ctypes as C
    import torch
    from . import _native as N
    ctx, world = backend.ctx, plan.G
    dev = torch.device(f"cuda:{ctx.device}")
    cur = torch.cuda.current_stream(dev)
    prev = ctx.stream_ptr
    comp = torch.cuda.Stream(dev) if prev is None else torch.cuda.ExternalStream(prev, dev)
    comp.wait_stream(cur)
    if prev is None:
        ctx.set_stream(comp.cuda_stream)
    peers = None
    try:
        with torch.cuda.stream(comp):
            try:
                peers = PeerRows(ctx, plan, backend.bank.d, backend.bank.w, dtype, group)
            except sk.N.NativeError:
                return None
            N.check(N.lib().mb200_bank_normalize(backend.bank.handle, sk._DTYPES[dtype], C.c_void_p(peers.rows.data_ptr()),
                                                 C.c_void_p(peers.valid.data_ptr())), ctx.handle)
            kw = dict(mixed_sign=backend.mixed_sign(precision, group))
            if precision == "certified":
                kw.update(a_counters=backend.counters(), counter_blocks=peers.map_counters(backend.bank))
            elif precision != "tensor":
                a_cnt = backend.counters()
                kw.update(a_counters=a_cnt, b_counters=_all_gather(a_cnt, world, group))
            try:
                res, err = fused_gather_cosine(backend, plan, peers, k, threshold, dtype, precision, **kw), None
            except sk.N.NativeError as ex:
                res, err = None, ex
            if not all_ranks_ok(err is None, dev, group):
                # a shard did not arrive through the copy engines in time on some rank (K3 reports it after ~4 s):
                # every rank repeats the stage through the NCCL all-gather
                import warnings
                warnings.warn(f"fused pull-gather abandoned ({err!r}); falling back to the all-gather form")
                peers.close()
                peers = None
                cur.wait_stream(comp)
                return None
            idx, sim, cnt = res
            if gather_result:
                parts = [_all_gather(t, world, group).cpu().numpy() for t in (idx, sim, cnt)]      # C3
                out = tuple(plan.assemble(list(p)) for p in parts)
            else:
                out = (idx, sim, cnt)
            peers.close()
            peers = None
        cur.wait_stream(comp)
    finally:
        if prev is None:
            ctx.sync()
            ctx.set_stream(None)
    backend.close()
    return out


def sharded_item_similarity(row, user, pref, num_items: int, k: int = DEFAULT_MAX_SIMILAR_ITEMS_PER_ITEM,
                            threshold: float | None = None, width: int = 4096, depth: int = 4, seed: int = 42,
                            frac_bits: int = 1, dtype: str = "f16", precision: str = "tensor",
                            group=None, backend=None, gather_result: bool = True, chunk_rows: int = 0,
                            fused: bool | None = None):
    """One call per rank (torch.distributed initialised; NCCL on GPUs).  `row, user, pref` are the
    events this rank holds (any subset of the stream: they are first routed to their owners).
    chunk_rows > 0 selects the pipelined form (`pipelined_cosine`): the all-gather runs in chunks of that
    many rows per shard, overlapped with K3.  fused (default on GPUs with world > 1 and chunk_rows == 0)
    selects `fused_gather_cosine`: the shards are pulled over NVLink by the copy engines while one K3
    launch consumes them in order of arrival.
    Returns (idx, sim, cnt) for all N items on every rank when gather_result, else this rank's
    shard in local row order."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    plan = ShardPlan(num_items, world, rank)
    backend = backend or GpuShardBackend()
    if world > 1:
        # route events to the owner of their item: one all-to-all of the 20-byte events, on the GPUs
        # (NCCL) when the backend computes there
        dev = getattr(backend, "device", None)
        t = [torch.as_tensor(np.asarray(x, dt)) for x, dt in ((row, np.int64), (user, np.int64), (pref, np.float32))]
        if dev is not None:
            t = [x.to(dev) for x in t]
        router = None
        if dev is not None and isinstance(backend, GpuShardBackend):
            # on the GPUs: partition + peer scatter in one kernel (csrc/route.cu), on the context's stream
            ctx = backend.ctx
            cur = torch.cuda.current_stream(torch.device(dev))
            prev = ctx.stream_ptr
            if prev is None:
                ctx.set_stream(cur.cuda_stream)
            try:
                lrow, luser, lpref, router = route_events_device(ctx, plan, *t, group=group)
                backend.build(plan, lrow, luser, lpref, width, depth, seed, frac_bits)
                torch.cuda.synchronize(torch.device(dev))
            finally:
                if prev is None:
                    ctx.set_stream(None)
            router.close()
            lrow = None
        else:
            lrow, luser, lpref = route_events(plan, *t, group=group)
        if dev is None:
            lrow, luser, lpref = lrow.numpy(), luser.numpy(), lpref.numpy()
    else:
        row, user, pref = np.asarray(row, np.int64), np.asarray(user, np.int64), np.asarray(pref, np.float32)
        lrow, luser, lpref = plan.my_events(row, user, pref)
    if lrow is not None:
        backend.build(plan, lrow, luser, lpref, width, depth, seed, frac_bits)
    if fused is None:
        fused = world > 1 and chunk_rows == 0 and isinstance(backend, GpuShardBackend)
    if fused and world > 1:
        out = _fused_path(backend, plan, k, threshold, dtype, precision, group, gather_result, num_items)
        if out is not None:
            return out
        # peer mappings are not available on this box (CUDA IPC refused), or a pull timed out: NCCL all-gather, then K3
    a_rows, a_valid = backend.normalized(dtype)
    a_cnt = backend.counters() if precision != "tensor" else None
    mixed = backend.mixed_sign(precision, group) if hasattr(backend, "mixed_sign") else False
    if world > 1 and chunk_rows > 0:
        # C1 in row chunks, overlapped with K3 through the incremental cosine job
        idx, sim, cnt = pipelined_cosine(backend, plan, a_rows, a_valid, k, threshold, dtype, precision, group,
                                         chunk_rows, a_cnt, mixed)
    else:
        if world > 1:
            b_rows = _all_gather(a_rows, world, group)          # C1 (SURVEY.md 8e)
            b_valid = _all_gather(a_valid, world, group)
        else:
            b_rows, b_valid = a_rows.unsqueeze(0), a_valid.unsqueeze(0)
        b_cnt = None
        if precision != "tensor":
            b_cnt = _all_gather(a_cnt, world, group) if world > 1 else a_cnt
        idx, sim, cnt = backend.cosine(plan, a_rows, a_valid, b_rows, b_valid, k, threshold, dtype, precision,
                                       a_cnt, b_cnt, **({"mixed_sign": True} if mixed else {}))
    if not gather_result:
        backend.close()
        return idx, sim, cnt
    if world > 1:
        parts = []
        for t in (idx, sim, cnt):
            parts.append(_all_gather(t, world, group).cpu().numpy())      # C3
        out = tuple(plan.assemble(list(p)) for p in parts)
    else:
        out = tuple(np.asarray(t.cpu().numpy())[:num_items] for t in (idx, sim, cnt))
    backend.close()
    return out
