// group.cu -- bank-mode K1: group the events by entity on the device, then update every entity's
// counter rows from a shared-memory tile.
//
// Reference semantics: one DoubleCountMinSketch per entity, built from that entity's own preference
// array (CosineCM.exportProfile, CosineCM.java:41-58; DoubleCountMinSketch.update,
// DoubleCountMinSketch.java:72-80).  The reference therefore *always* sees the events of an entity
// together; an unordered (entity, key, inc) stream scattered straight to HBM touches one 32-byte sector
// per counter update instead (measured: 176 B of DRAM traffic per event at d = 4).  Here:
//
//   P0  k_group_hist      per-entity histogram (8 B/event read), hot entities absorbed by a per-CTA
//                         shared-memory count cache
//       k_scan_*          exclusive prefix -> one segment per entity
//   P1  k_group_scatter1  tile partition by the high bits of the entity (coalesced runs through shared
//                         memory; 20 B read + 12 B write per event); events that do not fit the narrow
//                         record (key outside [0, 2^32), |quanta| >= 2^15) are applied on the spot with
//                         the direct d x RED.ADD.64 path, so the call never needs a host decision
//   P2  k_group_scatter2  the same partition inside each coarse bucket by the low bits -> records
//                         {u32 key, i32 quanta} grouped by entity (12 B read + 8 B write)
//   U   k_update_grouped  a CTA owns a window of 32 Ki grouped records: entities with >= 128 records in
//                         the window accumulate into an int32 tile of d x W counters in shared memory
//                         (4 hashes + 4 ATOMS per event, no global traffic) which is then added to the
//                         HBM rows with 32-byte read-modify-writes of the touched sectors only; the rest
//                         go warp-cooperatively through RED.ADD.64 (their rows are L2-resident because
//                         the records are grouped)
//
// Integer adds commute, so the result is the bank the direct kernel (and the reference's sequential
// FP64 sum, under the bank's exactness precondition) produces, bit for bit.
#include <string.h>

#include "common.cuh"
#include "k1_dev.cuh"

namespace {

constexpr int G_THREADS = 256;               // four CTAs per SM: four tiles in four different phases
constexpr int G_ITEMS = 8;
constexpr int G_TILE = G_THREADS * G_ITEMS;  // records per partition tile
constexpr int G_NB = 4 * G_THREADS;          // buckets per partition level
constexpr int U_WINDOW = 32768;              // grouped records per update work item
constexpr int U_TILE_MIN = 128;              // records of one entity in a window that pay for a tile
constexpr int Q_NARROW = 1 << 15;            // |quanta| below this: 32 Ki of them cannot overflow an int32
constexpr int HIST_SLOTS_LOG2 = 12;
constexpr long long SUB_BATCH = 1LL << 30;   // events grouped per pass (u32 record offsets; workspace: 20 B/event)

// bulk prefetch of a contiguous range into L2 (one instruction, no registers): the partition kernels issue it
// for the tile AFTER the one they are about to load, so that tile's loads find their lines in L2
__device__ __forceinline__ void l2_prefetch(const void* p, long long bytes) {
  if (bytes >= 16 && (((uintptr_t)p) & 15) == 0)
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"((unsigned)(bytes & ~15LL)) : "memory");
}

// ---- block-wide exclusive scan of nb <= 4 * G_THREADS shared-memory words ---------------------------
// in[] -> out[] (exclusive), returns the total to every thread.  wsum: G_THREADS / 32 + 1 words.
__device__ __forceinline__ unsigned block_excl_scan(const unsigned* in, unsigned* out, int nb, unsigned* wsum) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b0 = tid * 4;
  unsigned v[4], s = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    v[i] = (b0 + i) < nb ? in[b0 + i] : 0u;
    s += v[i];
  }
  unsigned inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    unsigned w = lane < (G_THREADS / 32) ? wsum[lane] : 0u;
    unsigned winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      unsigned t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    if (lane < (G_THREADS / 32)) wsum[lane] = winc - w;  // exclusive prefix of the warp totals
    if (lane == (G_THREADS / 32) - 1) wsum[G_THREADS / 32] = winc;
  }
  __syncthreads();
  unsigned run = wsum[warp] + inc - s;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    if ((b0 + i) < nb) out[b0 + i] = run;
    run += v[i];
  }
  const unsigned total = wsum[G_THREADS / 32];
  __syncthreads();  // out[] is complete (and wsum reusable) when the call returns
  return total;
}

// ---- P0: histogram by entity -------------------------------------------------------------------------
__global__ void __launch_bounds__(512) k_group_hist(const long long* __restrict__ entity, long long n, long long E,
                                                    unsigned* __restrict__ hist, unsigned long long* flags) {
  __shared__ unsigned tag[1 << HIST_SLOTS_LOG2];  // entity + 1; 0 = empty
  __shared__ unsigned cnt[1 << HIST_SLOTS_LOG2];
  for (int s = threadIdx.x; s < (1 << HIST_SLOTS_LOG2); s += blockDim.x) {
    tag[s] = 0;
    cnt[s] = 0;
  }
  __syncthreads();
  unsigned bad = 0;
  auto count = [&](long long e) {
    if (e < 0 || e >= E) {
      bad++;
      return;
    }
    const unsigned te = (unsigned)e + 1u;
    const unsigned slot = ((unsigned)e * 0x9E3779B1u) >> (32 - HIST_SLOTS_LOG2);
    unsigned cur = *reinterpret_cast<volatile unsigned*>(&tag[slot]);
    if (cur == 0) {
      cur = atomicCAS(&tag[slot], 0u, te);
      if (cur == 0) cur = te;
    }
    if (cur == te) atomicAdd(&cnt[slot], 1u);
    else atomicAdd(&hist[e], 1u);
  };
  // 16-byte loads, four entities per thread per trip (two loads in flight); the unaligned head and the
  // tail go one by one
  const long long head = ((uintptr_t)entity & 8) ? 1 : 0;
  const long long n8 = head + ((n - head) & ~7LL);
  const long long stride = (long long)gridDim.x * blockDim.x * 8;
  for (long long t = head + ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8; t < n8; t += stride) {
    const longlong2* src = reinterpret_cast<const longlong2*>(entity + t);
    const longlong2 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2), d = __ldg(src + 3);
    count(a.x);
    count(a.y);
    count(b.x);
    count(b.y);
    count(c.x);
    count(c.y);
    count(d.x);
    count(d.y);
  }
  if (blockIdx.x == 0) {
    if (threadIdx.x < head) count(entity[threadIdx.x]);
    if (n8 + threadIdx.x < n) count(entity[n8 + threadIdx.x]);
  }
  __syncthreads();
  for (int s = threadIdx.x; s < (1 << HIST_SLOTS_LOG2); s += blockDim.x)
    if (tag[s] && cnt[s]) atomicAdd(&hist[tag[s] - 1u], cnt[s]);
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&flags[FLAG_BAD_ENTITY], (unsigned long long)bad);
}

// ---- single-CTA scans (E <= a few million words: tens of microseconds) -------------------------------
// seg[e] = exclusive prefix of hist, seg[E] = total; cur2[e] = seg[e]
__global__ void __launch_bounds__(1024) k_scan_hist(const unsigned* __restrict__ hist, long long E,
                                                    unsigned* __restrict__ seg, unsigned* __restrict__ cur2) {
  __shared__ unsigned wsum[33];
  __shared__ unsigned carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (long long base = 0; base < E; base += 4096) {
    const long long i0 = base + (long long)tid * 4;
    unsigned v[4], s = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      v[i] = (i0 + i) < E ? hist[i0 + i] : 0u;
      s += v[i];
    }
    unsigned inc = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      unsigned w = wsum[lane], winc = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += t;
      }
      wsum[lane] = winc - w;
      if (lane == 31) wsum[32] = winc;
    }
    __syncthreads();
    unsigned run = carry + wsum[warp] + inc - s;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if ((i0 + i) < E) {
        seg[i0 + i] = run;
        cur2[i0 + i] = run;
      }
      run += v[i];
    }
    __syncthreads();
    if (tid == 0) carry += wsum[32];
    __syncthreads();
  }
  if (tid == 0) seg[E] = carry;
}

// cur1[b] = seg[min(b << shift, E)] for b <= nb
__global__ void k_init_coarse(const unsigned* __restrict__ seg, long long E, int shift, int nb,
                              unsigned* __restrict__ cur1, unsigned* __restrict__ base1) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > nb) return;
  long long e = (long long)b << shift;
  if (e > E) e = E;
  const unsigned v = seg[e];
  base1[b] = v;
  if (b < nb) cur1[b] = v;
}

// tile_ptr[b] = exclusive prefix over coarse buckets of ceil(records in bucket / G_TILE); tile_ptr[nb] = total
__global__ void __launch_bounds__(G_THREADS) k_scan_tiles(const unsigned* __restrict__ base1,
                                                          const unsigned* __restrict__ cur1, int nb,
                                                          unsigned* __restrict__ tile_ptr) {
  __shared__ unsigned a[4 * G_THREADS], o[4 * G_THREADS], wsum[G_THREADS / 32 + 1];
  for (int b = threadIdx.x; b < 4 * G_THREADS; b += G_THREADS)
    a[b] = b < nb ? (cur1[b] - base1[b] + G_TILE - 1) / G_TILE : 0u;
  __syncthreads();
  const unsigned total = block_excl_scan(a, o, nb, wsum);
  for (int b = threadIdx.x; b < nb; b += G_THREADS) tile_ptr[b] = o[b];
  if (threadIdx.x == 0) tile_ptr[nb] = total;
}

// one descriptor per P2 tile (coarse bucket, first record, end of the bucket's records) and per U window (first
// entity): the binary searches run here, thousands at a time, instead of as a chain of dependent loads at the head
// of every tile / window
__global__ void k_tile_desc(const unsigned* __restrict__ tile_ptr, const unsigned* __restrict__ base1,
                            const unsigned* __restrict__ end1, int nb1, uint4* __restrict__ desc) {
  const unsigned ntiles = tile_ptr[nb1];
  for (unsigned tile = blockIdx.x * blockDim.x + threadIdx.x; tile < ntiles; tile += gridDim.x * blockDim.x) {
    int lo = 0, hi = nb1;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (tile_ptr[mid] <= tile) lo = mid;
      else hi = mid;
    }
    desc[tile] = make_uint4((unsigned)lo, base1[lo] + (tile - tile_ptr[lo]) * G_TILE, end1[lo], 0u);
  }
}

template <typename IdxT>
__global__ void k_window_desc(const IdxT* __restrict__ seg, long long E, unsigned* __restrict__ win_first) {
  const long long total = (long long)seg[E];
  const long long nwin = (total + U_WINDOW - 1) / U_WINDOW;
  for (long long win = (long long)blockIdx.x * blockDim.x + threadIdx.x; win < nwin; win += (long long)gridDim.x * blockDim.x) {
    const long long w0 = win * U_WINDOW;
    long long lo = 0, hi = E;  // last entity whose segment starts at or before w0 (seg[0] = 0)
    while (hi - lo > 1) {
      const long long mid = (lo + hi) >> 1;
      if ((long long)seg[mid] <= w0) lo = mid;
      else hi = mid;
    }
    win_first[win] = (unsigned)lo;
  }
}

// ---- P1 / P2: tile partition through shared memory ---------------------------------------------------
struct ScatterSmem {
  unsigned hist[G_NB];
  unsigned loff[G_NB];
  unsigned gbase[G_NB];
  uint2 st_kq[G_TILE];
  unsigned st_ent[G_TILE];
  unsigned wsum[G_THREADS / 32 + 1];
};

template <typename T>
struct Scatter1Args {
  const long long* entity;
  const long long* key;
  const T* inc;
  long long n, E;
  int shift, nb;
  unsigned* cursor;   // [nb] running fill position of every bucket
  unsigned* out_ent;  // may be null (single level: the bucket IS the entity)
  uint2* out_kq;
  // direct path for events that do not fit the narrow record
  long long* counters;
  long long cells;
  double qscale;
  unsigned long long* flags;
  unsigned* wide_seen;  // set when an event took the direct path (the bank is then no longer all-zero)
  int prefetch;         // MB200_OPT_GROUP_PREFETCH
  HashFamily hf;
};

// float increments: with a power-of-two quantum the scaling is exact in float, and an integral value below
// 2^15 is the common case -- no FP64 on that path
__device__ __forceinline__ bool quanta_fast(float v, float qscale_f, int& q) {
  const float qf = v * qscale_f;
  q = (int)qf;
  return fabsf(qf) < (float)Q_NARROW && (float)q == qf;
}
__device__ __forceinline__ bool quanta_fast(double v, float qscale_f, int& q) {
  const double qd = v * (double)qscale_f;
  q = (int)qd;
  return fabs(qd) < (double)Q_NARROW && (double)q == qd;
}

// An event the fast conversion rejects (not an integral number of quanta below 2^15): rare, kept out of line so
// that the FP64 conversion and the 128-bit hash arithmetic do not inflate the registers of the partition loop.
// Publishes its own status words.  Returns the quanta when the event still fits the narrow record, else applies
// it with the direct d x RED.ADD.64 path and returns 0.
template <typename T, int D>
__device__ __noinline__ long long slow_event(const Scatter1Args<T>* p, long long e, long long k, T v) {
  unsigned bad = 0;
  unsigned long long maxabs = 0;
  const long long q = inc_to_quanta(v, p->qscale, bad, maxabs);
  if (bad) atomicAdd(&p->flags[FLAG_INEXACT], 1ull);
  if (maxabs) atomicMax(&p->flags[FLAG_MAXABS], maxabs);
  if (q == 0) return 0;
  if ((unsigned long long)k < (1ull << 32) && q > -Q_NARROW && q < Q_NARROW) return q;
  scatter_event<D>(p->counters + (size_t)e * p->cells, p->hf, k, q);
  *p->wide_seen = 1u;
  return 0;
}

// a narrow-quanta event whose key does not fit 32 bits
template <typename T, int D>
__device__ __noinline__ void wide_key_event(const Scatter1Args<T>* p, long long e, long long k, long long q) {
  scatter_event<D>(p->counters + (size_t)e * p->cells, p->hf, k, q);
  *p->wide_seen = 1u;
}

template <typename T, int D>
__global__ void __launch_bounds__(G_THREADS, 4) k_group_scatter1(const __grid_constant__ Scatter1Args<T> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ScatterSmem& sm = *reinterpret_cast<ScatterSmem*>(smem_raw);
  const int tid = threadIdx.x;
  unsigned maxabs = 0;
  const float qscale_f = (float)p.qscale;
  const long long ntiles = (p.n + G_TILE - 1) / G_TILE;
  auto prefetch_tile = [&](long long tile) {
    if (tid == 0 && tile < ntiles && p.prefetch) {
      const long long base = tile * G_TILE;
      const long long m = (p.n - base) < G_TILE ? (p.n - base) : G_TILE;
      l2_prefetch(p.entity + base, m * 8);
      l2_prefetch(p.key + base, m * 8);
      l2_prefetch(p.inc + base, m * (long long)sizeof(T));
    }
  };
  prefetch_tile(blockIdx.x);
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    // the kernel is bound by the latency of its loads, not by their bytes: the next tile is pulled into L2 now
    prefetch_tile(tile + gridDim.x);
    const long long base = tile * G_TILE;
    long long raw_e[G_ITEMS], raw_k[G_ITEMS];
    T raw_v[G_ITEMS];
#pragma unroll
    for (int i = 0; i < G_ITEMS; i++) {
      const long long idx = base + (long long)i * G_THREADS + tid;
      raw_e[i] = -1;
      if (idx < p.n) {
        raw_e[i] = __ldg(p.entity + idx);
        raw_k[i] = __ldg(p.key + idx);
        raw_v[i] = __ldg(p.inc + idx);
      }
    }
    for (int b = tid; b < p.nb; b += G_THREADS) sm.hist[b] = 0;
    __syncthreads();
    unsigned ent[G_ITEMS], rank[G_ITEMS];
    uint2 kq[G_ITEMS];
    bool ok[G_ITEMS];
#pragma unroll
    for (int i = 0; i < G_ITEMS; i++) {
      ok[i] = false;
      const long long e = raw_e[i];
      if (e >= 0 && e < p.E) {  // bad entities were counted by P0
        const long long k = raw_k[i];
        int q;
        if (quanta_fast(raw_v[i], qscale_f, q)) {
          const unsigned aq = (unsigned)(q < 0 ? -q : q);
          maxabs = aq > maxabs ? aq : maxabs;
          if (q != 0 && (unsigned long long)k >= (1ull << 32)) {
            wide_key_event<T, D>(&p, e, k, q);
            q = 0;
          }
        } else {
          q = (int)slow_event<T, D>(&p, e, k, raw_v[i]);
        }
        if (q != 0) {
          ok[i] = true;
          ent[i] = (unsigned)e;
          kq[i] = make_uint2((unsigned)k, (unsigned)q);
          rank[i] = atomicAdd(&sm.hist[(unsigned)e >> p.shift], 1u);
        }
      }
    }
    __syncthreads();
    const unsigned total = block_excl_scan(sm.hist, sm.loff, p.nb, sm.wsum);
    for (int b = tid; b < p.nb; b += G_THREADS) {
      const unsigned c = sm.hist[b];
      if (c) sm.gbase[b] = atomicAdd(&p.cursor[b], c) - sm.loff[b];
    }
#pragma unroll
    for (int i = 0; i < G_ITEMS; i++) {
      if (ok[i]) {
        const unsigned pos = sm.loff[ent[i] >> p.shift] + rank[i];
        sm.st_kq[pos] = kq[i];
        sm.st_ent[pos] = ent[i];
      }
    }
    __syncthreads();
    for (unsigned pos = tid; pos < total; pos += G_THREADS) {
      const unsigned e = sm.st_ent[pos];
      const unsigned o = sm.gbase[e >> p.shift] + pos;
      p.out_kq[o] = sm.st_kq[pos];
      if (p.out_ent) p.out_ent[o] = e;
    }
    __syncthreads();
  }
  publish_flags(p.flags, 0u, 0u, (unsigned long long)maxabs);
}

struct Scatter2Args {
  const unsigned* in_ent;
  const uint2* in_kq;
  const unsigned* base1;     // [nb1 + 1] start of every coarse bucket
  const unsigned* end1;      // [nb1] fill end of every coarse bucket (P1's cursors)
  const unsigned* tile_ptr;  // [nb1 + 1]
  const uint4* desc;         // [tiles] (bucket, first record, end of the bucket's records)
  int nb1, shift, prefetch;
  long long E;
  unsigned* cursor;  // [E] running fill position of every entity
  uint2* out_kq;
};

__global__ void __launch_bounds__(G_THREADS, 4) k_group_scatter2(const Scatter2Args p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ScatterSmem& sm = *reinterpret_cast<ScatterSmem*>(smem_raw);
  const int tid = threadIdx.x;
  const unsigned ntiles = p.tile_ptr[p.nb1];
  const int R = 1 << p.shift;
  auto locate = [&](unsigned tile, unsigned& bkt, unsigned& first, unsigned& last) {
    const uint4 dsc = __ldg(p.desc + tile);
    bkt = dsc.x;
    first = dsc.y;
    last = dsc.z;
  };
  unsigned bkt = 0, first = 0, last = 0;
  auto prefetch_tile = [&](unsigned tile) {
    if (tid == 0 && tile < ntiles && p.prefetch) {
      unsigned b2, f2, l2;
      locate(tile, b2, f2, l2);
      const long long m = (long long)(l2 - f2) < G_TILE ? (long long)(l2 - f2) : G_TILE;
      // record offsets inside a bucket are arbitrary: round the range out to 16-byte boundaries
      const unsigned f16 = f2 & ~3u;
      l2_prefetch(p.in_ent + f16, (m + (f2 - f16)) * 4);
      l2_prefetch(p.in_kq + (f2 & ~1u), (m + (f2 & 1u)) * 8);
    }
  };
  prefetch_tile(blockIdx.x);
  for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    prefetch_tile(tile + gridDim.x);
    locate(tile, bkt, first, last);
    unsigned raw_e[G_ITEMS];
    uint2 raw_kq[G_ITEMS];
#pragma unroll
    for (int i = 0; i < G_ITEMS; i++) {
      const unsigned idx = first + i * G_THREADS + tid;
      raw_e[i] = 0xFFFFFFFFu;
      if (idx < last) {
        raw_e[i] = __ldg(p.in_ent + idx);
        raw_kq[i] = __ldg(p.in_kq + idx);
      }
    }
    for (int b = tid; b < R; b += G_THREADS) sm.hist[b] = 0;
    __syncthreads();
    const unsigned ebase = bkt << p.shift;
    unsigned ent[G_ITEMS], rank[G_ITEMS];
    uint2 kq[G_ITEMS];
    bool ok[G_ITEMS];
#pragma unroll
    for (int i = 0; i < G_ITEMS; i++) {
      ok[i] = raw_e[i] != 0xFFFFFFFFu;
      if (ok[i]) {
        ent[i] = raw_e[i] - ebase;
        kq[i] = raw_kq[i];
        rank[i] = atomicAdd(&sm.hist[ent[i]], 1u);
      }
    }
    __syncthreads();
    const unsigned total = block_excl_scan(sm.hist, sm.loff, R, sm.wsum);
    for (int b = tid; b < R; b += G_THREADS) {
      const unsigned c = sm.hist[b];
      if (c) sm.gbase[b] = atomicAdd(&p.cursor[ebase + b], c) - sm.loff[b];
    }
#pragma unroll
    for (int i = 0; i < G_ITEMS; i++) {
      if (ok[i]) {
        const unsigned pos = sm.loff[ent[i]] + rank[i];
        sm.st_kq[pos] = kq[i];
        sm.st_ent[pos] = ent[i];
      }
    }
    __syncthreads();
    for (unsigned pos = tid; pos < total; pos += G_THREADS)
      p.out_kq[sm.gbase[sm.st_ent[pos]] + pos] = sm.st_kq[pos];
    __syncthreads();
  }
}

// ---- U: grouped update ------------------------------------------------------------------------------
// record sources: Narrow = {u32 key, i32 quanta} pairs produced by P1/P2; Wide = the caller's own grouped
// (CSR) columns, int64 key + float/double increment, converted on the fly
struct NarrowSrc {
  const uint2* kq;
};
template <typename T>
struct WideSrc {
  const long long* key;
  const T* inc;
};

template <typename IdxT>
struct GroupedArgs {
  const IdxT* seg;  // [E + 1] first record of every entity; seg[E] = end of the record space
  const IdxT* end;  // [E] one past the last record of every entity (<= seg[e + 1])
  long long E;
  long long* counters;
  long long cells;
  double qscale;
  unsigned long long* flags;
  unsigned* ticket;
  const unsigned* win_first;  // [windows] first entity of every window (k_window_desc)
  const unsigned* wide_seen;  // may be null
  int tile_ok;  // d * W int32 cells fit the shared-memory tile
  int virgin;   // the bank held only zeros when the call started: exclusive tiles are stored, not added
  HashFamily hf;
};

// pull the records of a window into L2 ahead of the entity walk
__device__ __forceinline__ void prefetch_window(const NarrowSrc& s, long long w0, long long w1) {
  const long long a = w0 & ~1LL;
  l2_prefetch(s.kq + a, (w1 - a) * 8);   // rounded DOWN to 16 bytes: never past the end
}
template <typename T>
__device__ __forceinline__ void prefetch_window(const WideSrc<T>& s, long long w0, long long w1) {
  const long long a = w0 & ~3LL;
  l2_prefetch(s.key + a, (w1 - a) * 8);
  l2_prefetch(s.inc + a, (w1 - a) * (long long)sizeof(T));
}

__device__ __forceinline__ uint32_t col_small(const HashFamily& hf, int i, uint32_t k) {
  const uint64_t s = cmh_mul_add_mod_small(hf.a[i], k, hf.b[i]);
  return hf.wmask ? (uint32_t)(s & (uint64_t)hf.wmask) : (uint32_t)(s % (uint64_t)hf.w);
}

// fetch record r: returns false when it contributes nothing; `narrow` tells whether (k32, q32) describe it
__device__ __forceinline__ bool fetch(const NarrowSrc& s, long long r, double, unsigned&, unsigned long long&,
                                      long long& key, long long& q, bool& narrow) {
  const uint2 v = __ldg(s.kq + r);
  key = (long long)v.x;
  q = (long long)(int)v.y;
  narrow = true;
  return true;
}
template <typename T>
__device__ __forceinline__ bool fetch(const WideSrc<T>& s, long long r, double qscale, unsigned& bad,
                                      unsigned long long& maxabs, long long& key, long long& q, bool& narrow) {
  key = __ldg(s.key + r);
  q = inc_to_quanta(__ldg(s.inc + r), qscale, bad, maxabs);
  narrow = (unsigned long long)key < (1ull << 32) && q > -Q_NARROW && q < Q_NARROW;
  return q != 0;
}

template <int D>
__device__ __forceinline__ void tile_add(int* tile, const HashFamily& hf, uint32_t k, int q) {
  if (D > 0) {
#pragma unroll
    for (int i = 0; i < D; i++) atomicAdd(&tile[i * hf.w + col_small(hf, i, k)], q);
  } else {
#pragma unroll 1
    for (int i = 0; i < hf.d; i++) atomicAdd(&tile[i * hf.w + col_small(hf, i, k)], q);
  }
}

constexpr int U_THREADS = 512;
constexpr int U_DENSE_MAX = U_WINDOW / U_TILE_MIN + 2;

template <typename Src, typename IdxT, int D>
__global__ void __launch_bounds__(U_THREADS, 2) k_update_grouped(const Src src, const GroupedArgs<IdxT> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int* tile = reinterpret_cast<int*>(smem_raw);
  __shared__ long long s_first;            // first entity of the window
  __shared__ unsigned s_next, s_work;      // next entity batch (relative), current window
  __shared__ int s_dense_n, s_wide;
  __shared__ unsigned s_dense[U_DENSE_MAX];  // entities (relative to s_first) that take the tile path
  const int tid = threadIdx.x, lane = tid & 31;
  unsigned bad = 0;
  unsigned long long maxabs = 0;
  const long long total = (long long)p.seg[p.E];
  const long long nwin = (total + U_WINDOW - 1) / U_WINDOW;
  const bool store_only = p.virgin && (p.wide_seen == nullptr || *p.wide_seen == 0u);
  for (;;) {
    __syncthreads();
    if (tid == 0) s_work = atomicAdd(p.ticket, 1u);
    __syncthreads();
    const long long win = s_work;
    if (win >= nwin) break;
    const long long w0 = win * U_WINDOW, w1 = (w0 + U_WINDOW) < total ? (w0 + U_WINDOW) : total;
    if (tid == 32) prefetch_window(src, w0, w1);
    if (tid == 0) {
      s_first = p.win_first[win];
      s_next = 0;
      s_dense_n = 0;
    }
    __syncthreads();
    const long long e_first = s_first;
    // ---- phase A: batches of 32 consecutive entities per warp; sparse ones are flattened over the lanes
    for (;;) {
      unsigned b = 0;
      if (lane == 0) b = atomicAdd(&s_next, 32u);
      b = __shfl_sync(0xffffffffu, b, 0);
      const long long e = e_first + b + lane;
      long long r0 = 0, r1 = 0;
      bool in_win = false;
      if (e < p.E) {
        const long long s0 = (long long)p.seg[e];
        in_win = s0 < w1;
        if (in_win) {
          r0 = s0 > w0 ? s0 : w0;
          r1 = (long long)p.end[e];
          if (r1 > w1) r1 = w1;
          if (r1 < r0) r1 = r0;
        }
      }
      int c = (int)(r1 - r0);
      if (c >= U_TILE_MIN && p.tile_ok) {
        const int at = atomicAdd(&s_dense_n, 1);
        s_dense[at] = b + lane;
        c = 0;
      }
      // inclusive prefix of the sparse record counts over the lanes
      int incl = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int tot = __shfl_sync(0xffffffffu, incl, 31);
      for (int t = lane; t < ((tot + 31) & ~31); t += 32) {
        // owner lane of flattened record t: first lane with incl > t
        int lo = 0;
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
          const int probe = __shfl_sync(0xffffffffu, incl, lo + step - 1);
          if (probe <= t) lo += step;
        }
        const int o_incl = __shfl_sync(0xffffffffu, incl, lo);
        const int o_c = __shfl_sync(0xffffffffu, c, lo);
        const long long o_r0 = __shfl_sync(0xffffffffu, r0, lo);
        if (t < tot) {
          const long long r = o_r0 + (t - (o_incl - o_c));
          long long key, q;
          bool narrow;
          if (fetch(src, r, p.qscale, bad, maxabs, key, q, narrow))
            scatter_event<D>(p.counters + (size_t)(e_first + b + lo) * p.cells, p.hf, key, q);
        }
      }
      // the batch whose last entity starts beyond the window ends the walk
      const unsigned any_out = __ballot_sync(0xffffffffu, !in_win);
      if (any_out) break;
    }
    __syncthreads();
    // ---- phase B: dense entities, one at a time, through the shared-memory tile
    const int nd = s_dense_n;
    for (int di = 0; di < nd; di++) {
      const long long e = e_first + s_dense[di];
      const long long s0 = (long long)p.seg[e], s1 = (long long)p.end[e];
      const long long r0 = s0 > w0 ? s0 : w0, r1 = s1 < w1 ? s1 : w1;
      const bool exclusive = s0 >= w0 && s1 <= w1;
      int4* t4 = reinterpret_cast<int4*>(tile);
      const int c4 = (int)((p.cells + 3) >> 2);
      for (int c = tid; c < c4; c += U_THREADS) t4[c] = make_int4(0, 0, 0, 0);
      if (tid == 0) s_wide = 0;
      __syncthreads();
      long long* ctr = p.counters + (size_t)e * p.cells;
      bool wide = false;
#pragma unroll 4
      for (long long r = r0 + tid; r < r1; r += U_THREADS) {
        long long key, q;
        bool narrow;
        if (fetch(src, r, p.qscale, bad, maxabs, key, q, narrow)) {
          if (narrow) {
            tile_add<D>(tile, p.hf, (uint32_t)key, (int)q);
          } else {
            scatter_event<D>(ctr, p.hf, key, q);
            wide = true;
          }
        }
      }
      if (wide) s_wide = 1;
      __syncthreads();
      // Only this CTA touches the entity during the kernel when all of its records sit in this window --
      // unless some of them just went straight to the counters with RED (a non-atomic read-modify-write
      // could then lose them).  Then: touched 32-byte sectors are stored (virgin bank) or read, added and
      // stored; otherwise every non-zero cell is added with RED.ADD.64.
      if (exclusive && (p.cells & 3) == 0 && !s_wide) {
        longlong2* g2 = reinterpret_cast<longlong2*>(ctr);
        if (store_only) {
          for (int c = tid; c < c4; c += U_THREADS) {
            const int4 v = t4[c];
            if (v.x | v.y | v.z | v.w) {
              g2[2 * c] = make_longlong2(v.x, v.y);
              g2[2 * c + 1] = make_longlong2(v.z, v.w);
            }
          }
        } else {
          for (int c = tid; c < c4; c += 2 * U_THREADS) {
            const int c1 = c + U_THREADS;
            const int4 v0 = t4[c];
            const int4 v1 = c1 < c4 ? t4[c1] : make_int4(0, 0, 0, 0);
            const bool n0 = (v0.x | v0.y | v0.z | v0.w) != 0, n1 = (v1.x | v1.y | v1.z | v1.w) != 0;
            longlong2 a0, b0, a1, b1;
            if (n0) {
              a0 = g2[2 * c];
              b0 = g2[2 * c + 1];
            }
            if (n1) {
              a1 = g2[2 * c1];
              b1 = g2[2 * c1 + 1];
            }
            if (n0) {
              g2[2 * c] = make_longlong2(a0.x + v0.x, a0.y + v0.y);
              g2[2 * c + 1] = make_longlong2(b0.x + v0.z, b0.y + v0.w);
            }
            if (n1) {
              g2[2 * c1] = make_longlong2(a1.x + v1.x, a1.y + v1.y);
              g2[2 * c1 + 1] = make_longlong2(b1.x + v1.z, b1.y + v1.w);
            }
          }
        }
      } else {
        for (int c = tid; c < (int)p.cells; c += U_THREADS) {
          const int v = tile[c];
          if (v) atomicAdd(reinterpret_cast<unsigned long long*>(ctr + c), (unsigned long long)(long long)v);
        }
      }
      __syncthreads();
    }
  }
  publish_flags(p.flags, bad, 0u, maxabs);
}

// CSR validation: row_ptr must be non-decreasing from 0 (otherwise the windows would read out of bounds)
__global__ void k_check_row_ptr(const long long* __restrict__ row_ptr, long long E, long long n,
                                unsigned long long* flags) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e > E) return;
  bool bad = false;
  if (e == 0) bad = row_ptr[0] != 0 || row_ptr[E] != n;
  if (e < E) bad = bad || row_ptr[e] > row_ptr[e + 1] || row_ptr[e] < 0;
  if (bad) atomicAdd(&flags[FLAG_BAD_ENTITY], 1ull);
}

template <typename Src, typename IdxT>
int launch_grouped(mb200_bank* bk, const Src& src, const IdxT* seg, const IdxT* end, unsigned* ticket,
                   const unsigned* wide_seen, long long max_records) {
  mb200_ctx* ctx = bk->ctx;
  GroupedArgs<IdxT> ga;
  ga.seg = seg;
  ga.end = end;
  ga.E = bk->E;
  ga.counters = bk->counters;
  ga.cells = (long long)bk->d * bk->W;
  ga.qscale = ldexp(1.0, bk->frac_bits);
  ga.flags = bk->flags;
  ga.ticket = ticket;
  ga.wide_seen = wide_seen;
  {
    void* wf;
    const long long max_win = max_records / U_WINDOW + 2;
    MB_CHECK(ws_slot(ctx, WS_GROUP_WINDOWS, (size_t)max_win * 4, &wf));
    ga.win_first = (const unsigned*)wf;
    const int g = (int)(max_win / 256 + 1 < 1024 ? max_win / 256 + 1 : 1024);
    k_window_desc<IdxT><<<g, 256, 0, ctx->stream>>>(seg, bk->E, (unsigned*)wf);
    ctx->launches++;
  }
  ga.virgin = bk->virgin ? 1 : 0;
  ga.hf = bk->hf;
  size_t tile_bytes = (((size_t)ga.cells * 4) + 15) & ~(size_t)15;
  // two CTAs per SM while the tile allows it
  const size_t budget = ctx->smem_optin > 4096 ? ctx->smem_optin - 4096 : 0;
  ga.tile_ok = tile_bytes <= budget ? 1 : 0;
  if (!ga.tile_ok) tile_bytes = 16;
  const int per_sm = tile_bytes <= (size_t)110 * 1024 ? 2 : 1;
  const int grid = ctx->num_sms * per_sm;
#define LAUNCH_U(DD)                                                                                          \
  do {                                                                                                        \
    MB_CUDA(ctx, cudaFuncSetAttribute(k_update_grouped<Src, IdxT, DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      (int)tile_bytes));                                                      \
    k_update_grouped<Src, IdxT, DD><<<grid, U_THREADS, tile_bytes, ctx->stream>>>(src, ga);                   \
  } while (0)
  if (bk->d == 4) LAUNCH_U(4);
  else if (bk->d == 1) LAUNCH_U(1);
  else LAUNCH_U(0);
#undef LAUNCH_U
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  bk->virgin = false;
  return MB200_OK;
}

}  // namespace

// ---- host orchestration (called with the context's mutex held) ------------------------------------------
bool mb200_group_applicable(const mb200_bank* bk, int64_t n) {
  // worth it once the events outnumber the fixed cost of the extra passes; the two partition levels cover
  // G_NB * G_NB entities
  return bk->E > 1 && bk->E <= (int64_t)G_NB * G_NB && n >= bk->ctx->group_min_events;
}

template <typename T>
int mb200_group_update(mb200_bank* bk, const long long* entity, const long long* key, const T* inc, int64_t n) {
  mb200_ctx* ctx = bk->ctx;
  const long long E = bk->E;
  const bool two_level = E > G_NB;
  int shift = 0;
  if (two_level) {
    shift = 10;
    while (((E + (1LL << shift) - 1) >> shift) > G_NB) shift++;
  }
  const int nb1 = two_level ? (int)((E + (1LL << shift) - 1) >> shift) : (int)E;
  const size_t smem = sizeof(ScatterSmem);
  for (int64_t off = 0; off < n; off += SUB_BATCH) {
    const int64_t m = (n - off) < SUB_BATCH ? (n - off) : SUB_BATCH;
    unsigned *hist, *seg, *cur2, *cur1, *base1, *tile_ptr, *ticket, *ent1;
    uint2 *kq1, *kq2;
    void* p;
    // the small arrays in one allocation
    const size_t words = (size_t)(E + 1) * 3 + (size_t)(G_NB + 1) * 3 + 8;
    MB_CHECK(ws_slot(ctx, WS_GROUP_SMALL, words * 4, &p));
    hist = (unsigned*)p;
    seg = hist + (E + 1);
    cur2 = seg + (E + 1);
    cur1 = cur2 + (E + 1);
    base1 = cur1 + (G_NB + 1);
    tile_ptr = base1 + (G_NB + 1);
    ticket = tile_ptr + (G_NB + 1);
    MB_CHECK(ws_slot(ctx, WS_GROUP_KQ2, (size_t)m * 8, &p));
    kq2 = (uint2*)p;
    kq1 = nullptr;
    ent1 = nullptr;
    if (two_level) {
      MB_CHECK(ws_slot(ctx, WS_GROUP_KQ1, (size_t)m * 8, &p));
      kq1 = (uint2*)p;
      MB_CHECK(ws_slot(ctx, WS_GROUP_ENT1, (size_t)m * 4, &p));
      ent1 = (unsigned*)p;
    }
    {
    ProfScope prof_group(ctx, MB200_K_GROUP);
    MB_CUDA(ctx, cudaMemsetAsync(hist, 0, (size_t)(E + 1) * 4, ctx->stream));
    MB_CUDA(ctx, cudaMemsetAsync(ticket, 0, 32, ctx->stream));
    {
      long long want = ceil_div64(m, 512 * 8);
      const int grid = (int)(want < (long long)ctx->num_sms * 4 ? want : (long long)ctx->num_sms * 4);
      k_group_hist<<<grid, 512, 0, ctx->stream>>>(entity + off, m, E, hist, bk->flags);
    }
    k_scan_hist<<<1, 1024, 0, ctx->stream>>>(hist, E, seg, cur2);
    Scatter1Args<T> a1;
    a1.entity = entity + off;
    a1.key = key + off;
    a1.inc = inc + off;
    a1.n = m;
    a1.E = E;
    a1.shift = shift;
    a1.nb = nb1;
    a1.counters = bk->counters;
    a1.cells = (long long)bk->d * bk->W;
    a1.qscale = ldexp(1.0, bk->frac_bits);
    a1.flags = bk->flags;
    a1.wide_seen = ticket + 1;
    a1.prefetch = ctx->group_prefetch;
    a1.hf = bk->hf;
    if (two_level) {
      k_init_coarse<<<(nb1 + 1 + 255) / 256, 256, 0, ctx->stream>>>(seg, E, shift, nb1, cur1, base1);
      a1.cursor = cur1;
      a1.out_ent = ent1;
      a1.out_kq = kq1;
    } else {
      a1.cursor = cur2;
      a1.out_ent = nullptr;
      a1.out_kq = kq2;
    }
    {
      long long want = ceil_div64(m, G_TILE);
      const int grid = (int)(want < (long long)ctx->num_sms * 4 ? want : (long long)ctx->num_sms * 4);
#define LAUNCH_S1(DD)                                                                                              \
  do {                                                                                                             \
    MB_CUDA(ctx, cudaFuncSetAttribute(k_group_scatter1<T, DD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    k_group_scatter1<T, DD><<<grid, G_THREADS, smem, ctx->stream>>>(a1);                                           \
  } while (0)
      if (bk->d == 4) LAUNCH_S1(4);
      else LAUNCH_S1(0);
#undef LAUNCH_S1
    }
    if (two_level) {
      k_scan_tiles<<<1, G_THREADS, 0, ctx->stream>>>(base1, cur1, nb1, tile_ptr);
      Scatter2Args a2;
      a2.in_ent = ent1;
      a2.in_kq = kq1;
      a2.base1 = base1;
      a2.end1 = cur1;
      a2.tile_ptr = tile_ptr;
      {
        void* dp;
        const long long max_tiles = m / G_TILE + nb1 + 2;
        MB_CHECK(ws_slot(ctx, WS_GROUP_TILES, (size_t)max_tiles * sizeof(uint4), &dp));
        a2.desc = (const uint4*)dp;
        const int g = (int)(max_tiles / 256 + 1 < 2048 ? max_tiles / 256 + 1 : 2048);
        k_tile_desc<<<g, 256, 0, ctx->stream>>>(tile_ptr, base1, cur1, nb1, (uint4*)dp);
      }
      a2.nb1 = nb1;
      a2.prefetch = ctx->group_prefetch;
      a2.shift = shift;
      a2.E = E;
      a2.cursor = cur2;
      a2.out_kq = kq2;
      MB_CUDA(ctx, cudaFuncSetAttribute(k_group_scatter2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      k_group_scatter2<<<ctx->num_sms * 4, G_THREADS, smem, ctx->stream>>>(a2);
    }
    ctx->launches += two_level ? 7 : 3;
    MB_CUDA(ctx, cudaGetLastError());
    }
    NarrowSrc src{kq2};
    ProfScope prof_update(ctx, MB200_K_UPDATE);
    MB_CHECK((launch_grouped<NarrowSrc, unsigned>(bk, src, seg, cur2, ticket, ticket + 1, m)));
  }
  bk->events_total += (double)n;
  return MB200_OK;
}

template int mb200_group_update<float>(mb200_bank*, const long long*, const long long*, const float*, int64_t);
template int mb200_group_update<double>(mb200_bank*, const long long*, const long long*, const double*, int64_t);

extern "C" int mb200_bank_update_grouped(mb200_bank* bk, const int64_t* row_ptr, const int64_t* key, const float* inc,
                                         int64_t n, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_update_grouped: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 0 || !row_ptr || (n > 0 && (!key || !inc)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update_grouped: bad arguments");
  if (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update_grouped: mem must be MB200_MEM_HOST or MB200_MEM_DEVICE");
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long E = bk->E;
  void* p;
  MB_CHECK(ws_slot(ctx, WS_GROUP_TICKET, 64, &p));
  unsigned* ticket = (unsigned*)p;
  if (mem == MB200_MEM_HOST && (row_ptr[0] != 0 || row_ptr[E] != n))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update_grouped: row_ptr[0] must be 0 and row_ptr[entities] must be n");
  ArgStage st(ctx, mem);
  const long long *d_ptr, *d_key;
  const float* d_inc;
  MB_CHECK(st.in((const long long*)row_ptr, (size_t)E + 1, &d_ptr));
  MB_CHECK(st.in((const long long*)key, (size_t)n, &d_key));
  MB_CHECK(st.in(inc, (size_t)n, &d_inc));
  MB_CUDA(ctx, cudaMemsetAsync(ticket, 0, 32, ctx->stream));
  k_check_row_ptr<<<(unsigned)ceil_div64(E + 1, 256), 256, 0, ctx->stream>>>(d_ptr, E, n, bk->flags);
  ctx->launches++;
  if (n > 0) {
    // a malformed row_ptr must not drive the windows out of bounds: look at the verdict first
    unsigned long long h[FLAG_WORDS];
    MB_CUDA(ctx, cudaMemcpyAsync(h, bk->flags, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (h[FLAG_BAD_ENTITY])
      return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update_grouped: row_ptr is not a non-decreasing sequence from 0 to n");
    WideSrc<float> src{d_key, d_inc};
    ProfScope prof(ctx, MB200_K_UPDATE);
    MB_CHECK((launch_grouped<WideSrc<float>, long long>(bk, src, d_ptr, d_ptr + 1, ticket, nullptr, n)));
  }
  bk->events_total += (double)n;
  return st.finish();
}
