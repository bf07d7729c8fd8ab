// sketch.cu -- sketch bank + K1 count-min update kernels, point query, read-back, pair cosine.
//
// Reference semantics: DoubleCountMinSketch.update / get / cosine
// (DoubleCountMinSketch.java:72-80, 94-103, 114-149) over one sketch per entity built from one
// HashFunctionBuilder (CosineCM.java:41-58).
//
// HBM layout: counters[E][d][W] as signed 64-bit fixed point, quantum 2^-frac_bits.  Integer
// adds commute, so any interleaving of atomics yields the exact sum; it equals the reference's
// sequential FP64 sum bit-for-bit while |counter| < 2^53 quanta (checked).
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "k1_dev.cuh"

template <typename T>
struct Quad {
  long long key[4];
  long long ent[4];
  T inc[4];
};

// vector load of the event columns; STREAM marks the lines evict-first (ld.global.cs), so that a stream of
// events does not push an L2-resident working set out
template <bool STREAM, typename V>
__device__ __forceinline__ V ld_ev(const V* ptr) {
  if constexpr (STREAM) return __ldcs(ptr);
  else return __ldg(ptr);
}

template <typename T, bool HAS_ENTITY, bool VEC, typename K, bool STREAM = false>
__device__ __forceinline__ void load_quad(const UpdateArgs<T, K>& p, long long base, Quad<T>& q) {
  if constexpr (sizeof(K) == 4) {
    // narrow wire format: four u32 keys in one 16-byte load, four u8 quanta in one 4-byte load
    if (VEC) {
      const uint4 k = ld_ev<STREAM>(reinterpret_cast<const uint4*>(p.key + base));
      q.key[0] = k.x; q.key[1] = k.y; q.key[2] = k.z; q.key[3] = k.w;
      if (HAS_ENTITY) {
        const uint4 e = __ldg(reinterpret_cast<const uint4*>(p.entity + base));
        q.ent[0] = e.x; q.ent[1] = e.y; q.ent[2] = e.z; q.ent[3] = e.w;
      }
      if constexpr (sizeof(T) == 1) {
        const uchar4 c = ld_ev<STREAM>(reinterpret_cast<const uchar4*>(p.inc + base));
        q.inc[0] = c.x; q.inc[1] = c.y; q.inc[2] = c.z; q.inc[3] = c.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; j++) q.inc[j] = p.inc[base + j];
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) {
        q.key[j] = p.key[base + j];
        if (HAS_ENTITY) q.ent[j] = p.entity[base + j];
        q.inc[j] = p.inc[base + j];
      }
    }
  } else if (VEC) {
    const longlong2* k2 = reinterpret_cast<const longlong2*>(p.key + base);
    longlong2 k01 = ld_ev<STREAM>(k2), k23 = ld_ev<STREAM>(k2 + 1);
    q.key[0] = k01.x; q.key[1] = k01.y; q.key[2] = k23.x; q.key[3] = k23.y;
    if (HAS_ENTITY) {
      const longlong2* e2 = reinterpret_cast<const longlong2*>(p.entity + base);
      longlong2 e01 = __ldg(e2), e23 = __ldg(e2 + 1);
      q.ent[0] = e01.x; q.ent[1] = e01.y; q.ent[2] = e23.x; q.ent[3] = e23.y;
    }
    if constexpr (sizeof(T) == 4) {
      float4 v = ld_ev<STREAM>(reinterpret_cast<const float4*>(p.inc + base));
      q.inc[0] = (T)v.x; q.inc[1] = (T)v.y; q.inc[2] = (T)v.z; q.inc[3] = (T)v.w;
    } else if constexpr (sizeof(T) == 8) {
      const double2* d2 = reinterpret_cast<const double2*>(p.inc + base);
      double2 a = ld_ev<STREAM>(d2), b = ld_ev<STREAM>(d2 + 1);
      q.inc[0] = (T)a.x; q.inc[1] = (T)a.y; q.inc[2] = (T)b.x; q.inc[3] = (T)b.y;
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) q.inc[j] = p.inc[base + j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      q.key[j] = p.key[base + j];
      if (HAS_ENTITY) q.ent[j] = p.entity[base + j];
      q.inc[j] = p.inc[base + j];
    }
  }
}

// ------------------------------------------------------------------------------------------
// K1 (bank mode): every event goes straight to its entity's counter rows.
// Coalesced 16-byte event loads, 4 events per thread per trip, d RED.ADD.64 per event.
// ------------------------------------------------------------------------------------------
template <typename T, bool HAS_ENTITY, bool VEC, int D, typename K = long long>
__global__ void __launch_bounds__(256) k_update_bank(const UpdateArgs<T, K> p) {
  unsigned int bad = 0, bad_entity = 0;
  unsigned long long maxabs = 0;
  const size_t cells = (size_t)p.hf.d * p.hf.w;
  const long long n4 = p.n & ~3LL;
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  for (long long base = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; base < n4;
       base += stride) {
    Quad<T> ev;
    load_quad<T, HAS_ENTITY, VEC, K>(p, base, ev);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      long long q = inc_to_quanta(ev.inc[j], p.qscale, bad, maxabs);
      long long e = HAS_ENTITY ? ev.ent[j] : 0;
      if (HAS_ENTITY && (e < 0 || e >= p.E)) {
        bad_entity++;
        continue;
      }
      if (q != 0) scatter_event<D>(p.counters + (size_t)e * cells, p.hf, ev.key[j], q);
    }
  }
  // tail (< 4 events)
  if (blockIdx.x == 0 && threadIdx.x < (unsigned)(p.n - n4)) {
    long long t = n4 + threadIdx.x;
    long long q = inc_to_quanta(p.inc[t], p.qscale, bad, maxabs);
    long long e = HAS_ENTITY ? p.entity[t] : 0;
    if (HAS_ENTITY && (e < 0 || e >= p.E)) bad_entity++;
    else if (q != 0) scatter_event<D>(p.counters + (size_t)e * cells, p.hf, p.key[t], q);
  }
  publish_flags(p.flags, bad, bad_entity, maxabs);
}

// ------------------------------------------------------------------------------------------
// K1 (single-sketch mode, E == 1): Zipf-skewed keys hammer a handful of counters, and L2 serialises same-address
// reductions.  ONE CTA of 1024 threads per SM owns a 2-way set-associative shared-memory cache of SETS x 2 keys
// (32-bit tags; slot = {tag, 64-bit sum as lo/hi 32-bit words}), keyed by the KEY, so one lookup covers all d rows.
// The first key to claim a way owns it for the CTA's lifetime (hot keys show up first); owned keys cost one LDS + one
// ATOMS.ADD.32 (+ a rare carry add).  Keys outside [0, 2^32 - 1) and keys whose set is full are misses: they take the
// direct d x RED.ADD.64 path, or the key table on large calls (below).  At the end each slot is flushed with d global
// reductions.
// ------------------------------------------------------------------------------------------
static constexpr int V2_THREADS = 1024;
static constexpr int V2_SETS = 7168;            // 2 ways each; 24 bytes per set
static constexpr unsigned V2_EMPTY = 0xFFFFFFFFu;

// Events the cache does not own are not scattered by the lane that met them -- with ~1/3 of the lanes
// missing, every warp would run the d hashes + d REDs at 1/3 occupancy.  They are queued per warp in
// shared memory and drained 32 at a time, every lane busy.
static constexpr int MISS_Q = 64;  // entries per warp (a trip adds at most 32)

struct CacheV2 {
  uint2* tags;       // [SETS] two 32-bit tags per set
  unsigned int* lo;  // [2 * SETS]
  int* hi;           // [2 * SETS]
};

// returns true when (key, q) was added to the CTA's cache; key < 2^32 - 1
__device__ __forceinline__ bool cache_add(const CacheV2& c, unsigned int t, long long q) {
  const unsigned int set = __umulhi(t * 0x9E3779B1u, (unsigned)V2_SETS);
  unsigned int* tg = reinterpret_cast<unsigned int*>(c.tags + set);
  const unsigned long long both = *reinterpret_cast<volatile unsigned long long*>(c.tags + set);
  const uint2 cur = make_uint2((unsigned)both, (unsigned)(both >> 32));
  int way = -1;
  if (cur.x == t) way = 0;
  else if (cur.y == t) way = 1;
  else {
    if (cur.x == V2_EMPTY) {
      const unsigned old = atomicCAS(tg, V2_EMPTY, t);
      if (old == V2_EMPTY || old == t) way = 0;
    }
    if (way < 0) {
      const unsigned y = *reinterpret_cast<volatile unsigned int*>(tg + 1);
      if (y == t) way = 1;
      else if (y == V2_EMPTY) {
        const unsigned old = atomicCAS(tg + 1, V2_EMPTY, t);
        if (old == V2_EMPTY || old == t) way = 1;
      }
    }
  }
  if (way < 0) return false;
  const unsigned slot = 2u * set + (unsigned)way;
  const unsigned int qlo = (unsigned int)(unsigned long long)q;
  const int qhi = (int)(q >> 32);
  const unsigned int old = atomicAdd(&c.lo[slot], qlo);
  const int h = qhi + ((unsigned int)(old + qlo) < qlo ? 1 : 0);
  if (h != 0) atomicAdd(&c.hi[slot], h);
  return true;
}

__device__ __forceinline__ long long quanta_of(float v, double qscale, float qscale_f, unsigned& bad, unsigned long long& maxabs) {
  // power-of-two quantum: the scaling is exact in float; an integral result below 2^23 needs no FP64
  const float qf = v * qscale_f;
  const int qi = (int)qf;
  if (fabsf(qf) < 8388608.0f && (float)qi == qf) {
    const unsigned long long aq = (unsigned long long)(qi < 0 ? -qi : qi);
    maxabs = aq > maxabs ? aq : maxabs;
    return qi;
  }
  return inc_to_quanta(v, qscale, bad, maxabs);
}
__device__ __forceinline__ long long quanta_of(double v, double qscale, float, unsigned& bad, unsigned long long& maxabs) {
  return inc_to_quanta(v, qscale, bad, maxabs);
}
__device__ __forceinline__ long long quanta_of(unsigned char v, double qscale, float, unsigned& bad, unsigned long long& maxabs) {
  return inc_to_quanta(v, qscale, bad, maxabs);
}

// Key table (large calls).  The keys the cache does not hold are the Zipf tail: unique inside any window a CTA sees,
// so nothing on the chip can merge them, but they do repeat over a call of 10^8+ events.  With KT a queued miss whose
// key is in [0, KT_ROWS) is drained with ONE reduction into ktab[key] (its per-call total, int64 quanta) instead of d
// hashes and d reductions; k_keytab_flush then scatters every nonzero total once and zeroes it.  The decision is taken
// at drain time, with every lane busy, so the per-event loop is the direct path's (measured: 4.53 ms per 10^9 Zipf 1.1
// events against 4.90 with a predicated reduction in the lane that met the miss).  Integer adds commute: the
// counters are the direct path's bit for bit, and an entry is a partial sum of the counters it ends up in, so the
// exactness bound is untouched.  The table's lines are reduced with an L2 evict_last policy and the events are
// loaded evict-first, so that the touched part of the table stays in L2 while the event stream passes.
static constexpr int KT_LOG2 = 24;
static constexpr long long KT_ROWS = 1LL << KT_LOG2;  // 128 MiB of int64 totals
// trace counters (MB200_TRACE): misses into the table, events scattered directly, cache slots flushed, table keys
// flushed
enum { KS_TABLE = 0, KS_DIRECT = 1, KS_CACHE = 2, KS_FLUSHED = 3, KS_WORDS = 4 };

__device__ __forceinline__ unsigned long long l2_evict_last_policy() {
  unsigned long long pol;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

__device__ __forceinline__ void red_add_hinted(long long* addr, long long v, unsigned long long pol) {
  asm volatile("red.global.add.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(addr), "l"(v), "l"(pol) : "memory");
}

// one count per lane, one atomic per warp (whole warps only)
__device__ __forceinline__ void publish_count(unsigned long long* stats, int word, unsigned v) {
  v = __reduce_add_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v) atomicAdd(&stats[word], (unsigned long long)v);
}

// COUNT: keep the trace counters (MB200_TRACE only: the counting costs issue slots)
template <typename T, bool VEC, int D, typename K, bool KT, bool COUNT>
__global__ void __launch_bounds__(V2_THREADS, 1)
    k_update_single_v2(const UpdateArgs<T, K> p, long long* __restrict__ ktab, unsigned long long* __restrict__ stats) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CacheV2 c;
  c.tags = reinterpret_cast<uint2*>(smem_raw);
  c.lo = reinterpret_cast<unsigned int*>(c.tags + V2_SETS);
  c.hi = reinterpret_cast<int*>(c.lo + 2 * V2_SETS);
  long long* mq_key = reinterpret_cast<long long*>(c.hi + 2 * V2_SETS) + (threadIdx.x >> 5) * (2 * MISS_Q);
  long long* mq_val = mq_key + MISS_Q;
  for (int s = threadIdx.x; s < V2_SETS; s += blockDim.x) {
    c.tags[s] = make_uint2(V2_EMPTY, V2_EMPTY);
    c.lo[2 * s] = c.lo[2 * s + 1] = 0;
    c.hi[2 * s] = c.hi[2 * s + 1] = 0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  int qn = 0;
  unsigned int bad = 0;
  unsigned long long maxabs = 0;
  unsigned n_table = 0, n_direct = 0;  // this lane's table reductions / direct scatters (trace counters)
  unsigned long long pol = 0;
  if (KT) pol = l2_evict_last_policy();
  const float qscale_f = (float)p.qscale;
  const long long n4 = p.n & ~3LL;
  const long long stride = (long long)gridDim.x * blockDim.x * 4;
  const long long first = ((long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) * 4;
  for (long long wbase = first; wbase < n4; wbase += stride) {
    const long long base = wbase + (long long)lane * 4;
    const bool live = base < n4;
    Quad<T> ev;
    if (live) load_quad<T, false, VEC, K, KT>(p, base, ev);
#pragma unroll
    for (int j = 0; j < 4; j++) {
      long long q = 0;
      if (live) q = quanta_of(ev.inc[j], p.qscale, qscale_f, bad, maxabs);
      const long long key = ev.key[j];
      const bool act = live && q != 0;
      // cacheable: the key fits the 32-bit tag
      const bool elig = act && (unsigned long long)key < 0xFFFFFFFFull;
      bool miss = act && !elig;
      if (elig) miss = !cache_add(c, (unsigned)key, q);
      const unsigned m = __ballot_sync(0xffffffffu, miss);
      if (miss) {
        const int at = qn + __popc(m & ((1u << lane) - 1u));
        mq_key[at] = key;
        mq_val[at] = q;
      }
      qn += __popc(m);
      __syncwarp();
      if (qn >= 32) {
        qn -= 32;
        {
          const long long k = mq_key[qn + lane], v = mq_val[qn + lane];
          if (KT && (unsigned long long)k < (unsigned long long)KT_ROWS) {
            red_add_hinted(ktab + k, v, pol);
            if (COUNT) n_table++;
          } else {
            scatter_event<D>(p.counters, p.hf, k, v);
            if (COUNT) n_direct++;
          }
        }
        __syncwarp();
      }
    }
  }
  if (lane < qn) {
    const long long k = mq_key[lane], v = mq_val[lane];
    if (KT && (unsigned long long)k < (unsigned long long)KT_ROWS) {
      red_add_hinted(ktab + k, v, pol);
      if (COUNT) n_table++;
    } else {
      scatter_event<D>(p.counters, p.hf, k, v);
      if (COUNT) n_direct++;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < (unsigned)(p.n - n4)) {
    long long t = n4 + threadIdx.x;
    long long q = inc_to_quanta(p.inc[t], p.qscale, bad, maxabs);
    if (q != 0) {
      scatter_event<D>(p.counters, p.hf, (long long)p.key[t], q);
      if (COUNT) n_direct++;
    }
  }
  __syncthreads();
  unsigned n_cache = 0;
  for (int s = threadIdx.x; s < 2 * V2_SETS; s += blockDim.x) {
    const unsigned t = reinterpret_cast<const unsigned*>(c.tags)[s];
    if (t == V2_EMPTY) continue;
    const long long sum = (long long)(((unsigned long long)(unsigned int)c.hi[s] << 32) | c.lo[s]);
    if (sum != 0) {
      scatter_event<D>(p.counters, p.hf, (long long)t, sum);
      if (COUNT) n_cache++;
    }
  }
  publish_flags(p.flags, bad, 0u, maxabs);
  if (COUNT) {
    publish_count(stats, KS_TABLE, n_table);
    publish_count(stats, KS_DIRECT, n_direct);
    publish_count(stats, KS_CACHE, n_cache);
  }
}

// the key table's second half: every nonzero total -> d reductions, and the entry back to 0 (untouched entries are
// only read).  One pass: each thread owns KT_FLUSH_PER entries, loaded up front (two 16-byte loads in flight per
// thread, the whole table in flight across the grid -- a grid-stride loop left the scan latency-bound).
static constexpr int KT_FLUSH_THREADS = 256, KT_FLUSH_PER = 4;

template <int D>
__global__ void __launch_bounds__(KT_FLUSH_THREADS) k_keytab_flush(long long* __restrict__ ktab, long long* __restrict__ counters,
                                                                   const HashFamily hf, unsigned long long* __restrict__ stats) {
  unsigned n_keys = 0;
  const long long i0 = ((long long)blockIdx.x * KT_FLUSH_THREADS + threadIdx.x) * KT_FLUSH_PER;
  const longlong2 a = __ldcs(reinterpret_cast<const longlong2*>(ktab + i0));
  const longlong2 b = __ldcs(reinterpret_cast<const longlong2*>(ktab + i0 + 2));
  const long long v[KT_FLUSH_PER] = {a.x, a.y, b.x, b.y};
#pragma unroll
  for (int j = 0; j < KT_FLUSH_PER; j++) {
    if (v[j] != 0) {
      ktab[i0 + j] = 0;
      scatter_event<D>(counters, hf, i0 + j, v[j]);
      n_keys++;
    }
  }
  if (stats) publish_count(stats, KS_FLUSHED, n_keys);
}

// ------------------------------------------------------------------------------------------
// small kernels: hash, point query, read-back, pair cosine
// ------------------------------------------------------------------------------------------
__global__ void k_hash_keys(uint64_t a_res, uint64_t b_res, uint32_t w, uint32_t wmask,
                            const long long* __restrict__ keys, long long n, int* __restrict__ out) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = (int)cmh_column(a_res, b_res, cmh_residue(keys[t]), w, wmask);
}

// DoubleCountMinSketch.get (DoubleCountMinSketch.java:94-103)
__global__ void k_query(const long long* __restrict__ counters, HashFamily hf, long long E,
                        double inv_q, const long long* __restrict__ entity,
                        const long long* __restrict__ key, long long n, double* __restrict__ out,
                        unsigned long long* flags) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  long long e = entity ? entity[t] : 0;
  if (e < 0 || e >= E) {
    atomicAdd(&flags[FLAG_BAD_ENTITY], 1ull);
    out[t] = nan("");
    return;
  }
  const long long* sk = counters + (size_t)e * hf.d * hf.w;
  const uint64_t kr = cmh_residue(key[t]);
  double est = 1.7976931348623157e308;  // Double.MAX_VALUE
  for (int i = 0; i < hf.d; i++) {
    uint32_t col = cmh_column(hf.a[i], hf.b[i], kr, hf.w, hf.wmask);
    double v = (double)sk[(size_t)i * hf.w + col] * inv_q;
    if (v < est) est = v;
  }
  out[t] = est;
}

__global__ void k_read(const long long* __restrict__ counters, long long n, double inv_q,
                       double* __restrict__ out, unsigned long long* flags) {
  unsigned int range = 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n;
       t += (long long)gridDim.x * blockDim.x) {
    long long c = counters[t];
    if (c >= (1LL << 53) || c <= -(1LL << 53)) range++;
    out[t] = (double)c * inv_q;
  }
  range = __reduce_add_sync(0xffffffffu, range);
  if ((threadIdx.x & 31) == 0 && range) atomicAdd(&flags[FLAG_RANGE], (unsigned long long)range);
}

__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < nw; i++) s += red[i];
  return s;
}

// DoubleCountMinSketch.cosine (DoubleCountMinSketch.java:114-149); one CTA per pair
__global__ void __launch_bounds__(256) k_pair_cosine(const long long* __restrict__ counters_a,
                                                     const long long* __restrict__ counters_b, int d,
                                                     int w, long long Ea, long long Eb, double inv_qa,
                                                     double inv_qb,
                                                     const long long* __restrict__ ea,
                                                     const long long* __restrict__ eb,
                                                     double* __restrict__ out,
                                                     unsigned long long* flags) {
  __shared__ double red[8];
  const long long p = blockIdx.x;
  const long long a = ea[p], b = eb[p];
  if (a < 0 || a >= Ea || b < 0 || b >= Eb) {
    if (threadIdx.x == 0) {
      atomicAdd(&flags[FLAG_BAD_ENTITY], 1ull);
      out[p] = nan("");
    }
    return;
  }
  const long long* ca = counters_a + (size_t)a * d * w;
  const long long* cb = counters_b + (size_t)b * d * w;
  double min_cos = 1.7976931348623157e308;
  for (int i = 0; i < d; i++) {
    double va = 0.0, vb = 0.0, vab = 0.0;
    for (int j = threadIdx.x; j < w; j += blockDim.x) {
      double xa = (double)ca[(size_t)i * w + j] * inv_qa;
      double xb = (double)cb[(size_t)i * w + j] * inv_qb;
      va += xa * xa;
      vb += xb * xb;
      vab += xa * xb;
    }
    va = block_sum(va, red);
    vb = block_sum(vb, red);
    vab = block_sum(vab, red);
    double den = sqrt(va) * sqrt(vb);
    if (den != 0.0) {
      double c = vab / den;
      min_cos = c < min_cos ? c : min_cos;
    }
  }
  if (threadIdx.x == 0) out[p] = (min_cos == 1.7976931348623157e308) ? nan("") : min_cos;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int fill_family(mb200_bank* bk, const int64_t* a, const int64_t* b) {
  bk->hf.d = bk->d;
  bk->hf.w = (uint32_t)bk->W;
  bk->hf.wmask = (bk->W > 1 && (bk->W & (bk->W - 1)) == 0) ? (uint32_t)(bk->W - 1) : 0u;
  for (int i = 0; i < MB200_MAX_DEPTH; i++) {
    bk->hf.a[i] = 0;
    bk->hf.b[i] = 0;
    bk->a_raw[i] = 0;
    bk->b_raw[i] = 0;
  }
  for (int i = 0; i < bk->d; i++) {
    bk->a_raw[i] = a[i];
    bk->b_raw[i] = b[i];
    bk->hf.a[i] = cmh_residue(a[i]);
    bk->hf.b[i] = cmh_residue(b[i]);
  }
  return MB200_OK;
}

static int check_flags(mb200_bank* bk) {
  mb200_ctx* ctx = bk->ctx;
  unsigned long long h[FLAG_WORDS];
  MB_CUDA(ctx, cudaMemcpyAsync(h, bk->flags, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (h[FLAG_BAD_ENTITY])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "%llu event(s)/queries name an entity outside [0,%lld)",
                      h[FLAG_BAD_ENTITY], (long long)bk->E);
  if (h[FLAG_INEXACT])
    return mb200_fail(ctx, MB200_ERR_INEXACT,
                      "%llu increment(s) are not multiples of 2^-%d (or not finite): the bank cannot "
                      "hold them exactly; create the bank with a larger frac_bits",
                      h[FLAG_INEXACT], bk->frac_bits);
  // conservative: every event at the largest magnitude seen, all into one counter
  double bound = bk->events_total * (double)h[FLAG_MAXABS];
  if (h[FLAG_RANGE] || bound >= 9.0e18)
    return mb200_fail(ctx, MB200_ERR_RANGE,
                      "counter magnitude may exceed the exact range (events %.0f x max quanta %llu; "
                      "%llu counters beyond 2^53): use a smaller frac_bits",
                      bk->events_total, h[FLAG_MAXABS], h[FLAG_RANGE]);
  return MB200_OK;
}

// narrow wire format, bank mode: widen to the (int64, int64, float) columns on the device (HBM-cheap next to
// the PCIe bytes saved), then the ordinary path
__global__ void __launch_bounds__(256) k_widen_events(const uint32_t* __restrict__ entity, const uint32_t* __restrict__ key,
                                                      const unsigned char* __restrict__ quanta, long long n,
                                                      float inv_q, long long* __restrict__ out_entity,
                                                      long long* __restrict__ out_key, float* __restrict__ out_inc) {
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    out_entity[t] = entity[t];
    out_key[t] = key[t];
    out_inc[t] = (float)quanta[t] * inv_q;
  }
}

// Single-sketch calls of at least this many events take the key table (k_update_single_v2<KT> + k_keytab_flush).
// The flush costs a scan of the table plus d reductions per distinct key, so the table pays off on large calls only;
// the host-memory path stages 2^23-event chunks, which stay on the direct path.  DESIGN.md §3 has the crossover.
static constexpr int64_t KT_MIN_EVENTS = 1LL << 26;

static int64_t keytab_min_events() {
  if (const char* ev = getenv("MB200_K1_KEYTABLE_MIN_EVENTS"))  // tuning / test override: 0 = always, huge = never
    return strtoll(ev, nullptr, 10);
  return KT_MIN_EVENTS;
}

// the table is zeroed when it is allocated and every call leaves it zeroed (k_keytab_flush)
static int keytab(mb200_ctx* ctx, long long** out) {
  void* p = nullptr;
  bool fresh = false;
  MB_CHECK(ws_slot(ctx, WS_KEYTAB, (size_t)KT_ROWS * sizeof(long long), &p, &fresh));
  if (fresh) MB_CUDA(ctx, cudaMemsetAsync(p, 0, (size_t)KT_ROWS * sizeof(long long), ctx->stream));
  *out = (long long*)p;
  return MB200_OK;
}

template <typename T, typename K = long long>
static int launch_update(mb200_bank* bk, const K* entity, const K* key, const T* inc, int64_t n) {
  mb200_ctx* ctx = bk->ctx;
  if (n <= 0) return MB200_OK;
  if constexpr (sizeof(K) == 4) {
    if (bk->E > 1) {
      if (!entity) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update_u8: entity is NULL but the bank has %lld entities", (long long)bk->E);
      if (bk->frac_bits > 24) return mb200_fail(ctx, MB200_ERR_UNSUPPORTED, "mb200_bank_update_u8: bank mode needs frac_bits <= 24");
      void *we, *wk, *wi;
      MB_CHECK(ws_slot(ctx, WS_WIDEN_ENTITY, (size_t)n * 8, &we));
      MB_CHECK(ws_slot(ctx, WS_WIDEN_KEY, (size_t)n * 8, &wk));
      MB_CHECK(ws_slot(ctx, WS_WIDEN_INC, (size_t)n * 4, &wi));
      long long want = ceil_div64(n, 256);
      const int grid = (int)(want < (long long)ctx->num_sms * 16 ? want : (long long)ctx->num_sms * 16);
      k_widen_events<<<grid, 256, 0, ctx->stream>>>((const uint32_t*)entity, (const uint32_t*)key, (const unsigned char*)inc, n,
                                                   (float)ldexp(1.0, -bk->frac_bits), (long long*)we, (long long*)wk, (float*)wi);
      ctx->launches++;
      MB_CUDA(ctx, cudaGetLastError());
      return launch_update<float, long long>(bk, (const long long*)we, (const long long*)wk, (const float*)wi, n);
    }
  }
  UpdateArgs<T, K> p;
  p.counters = bk->counters;
  p.entity = entity;
  p.key = key;
  p.inc = inc;
  p.n = n;
  p.E = bk->E;
  p.qscale = ldexp(1.0, bk->frac_bits);
  p.flags = bk->flags;
  p.hf = bk->hf;
  const bool vec = sizeof(K) == 4 ? ((((uintptr_t)key | (uintptr_t)entity) & 15) == 0 && ((uintptr_t)inc & 3) == 0)
                                  : ((((uintptr_t)key | (uintptr_t)inc | (uintptr_t)entity) & 15) == 0);
  const bool d4 = bk->d == 4;
  if constexpr (sizeof(K) == 8 && sizeof(T) != 1) {
    if (bk->E > 1 && entity && mb200_group_applicable(bk, n)) return mb200_group_update<T>(bk, entity, key, inc, n);
  }
  ProfScope prof(ctx, MB200_K_UPDATE);
  if (bk->E == 1) {
    // single-sketch mode (the entity column, if any, is not needed): one 1024-thread CTA per SM; the cache's misses of
    // a large call go through the key table
    const size_t smem = (size_t)V2_SETS * 24 + (size_t)(V2_THREADS / 32) * 2 * MISS_Q * sizeof(long long);
    long long want = ceil_div64(n, (int64_t)V2_THREADS * 4);
    int grid = (int)(want < (long long)ctx->num_sms ? want : (long long)ctx->num_sms);
    const bool table = n >= keytab_min_events();
    const bool trace = getenv("MB200_TRACE") != nullptr;
    long long* ktab = nullptr;
    StatusWords sw(ctx, KS_WORDS);
    if (table) MB_CHECK(keytab(ctx, &ktab));
    if (trace) MB_CHECK(sw.zero(WS_K1_STATS));
    unsigned long long* stats = sw.dev;
#define LAUNCH_V2_C(VEC, D, KT, COUNT)                                                                    \
  do {                                                                                                    \
    MB_CUDA(ctx, cudaFuncSetAttribute(k_update_single_v2<T, VEC, D, K, KT, COUNT>,                        \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));           \
    k_update_single_v2<T, VEC, D, K, KT, COUNT><<<grid, V2_THREADS, smem, ctx->stream>>>(p, ktab, stats); \
  } while (0)
#define LAUNCH_V2(VEC, D, KT)                 \
  do {                                        \
    if (trace) LAUNCH_V2_C(VEC, D, KT, true); \
    else LAUNCH_V2_C(VEC, D, KT, false);      \
  } while (0)
    if (d4) {
      if (table && vec) LAUNCH_V2(true, 4, true);
      else if (table) LAUNCH_V2(false, 4, true);
      else if (vec) LAUNCH_V2(true, 4, false);
      else LAUNCH_V2(false, 4, false);
    } else {
      if (table && vec) LAUNCH_V2(true, 0, true);
      else if (table) LAUNCH_V2(false, 0, true);
      else if (vec) LAUNCH_V2(true, 0, false);
      else LAUNCH_V2(false, 0, false);
    }
#undef LAUNCH_V2
#undef LAUNCH_V2_C
    if (table) {
      ctx->launches++;
      MB_CUDA(ctx, cudaGetLastError());
      const unsigned fgrid = (unsigned)(KT_ROWS / (KT_FLUSH_THREADS * KT_FLUSH_PER));
      if (d4) k_keytab_flush<4><<<fgrid, KT_FLUSH_THREADS, 0, ctx->stream>>>(ktab, p.counters, p.hf, stats);
      else k_keytab_flush<0><<<fgrid, KT_FLUSH_THREADS, 0, ctx->stream>>>(ktab, p.counters, p.hf, stats);
    }
    if (trace) {
      MB_CUDA(ctx, cudaGetLastError());
      unsigned long long h[KS_WORDS];
      MB_CHECK(sw.read(h));
      // L2 reductions of the call: one per table miss, d per direct event, cached key and flushed table key
      const double reds = (double)h[KS_TABLE] + (double)bk->d * (double)(h[KS_DIRECT] + h[KS_CACHE] + h[KS_FLUSHED]);
      fprintf(stderr,
              "[mb200 trace] k1: path=%s n=%lld misses_table=%llu misses_direct=%llu cache_keys=%llu flushed_keys=%llu "
              "reds_per_event=%.4f\n",
              table ? "table" : "direct", (long long)n, h[KS_TABLE], h[KS_DIRECT], h[KS_CACHE], h[KS_FLUSHED],
              reds / (double)n);
    }
  } else {
    const int threads = 256;
    long long want = ceil_div64(n, (int64_t)threads * 4);
    long long cap = (long long)ctx->num_sms * 16;
    int grid = (int)(want < cap ? want : cap);
    if (!entity) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update: entity is NULL but the bank has %lld entities", (long long)bk->E);
    if constexpr (sizeof(K) == 8) {
#define LAUNCH_BANK(VEC, D) k_update_bank<T, true, VEC, D><<<grid, threads, 0, ctx->stream>>>(p)
      if (vec && d4) LAUNCH_BANK(true, 4);
      else if (vec) LAUNCH_BANK(true, 0);
      else if (d4) LAUNCH_BANK(false, 4);
      else LAUNCH_BANK(false, 0);
#undef LAUNCH_BANK
    }
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  bk->events_total += (double)n;
  bk->virgin = false;
  return MB200_OK;
}

static int ensure_stage(mb200_ctx* ctx, size_t bytes) {
  if (ctx->stage_bytes >= bytes) return MB200_OK;
  for (int i = 0; i < 2; i++) {
    if (ctx->stage[i]) MB_CUDA(ctx, cudaFree(ctx->stage[i]));
    ctx->stage[i] = nullptr;
  }
  ctx->stage_bytes = 0;
  for (int i = 0; i < 2; i++) MB_CUDA(ctx, cudaMalloc(&ctx->stage[i], bytes));
  ctx->stage_bytes = bytes;
  return MB200_OK;
}

// host-resident events: chunked, double-buffered H2D on the copy stream overlapped with K1
template <typename T, typename K = long long>
static int update_from_host(mb200_bank* bk, const K* entity, const K* key, const T* inc, int64_t n) {
  mb200_ctx* ctx = bk->ctx;
  const int64_t chunk = 1 << 23;  // 8 Mi events
  const bool has_e = entity != nullptr && bk->E > 1;
  const size_t per_event = sizeof(K) + sizeof(T) + (has_e ? sizeof(K) : 0);
  const int64_t c_events = n < chunk ? n : chunk;
  // each array starts 256-byte aligned inside the staging buffer
  const size_t off_key = 0;
  const size_t off_ent = ((size_t)c_events * sizeof(K) + 255) & ~(size_t)255;
  const size_t off_inc = off_ent + (has_e ? (((size_t)c_events * sizeof(K) + 255) & ~(size_t)255) : 0);
  const size_t need = off_inc + (((size_t)c_events * sizeof(T) + 255) & ~(size_t)255);
  (void)per_event;
  MB_CHECK(ensure_stage(ctx, need));
  int buf = 0;
  for (int64_t off = 0; off < n; off += chunk, buf ^= 1) {
    const int64_t m = (n - off) < chunk ? (n - off) : chunk;
    char* base = (char*)ctx->stage[buf];
    MB_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->stage_free[buf], 0));
    MB_CUDA(ctx, cudaMemcpyAsync(base + off_key, key + off, (size_t)m * sizeof(K), cudaMemcpyHostToDevice,
                                 ctx->copy_stream));
    if (has_e)
      MB_CUDA(ctx, cudaMemcpyAsync(base + off_ent, entity + off, (size_t)m * sizeof(K),
                                   cudaMemcpyHostToDevice, ctx->copy_stream));
    MB_CUDA(ctx, cudaMemcpyAsync(base + off_inc, inc + off, (size_t)m * sizeof(T),
                                 cudaMemcpyHostToDevice, ctx->copy_stream));
    MB_CUDA(ctx, cudaEventRecord(ctx->stage_full[buf], ctx->copy_stream));
    MB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->stage_full[buf], 0));
    MB_CHECK((launch_update<T, K>(bk, has_e ? (const K*)(base + off_ent) : nullptr, (const K*)(base + off_key),
                                  (const T*)(base + off_inc), m)));
    MB_CUDA(ctx, cudaEventRecord(ctx->stage_free[buf], ctx->stream));
  }
  // the caller's buffers are only borrowed for the call
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
  return MB200_OK;
}

template <typename T, typename KIn = int64_t, typename K = long long>
static int bank_update_impl(mb200_bank* bk, const KIn* entity, const KIn* key, const T* inc,
                            int64_t n, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_update: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 0) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update: n < 0");
  if (n == 0) return MB200_OK;
  if (!key || !inc) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update: key/inc is NULL");
  if (bk->E > 1 && !entity)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update: entity is NULL but the bank has %lld entities", (long long)bk->E);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->stat_events += n;
  if (mem == MB200_MEM_HOST) ctx->stat_h2d += n * (int64_t)(sizeof(K) + sizeof(T) + (entity && bk->E > 1 ? sizeof(K) : 0));
  if (mem == MB200_MEM_DEVICE)
    return launch_update<T, K>(bk, (const K*)entity, (const K*)key, inc, n);
  if (mem == MB200_MEM_HOST) return update_from_host<T, K>(bk, (const K*)entity, (const K*)key, inc, n);
  return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_update: mem must be MB200_MEM_HOST or MB200_MEM_DEVICE");
}

extern "C" {

int mb200_hash_keys(mb200_ctx* ctx, int64_t a, int64_t b, int32_t w, const int64_t* keys, int64_t n,
                    int32_t* out, int mem) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_hash_keys: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  if (w <= 0 || n < 0 || (n > 0 && (!keys || !out)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_hash_keys: bad arguments (w=%d n=%lld)", w, (long long)n);
  if (n == 0) return MB200_OK;
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ArgStage st(ctx, mem);
  const long long* d_keys;
  int* d_out;
  MB_CHECK(st.in((const long long*)keys, (size_t)n, &d_keys));
  MB_CHECK(st.out((int*)out, (size_t)n, &d_out));
  uint32_t wmask = (w > 1 && (w & (w - 1)) == 0) ? (uint32_t)(w - 1) : 0u;
  k_hash_keys<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(
      cmh_residue(a), cmh_residue(b), (uint32_t)w, wmask, d_keys, n, d_out);
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  return st.finish();
}

int mb200_bank_create_params(mb200_ctx* ctx, int64_t entities, int32_t depth, int32_t width,
                             const int64_t* a, const int64_t* b, int32_t frac_bits,
                             mb200_bank** out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_create: ctx/out is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  *out = nullptr;
  if (entities <= 0 || depth <= 0 || depth > MB200_MAX_DEPTH || width <= 0 || !a || !b)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_bank_create: need entities > 0, 0 < depth <= %d, width > 0 (got %lld, %d, %d)",
                      MB200_MAX_DEPTH, (long long)entities, depth, width);
  if (frac_bits < 0 || frac_bits > 40)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_create: frac_bits must be in [0,40] (got %d)", frac_bits);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  mb200_bank* bk = new mb200_bank();
  bk->ctx = ctx;
  bk->E = entities;
  bk->d = depth;
  bk->W = width;
  bk->frac_bits = frac_bits;
  fill_family(bk, a, b);
  size_t bytes = (size_t)entities * depth * width * sizeof(long long);
  cudaError_t e = cudaMalloc(&bk->counters, bytes);
  if (e != cudaSuccess) {
    delete bk;
    return mb200_fail(ctx, MB200_ERR_OOM, "mb200_bank_create: cannot allocate %zu bytes of counters: %s", bytes, cudaGetErrorString(e));
  }
  e = cudaMalloc(&bk->flags, FLAG_WORDS * sizeof(unsigned long long));
  if (e != cudaSuccess) {
    cudaFree(bk->counters);
    delete bk;
    return mb200_fail(ctx, MB200_ERR_OOM, "mb200_bank_create: flags: %s", cudaGetErrorString(e));
  }
  MB_CUDA(ctx, cudaMemsetAsync(bk->counters, 0, bytes, ctx->stream));
  MB_CUDA(ctx, cudaMemsetAsync(bk->flags, 0, FLAG_WORDS * sizeof(unsigned long long), ctx->stream));
  *out = bk;
  return MB200_OK;
}

int mb200_bank_create(mb200_ctx* ctx, int64_t entities, int32_t depth, int32_t width, int64_t seed,
                      int32_t frac_bits, mb200_bank** out) {
  if (depth <= 0 || depth > MB200_MAX_DEPTH)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_create: depth must be in (0,%d] (got %d)", MB200_MAX_DEPTH, depth);
  int64_t a[MB200_MAX_DEPTH], b[MB200_MAX_DEPTH];
  MB_CHECK(mb200_hash_params(seed, depth, a, b));
  return mb200_bank_create_params(ctx, entities, depth, width, a, b, frac_bits, out);
}

int mb200_bank_destroy(mb200_bank* bk) {
  if (!bk) return MB200_OK;
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaFree(bk->counters);
  cudaFree(bk->flags);
  delete bk;
  return MB200_OK;
}

int mb200_bank_clear(mb200_bank* bk) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_clear: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CUDA(ctx, cudaMemsetAsync(bk->counters, 0, (size_t)bk->E * bk->d * bk->W * sizeof(long long), ctx->stream));
  MB_CUDA(ctx, cudaMemsetAsync(bk->flags, 0, FLAG_WORDS * sizeof(unsigned long long), ctx->stream));
  bk->events_total = 0;
  bk->virgin = true;
  return MB200_OK;
}

// ---- checkpoint ----------------------------------------------------------------------------------------------
struct DumpHeader {
  char magic[8];  // "MB200BK1"
  int64_t E;
  int32_t d, W, frac_bits, reserved;
  double events_total;
  int64_t a[MB200_MAX_DEPTH], b[MB200_MAX_DEPTH];
};

int mb200_bank_dump(mb200_bank* bk, const char* path) {
  if (!bk || !path) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_dump: NULL argument");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CHECK(check_flags(bk));  // a bank with pending errors is not worth keeping
  FILE* f = fopen(path, "wb");
  if (!f) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_dump: cannot write %s", path);
  DumpHeader h;
  memset(&h, 0, sizeof(h));
  memcpy(h.magic, "MB200BK1", 8);
  h.E = bk->E;
  h.d = bk->d;
  h.W = bk->W;
  h.frac_bits = bk->frac_bits;
  h.events_total = bk->events_total;
  memcpy(h.a, bk->a_raw, sizeof(h.a));
  memcpy(h.b, bk->b_raw, sizeof(h.b));
  bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
  const size_t cells = (size_t)bk->E * bk->d * bk->W, chunk = (size_t)8 << 20;  // 64 MiB of counters per copy
  std::vector<long long> host(cells < chunk ? cells : chunk);
  for (size_t off = 0; off < cells && ok; off += chunk) {
    const size_t m = cells - off < chunk ? cells - off : chunk;
    cudaError_t e = cudaMemcpyAsync(host.data(), bk->counters + off, m * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      fclose(f);
      return mb200_fail(ctx, MB200_ERR_CUDA, "mb200_bank_dump: %s", cudaGetErrorString(e));
    }
    ok = fwrite(host.data(), 8, m, f) == m;
  }
  ok = (fclose(f) == 0) && ok;
  if (!ok) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_dump: short write to %s", path);
  ctx->stat_d2h += (int64_t)cells * 8;
  return MB200_OK;
}

int mb200_bank_load(mb200_ctx* ctx, const char* path, mb200_bank** out) {
  if (!ctx || !path || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_load: NULL argument");
  *out = nullptr;
  FILE* f = fopen(path, "rb");
  if (!f) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_load: cannot read %s", path);
  DumpHeader h;
  if (fread(&h, sizeof(h), 1, f) != 1 || memcmp(h.magic, "MB200BK1", 8) != 0 || h.E <= 0 || h.d <= 0 ||
      h.d > MB200_MAX_DEPTH || h.W <= 0) {
    fclose(f);
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_load: %s is not a bank dump", path);
  }
  mb200_bank* bk = nullptr;
  int rc = mb200_bank_create_params(ctx, h.E, h.d, h.W, h.a, h.b, h.frac_bits, &bk);
  if (rc != MB200_OK) {
    fclose(f);
    return rc;
  }
  std::lock_guard<std::mutex> g(ctx->mu);
  const size_t cells = (size_t)h.E * h.d * h.W, chunk = (size_t)8 << 20;
  std::vector<long long> host(cells < chunk ? cells : chunk);
  for (size_t off = 0; off < cells; off += chunk) {
    const size_t m = cells - off < chunk ? cells - off : chunk;
    cudaError_t e = cudaSuccess;
    if (fread(host.data(), 8, m, f) != m) {
      fclose(f);
      cudaStreamSynchronize(ctx->stream);
      cudaFree(bk->counters);
      cudaFree(bk->flags);
      delete bk;
      return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_load: %s is truncated", path);
    }
    e = cudaMemcpyAsync(bk->counters + off, host.data(), m * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      fclose(f);
      return mb200_fail(ctx, MB200_ERR_CUDA, "mb200_bank_load: %s", cudaGetErrorString(e));
    }
  }
  fclose(f);
  bk->events_total = h.events_total;
  bk->virgin = false;
  ctx->stat_h2d += (int64_t)cells * 8;
  *out = bk;
  return MB200_OK;
}

int mb200_bank_counters(mb200_bank* bk, void** device_ptr, int64_t* cells) {
  if (!bk || !device_ptr) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_counters: NULL argument");
  *device_ptr = bk->counters;
  bk->virgin = false;  // the caller may write through the pointer (e.g. an all-reduce in place)
  if (cells) *cells = bk->E * (int64_t)bk->d * bk->W;
  return MB200_OK;
}

int mb200_bank_ipc_handle(mb200_bank* bk, void* ipc_handle) {
  if (!bk || !ipc_handle) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_ipc_handle: NULL argument");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CUDA(ctx, cudaIpcGetMemHandle((cudaIpcMemHandle_t*)ipc_handle, bk->counters));
  return MB200_OK;
}

int mb200_bank_update(mb200_bank* bk, const int64_t* entity, const int64_t* key, const float* inc,
                      int64_t n, int mem) {
  return bank_update_impl<float>(bk, entity, key, inc, n, mem);
}

int mb200_bank_update_f64(mb200_bank* bk, const int64_t* entity, const int64_t* key,
                          const double* inc, int64_t n, int mem) {
  return bank_update_impl<double>(bk, entity, key, inc, n, mem);
}

int mb200_bank_update_u8(mb200_bank* bk, const uint32_t* entity, const uint32_t* key, const uint8_t* quanta,
                         int64_t n, int mem) {
  return bank_update_impl<unsigned char, uint32_t, uint32_t>(bk, entity, key, (const unsigned char*)quanta, n, mem);
}

int mb200_bank_check(mb200_bank* bk) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_check: bank is NULL");
  std::lock_guard<std::mutex> g(bk->ctx->mu);
  MB_CUDA(bk->ctx, cudaSetDevice(bk->ctx->device));
  return check_flags(bk);
}

int mb200_bank_read(mb200_bank* bk, int64_t e0, int64_t e1, double* out, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_read: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (e0 < 0 || e1 > bk->E || e0 > e1 || (e1 > e0 && !out))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_read: bad entity range [%lld,%lld) of %lld", (long long)e0, (long long)e1, (long long)bk->E);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t cells_per = (int64_t)bk->d * bk->W;
  const double inv_q = ldexp(1.0, -bk->frac_bits);
  // at most 256 MiB of doubles per pass when the destination is host memory
  int64_t step = mem == MB200_MEM_HOST ? ((32LL << 20) / cells_per > 0 ? (32LL << 20) / cells_per : 1) : (e1 - e0);
  for (int64_t e = e0; e < e1; e += step) {
    int64_t m = (e1 - e) < step ? (e1 - e) : step;
    int64_t cells = m * cells_per;
    ArgStage st(ctx, mem);
    double* d_out;
    MB_CHECK(st.out(out + (e - e0) * cells_per, (size_t)cells, &d_out));
    long long want = ceil_div64(cells, 256);
    int grid = (int)(want < (long long)ctx->num_sms * 32 ? want : (long long)ctx->num_sms * 32);
    k_read<<<grid, 256, 0, ctx->stream>>>(bk->counters + e * cells_per, cells, inv_q, d_out, bk->flags);
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
    MB_CHECK(st.finish());
  }
  return check_flags(bk);
}

__global__ void k_read_i32(const long long* __restrict__ counters, long long n, int* __restrict__ out,
                           unsigned long long* flags) {
  unsigned int range = 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const long long c = counters[t];
    if (c > 2147483647LL || c < -2147483647LL) range++;
    out[t] = (int)c;
  }
  range = __reduce_add_sync(0xffffffffu, range);
  if ((threadIdx.x & 31) == 0 && range) atomicAdd(&flags[FLAG_RANGE], (unsigned long long)range);
}

int mb200_bank_read_i32(mb200_bank* bk, int64_t e0, int64_t e1, int32_t* out, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_read_i32: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (e0 < 0 || e1 > bk->E || e0 > e1 || (e1 > e0 && !out))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_read_i32: bad entity range [%lld,%lld) of %lld", (long long)e0, (long long)e1, (long long)bk->E);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const int64_t cells_per = (int64_t)bk->d * bk->W;
  int64_t step = mem == MB200_MEM_HOST ? ((64LL << 20) / cells_per > 0 ? (64LL << 20) / cells_per : 1) : (e1 - e0);
  for (int64_t e = e0; e < e1; e += step) {
    int64_t m = (e1 - e) < step ? (e1 - e) : step;
    int64_t cells = m * cells_per;
    ArgStage st(ctx, mem);
    int* d_out;
    MB_CHECK(st.out((int*)out + (e - e0) * cells_per, (size_t)cells, &d_out));
    long long want = ceil_div64(cells, 256);
    int grid = (int)(want < (long long)ctx->num_sms * 32 ? want : (long long)ctx->num_sms * 32);
    k_read_i32<<<grid, 256, 0, ctx->stream>>>(bk->counters + e * cells_per, cells, d_out, bk->flags);
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
    MB_CHECK(st.finish());
  }
  return check_flags(bk);
}

int mb200_bank_query(mb200_bank* bk, const int64_t* entity, const int64_t* key, int64_t n,
                     double* out, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_query: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 0 || (n > 0 && (!key || !out)) || (n > 0 && bk->E > 1 && !entity))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_query: bad arguments");
  if (n == 0) return MB200_OK;
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ArgStage st(ctx, mem);
  const long long *d_entity, *d_key;
  double* d_out;
  MB_CHECK(st.in((const long long*)entity, (size_t)n, &d_entity));
  MB_CHECK(st.in((const long long*)key, (size_t)n, &d_key));
  MB_CHECK(st.out(out, (size_t)n, &d_out));
  k_query<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(
      bk->counters, bk->hf, bk->E, ldexp(1.0, -bk->frac_bits), d_entity, d_key, n, d_out, bk->flags);
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  return check_flags(bk);
}

int mb200_bank_cross_cosine(mb200_bank* bka, const int64_t* ea, mb200_bank* bkb, const int64_t* eb,
                            int64_t n, double* out, int mem) {
  if (!bka || !bkb) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_cross_cosine: bank is NULL");
  mb200_ctx* ctx = bka->ctx;
  if (bkb->ctx != ctx) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_cross_cosine: banks belong to different contexts");
  std::lock_guard<std::mutex> g(ctx->mu);
  // Preconditions.checkArgument of DoubleCountMinSketch.cosine (DoubleCountMinSketch.java:117-118)
  if (bka->W != bkb->W)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "Widths of a (%d) and b (%d) must be the same", bka->W, bkb->W);
  if (bka->d != bkb->d)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "Depths of a (%d) and b (%d) must be the same", bka->d, bkb->d);
  if (n < 0 || (n > 0 && (!ea || !eb || !out)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_cross_cosine: bad arguments");
  if (n == 0) return MB200_OK;
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ArgStage st(ctx, mem);
  const long long *d_a, *d_b;
  double* d_out;
  MB_CHECK(st.in((const long long*)ea, (size_t)n, &d_a));
  MB_CHECK(st.in((const long long*)eb, (size_t)n, &d_b));
  MB_CHECK(st.out(out, (size_t)n, &d_out));
  const int64_t max_grid = 1 << 30;
  for (int64_t off = 0; off < n; off += max_grid) {
    int64_t m = (n - off) < max_grid ? (n - off) : max_grid;
    k_pair_cosine<<<(unsigned)m, 256, 0, ctx->stream>>>(
        bka->counters, bkb->counters, bka->d, bka->W, bka->E, bkb->E, ldexp(1.0, -bka->frac_bits),
        ldexp(1.0, -bkb->frac_bits), d_a + off, d_b + off, d_out + off, bka->flags);
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
  }
  MB_CHECK(st.finish());
  MB_CHECK(check_flags(bka));
  return bka == bkb ? MB200_OK : check_flags(bkb);
}

int mb200_bank_pair_cosine(mb200_bank* bk, const int64_t* ea, const int64_t* eb, int64_t n,
                           double* out, int mem) {
  return mb200_bank_cross_cosine(bk, ea, bk, eb, n, out, mem);
}

}  // extern "C"
