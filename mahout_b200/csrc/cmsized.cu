// cmsized.cu -- CosineCM with a CountMinSketchConfig: every user's sketch at its own (w_u, d_u), one hash family.
//
// Reference semantics (CosineCM.java:84-96, DoubleCountMinSketch.java:114-149, restated in DESIGN.md section 3):
//   userSimilarity(u1, u2) = clamp(cosine(sketch of u1's prefs at u2's shape, u2's own sketch), -1, 1), NaN kept;
//   cosine = min over rows of AB / (sqrt(AA) * sqrt(BB)), rows with a zero denominator skipped, NaN if none.
// NearestNUserNeighborhood keeps the best n admitted similarities under (sim desc, user row asc);
// doEstimatePreference point-queries each neighbour's own sketch (getExportedCMProfile).
//
// Exactness: counters are integer quanta.  AA, BB and AB are summed as FP64 FMAs on integer-valued doubles and scaled
// by 2^-2f at the end; that is exact in any order while AA and BB stay below 2^53 quanta^2 (Cauchy-Schwarz bounds every
// partial sum of AB by the same), and then equals the reference's sequential sum over the scaled counters bit for bit.
// The bound is checked on the device (MB200_ERR_RANGE).  The finishing arithmetic is k_pair_cosine's (sketch.cu).
//
// Kernels:
//   k_sized_build     one CTA per user: prefs -> quanta, (a_i k + b_i) mod p for every (pref, row < dmax) kept for
//                     the queries, the user's sketch in shared memory (global atomics when it does not fit), per-row
//                     sum of squares
//   k_sized_score     persistent CTAs walk work items (shape class, member chunk, query tile) in class order, so a
//                     class's member sketches are read from L2 by every tile: the tile's query sketches are built at
//                     the class shape in shared memory (a per-CTA global slice when one does not fit), then every
//                     warp streams four member sketches and forms AB for eight queries at a time
//   k_sized_select    one CTA per query: radix select + bitonic sort of the admitted similarities of one batch row
//   k_sized_pair      one CTA per pair (pair cosine of the batched Python call)
//   k_sized_estimate  one thread per query, as k_estimate_prefs
//   k_sized_recommend one persistent CTA per SM, one list row at a time, k_recommend's phases: candidate bitmap and
//                     compaction; estimates per chunk of candidates, each neighbour either streamed (its whole
//                     sketch or row by row, cp.async.bulk into an mbarrier ring) or gathered, whichever moves fewer
//                     bytes; top-N
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <map>
#include <utility>
#include <vector>

#include "common.cuh"
#include "k1_dev.cuh"
#include "nb_terms.cuh"
#include "rec_topn.cuh"
#include "tc05.cuh"

struct mb200_sized_bank {
  mb200_ctx* ctx = nullptr;
  int64_t U = 0, nnz = 0, cells = 0, rows = 0, max_cells = 0;
  int32_t frac_bits = 0, dmax = 0;
  uint64_t a_res[MB200_MAX_DEPTH] = {}, b_res[MB200_MAX_DEPTH] = {};
  std::vector<int32_t> w_h, d_h;
  std::vector<int64_t> off_h;
  // device
  int* w = nullptr;
  int* d = nullptr;
  long long* off = nullptr;      // [U+1] first counter of user u (exclusive scan of d_u * w_u)
  long long* rowoff = nullptr;   // [U+1] first row of user u (exclusive scan of d_u)
  long long* counters = nullptr; // [cells]
  double* sumsq = nullptr;       // [rows] sum of squared quanta of each sketch row (integer-valued)
  long long* ptr = nullptr;      // [U+1]
  long long* quanta = nullptr;   // [nnz]
  unsigned long long* hres = nullptr;  // [dmax][nnz] (a_i * item + b_i) mod p
  // shape classes: distinct (w, d), ascending by cells; members sorted by class, then row
  std::vector<int32_t> cw, cd;
  std::vector<int64_t> cptr;
  int* members = nullptr;        // [U]
};

namespace {

constexpr int SZ_THREADS = 256;
constexpr int SZ_TQ = 32;            // largest query tile
constexpr int SZ_MQ = 4, SZ_QO = 8;  // members x queries per warp pass (32 pairs: one per lane)
constexpr int SZ_BUILD_CELLS = 6144; // 48 KiB of shared memory for the build
constexpr int SEL_THREADS = 512;
constexpr int SEL_MAX_N = 1024;
constexpr int EST_THREADS = 128;
constexpr size_t SZ_QSMEM_DEFAULT = 96 * 1024;  // query sketches: two CTAs per SM
constexpr size_t SZ_GSLICE = 256 * 1024;        // per-CTA global slice of the large shapes
constexpr size_t SZ_DENSE = 1ull << 30;         // similarities of one query batch
constexpr double TWO53 = 9007199254740992.0;
constexpr double DMAX = 1.7976931348623157e308;

enum { SW_BAD = 0, SW_INEXACT, SW_RANGE, SW_MAXABS, SW_NEXT, SW_WORDS };

struct SizedHash {
  unsigned long long a[MB200_MAX_DEPTH], b[MB200_MAX_DEPTH];
};

__device__ __forceinline__ unsigned long long mod_p(unsigned long long a, unsigned long long b, unsigned long long kr) {
  return (kr >> 32) == 0 ? cmh_mul_add_mod_small(a, (uint32_t)kr, b) : cmh_mul_add_mod(a, kr, b);
}

// k_pair_cosine's finishing step for one row: AA, BB, AB are integer-valued sums of quanta^2, s2 = 2^-2f
__device__ __forceinline__ void finish_row(double AA, double BB, double AB, double s2, double& min_cos) {
  const double va = AA * s2, vb = BB * s2, vab = AB * s2;
  const double den = sqrt(va) * sqrt(vb);
  if (den != 0.0) {
    const double c = vab / den;
    min_cos = c < min_cos ? c : min_cos;
  }
}

__device__ __forceinline__ double finish_sim(double min_cos) {
  return clamp_sim(min_cos == DMAX ? __longlong_as_double(0x7ff8000000000000ll) : min_cos);
}

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------------------------------
// checks that come before any load they guard
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_sized_validate(const int* __restrict__ w, const int* __restrict__ d, const long long* __restrict__ ptr,
                                 long long U, unsigned long long* sw) {
  unsigned bad = 0;
  for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u <= U; u += (long long)gridDim.x * blockDim.x) {
    if (u == 0) bad += ptr[0] != 0;
    if (u < U) bad += (w[u] < 1) + (d[u] < 1 || d[u] > MB200_MAX_DEPTH) + (ptr[u + 1] < ptr[u]);
  }
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&sw[SW_BAD], (unsigned long long)bad);
}

__global__ void k_sized_check_rows(const long long* __restrict__ rows, long long n, long long U, unsigned long long* sw) {
  unsigned bad = 0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
    bad += rows[t] < 0 || rows[t] >= U;
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&sw[SW_BAD], (unsigned long long)bad);
}

// ---------------------------------------------------------------------------------------------------------------
// build: one CTA per user
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SZ_THREADS) k_sized_build(
    const int* __restrict__ W, const int* __restrict__ D, const long long* __restrict__ off,
    const long long* __restrict__ rowoff, const long long* __restrict__ ptr, const long long* __restrict__ item,
    const float* __restrict__ pref, long long nnz, int dmax, SizedHash hf, double qscale, long long* counters,
    double* __restrict__ sumsq, long long* __restrict__ quanta, unsigned long long* __restrict__ hres,
    unsigned long long* sw) {
  __shared__ long long sk[SZ_BUILD_CELLS];
  const long long u = blockIdx.x;
  const int w = W[u], d = D[u];
  const long long cells = (long long)w * d;
  const bool in_smem = cells <= SZ_BUILD_CELLS;
  long long* dst = counters + off[u];
  long long* acc = in_smem ? sk : dst;
  if (in_smem)
    for (long long c = threadIdx.x; c < cells; c += blockDim.x) sk[c] = 0;
  __syncthreads();
  unsigned bad = 0, range = 0;
  unsigned long long maxabs = 0;
  for (long long t = ptr[u] + threadIdx.x; t < ptr[u + 1]; t += blockDim.x) {
    const long long q = inc_to_quanta(pref[t], qscale, bad, maxabs);
    quanta[t] = q;
    const unsigned long long kr = cmh_residue(item[t]);
    for (int r = 0; r < dmax; r++) {
      const unsigned long long s = mod_p(hf.a[r], hf.b[r], kr);
      hres[(size_t)r * nnz + t] = s;
      if (r < d && q != 0)
        atomicAdd(reinterpret_cast<unsigned long long*>(acc + (size_t)r * w + (s % (unsigned)w)), (unsigned long long)q);
    }
  }
  __syncthreads();
  if (in_smem)
    for (long long c = threadIdx.x; c < cells; c += blockDim.x) dst[c] = sk[c];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = warp; r < d; r += blockDim.x >> 5) {
    double ss = 0.0;
    for (int j = lane; j < w; j += 32) {
      const long long c = acc[(size_t)r * w + j];
      range += c >= (1ll << 53) || c <= -(1ll << 53);
      const double x = (double)c;
      ss = __fma_rn(x, x, ss);
    }
    ss = warp_sum(ss);
    if (lane == 0) {
      range += !(ss < TWO53);
      sumsq[rowoff[u] + r] = ss;
    }
  }
  bad = __reduce_add_sync(0xffffffffu, bad);
  range = __reduce_add_sync(0xffffffffu, range);
  if (lane == 0) {
    if (bad) atomicAdd(&sw[SW_INEXACT], (unsigned long long)bad);
    if (range) atomicAdd(&sw[SW_RANGE], (unsigned long long)range);
  }
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long y = __shfl_xor_sync(0xffffffffu, maxabs, o);
    maxabs = y > maxabs ? y : maxabs;
  }
  if (lane == 0 && maxabs) atomicMax(&sw[SW_MAXABS], maxabs);
}

// ---------------------------------------------------------------------------------------------------------------
// the query sketches of a tile at shape (w, d): int64 quanta accumulated in place, then converted in place to
// integer-valued doubles, with each row's sum of squares in aa[qi * 32 + r]
// ---------------------------------------------------------------------------------------------------------------
struct SizedDev {
  const int* W;
  const int* D;
  const long long* off;
  const long long* rowoff;
  const long long* counters;
  const double* sumsq;
  const long long* ptr;
  const long long* quanta;
  const unsigned long long* hres;
  long long nnz, U;
  double s2;
};

__device__ void build_queries(const SizedDev& b, const long long* qrows, int T, int w, int d, long long* Q,
                              double* aa, unsigned& range) {
  const long long cells = (long long)w * d;
  for (long long i = threadIdx.x; i < (long long)T * cells; i += blockDim.x) Q[i] = 0;
  __syncthreads();
  for (int qi = 0; qi < T; qi++) {
    const long long u = qrows[qi];
    const long long p0 = b.ptr[u], n = b.ptr[u + 1] - p0;
    long long* Qq = Q + (size_t)qi * cells;
    for (long long k = threadIdx.x; k < n * d; k += blockDim.x) {
      const long long t = p0 + k / d;
      const int r = (int)(k % d);
      const long long q = b.quanta[t];
      if (q != 0)
        atomicAdd(reinterpret_cast<unsigned long long*>(Qq + (size_t)r * w + (b.hres[(size_t)r * b.nnz + t] % (unsigned)w)),
                  (unsigned long long)q);
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = warp; k < T * d; k += blockDim.x >> 5) {
    const int qi = k / d, r = k % d;
    long long* row = Q + (size_t)qi * cells + (size_t)r * w;
    double ss = 0.0;
    for (int j = lane; j < w; j += 32) {
      const long long c = row[j];
      range += c >= (1ll << 53) || c <= -(1ll << 53);
      const double x = (double)c;
      reinterpret_cast<double*>(row)[j] = x;
      ss = __fma_rn(x, x, ss);
    }
    ss = warp_sum(ss);
    if (lane == 0) {
      range += !(ss < TWO53);
      aa[qi * 32 + r] = ss;
    }
  }
  __syncthreads();
}

// 32 partial sums per lane -> lane l holds the warp total of value l (31 shuffles)
__device__ __forceinline__ double reduce_scatter32(double (&v)[32]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool upper = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; i++) {
      const double send = upper ? v[i] : v[i + s];
      const double keep = upper ? v[i + s] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0];
}

struct SzItem {
  int cls, mbeg, mcnt, qbeg;  // qbeg: first query of the tile within the batch
};

struct ScoreArgs {
  SizedDev b;
  const int* members;
  const int* cw;
  const int* cd;
  const int* ctile;        // query tile of each class
  const int* cglobal;      // 1: the class's query sketches live in the per-CTA global slice
  const SzItem* items;
  long long n_items;
  const long long* queries;  // this batch's query rows
  long long nq;
  double* sims;              // [nq][U]
  long long* gslice;         // [grid][slice_cells]
  long long slice_cells;
  unsigned long long* sw;
};

__global__ void __launch_bounds__(SZ_THREADS, 2) k_sized_score(const ScoreArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  double* aa = reinterpret_cast<double*>(smem);                          // [SZ_TQ][32]
  long long* qsm = reinterpret_cast<long long*>(smem + SZ_TQ * 32 * 8);  // query sketches
  __shared__ long long next_item;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned range = 0;
  for (;;) {
    if (threadIdx.x == 0) next_item = (long long)atomicAdd(&a.sw[SW_NEXT], 1ull);
    __syncthreads();
    const long long it = next_item;
    __syncthreads();
    if (it >= a.n_items) break;
    const SzItem item = a.items[it];
    const int w = a.cw[item.cls], d = a.cd[item.cls];
    const long long cells = (long long)w * d;
    const int T = min(a.ctile[item.cls], (int)(a.nq - item.qbeg));
    long long* Q = a.cglobal[item.cls] ? a.gslice + (size_t)blockIdx.x * a.slice_cells : qsm;
    build_queries(a.b, a.queries + item.qbeg, T, w, d, Q, aa, range);
    const double* Qd = reinterpret_cast<const double*>(Q);
    const int nquad = (item.mcnt + SZ_MQ - 1) / SZ_MQ, noct = (T + SZ_QO - 1) / SZ_QO;
    const int my_q = lane / SZ_MQ, my_m = lane % SZ_MQ;  // the pair this lane finishes
    for (int k = warp; k < nquad * noct; k += SZ_THREADS / 32) {
      const int mq = k / noct, qo = k % noct;
      long long v[SZ_MQ];
      const long long* B[SZ_MQ];
#pragma unroll
      for (int m = 0; m < SZ_MQ; m++) {
        const int mi = mq * SZ_MQ + m;
        v[m] = mi < item.mcnt ? a.members[item.mbeg + mi] : -1;
        B[m] = v[m] >= 0 ? a.b.counters + a.b.off[v[m]] : nullptr;
      }
      const int nqo = min(SZ_QO, T - qo * SZ_QO);
      const long long my_v = mq * SZ_MQ + my_m < item.mcnt ? a.members[item.mbeg + mq * SZ_MQ + my_m] : -1;
      const int qi = qo * SZ_QO + my_q;
      double min_cos = DMAX;
      for (int r = 0; r < d; r++) {
        double acc[32];
#pragma unroll
        for (int i = 0; i < 32; i++) acc[i] = 0.0;
        for (int j = lane; j < w; j += 32) {
          double bv[SZ_MQ];
#pragma unroll
          for (int m = 0; m < SZ_MQ; m++) bv[m] = B[m] ? (double)__ldg(B[m] + (size_t)r * w + j) : 0.0;
#pragma unroll
          for (int qq = 0; qq < SZ_QO; qq++) {
            const double x = qq < nqo ? Qd[(size_t)(qo * SZ_QO + qq) * cells + (size_t)r * w + j] : 0.0;
#pragma unroll
            for (int m = 0; m < SZ_MQ; m++) acc[qq * SZ_MQ + m] = __fma_rn(x, bv[m], acc[qq * SZ_MQ + m]);
          }
        }
        const double AB = reduce_scatter32(acc);
        if (my_v >= 0 && my_q < nqo) finish_row(aa[qi * 32 + r], a.b.sumsq[a.b.rowoff[my_v] + r], AB, a.b.s2, min_cos);
      }
      if (my_v >= 0 && my_q < nqo) {
        const long long qrow = item.qbeg + qi;
        a.sims[(size_t)qrow * a.b.U + my_v] =
            my_v == a.queries[qrow] ? __longlong_as_double(0x7ff8000000000000ll) : finish_sim(min_cos);
      }
    }
    __syncthreads();
  }
  range = __reduce_add_sync(0xffffffffu, range);
  if (lane == 0 && range) atomicAdd(&a.sw[SW_RANGE], (unsigned long long)range);
}

// ---------------------------------------------------------------------------------------------------------------
// selection: (sim desc, row asc), admitted = not NaN and sim >= min_similarity
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long sim_key(double s, double min_sim) {
  if (s != s || !(s >= min_sim)) return 0ull;
  const long long bits = __double_as_longlong(s == 0.0 ? 0.0 : s);  // -0.0 ranks as 0.0
  return bits < 0 ? ~(unsigned long long)bits : ((unsigned long long)bits | 0x8000000000000000ull);
}

__global__ void __launch_bounds__(SEL_THREADS) k_sized_select(const double* __restrict__ sims, long long U, int n,
                                                              double min_sim, long long* __restrict__ out_idx,
                                                              double* __restrict__ out_sim, int* __restrict__ out_cnt) {
  __shared__ unsigned hist[256];
  __shared__ int scan_sh[32];
  __shared__ unsigned long long sel_key[SEL_MAX_N];
  __shared__ int sel_row[SEL_MAX_N];
  __shared__ unsigned long long bc_prefix;
  __shared__ unsigned bc_want;
  const int tid = threadIdx.x;
  const double* row = sims + (size_t)blockIdx.x * U;
  long long* oi = out_idx + (size_t)blockIdx.x * n;
  double* os = out_sim + (size_t)blockIdx.x * n;
  int valid = 0, nvalid = 0;
  for (long long v = tid; v < U; v += SEL_THREADS) valid += sim_key(row[v], min_sim) != 0ull;
  block_exscan<SEL_THREADS>(valid, scan_sh, &nvalid);
  // keys > kstar are all taken; of the keys == kstar the first `need_eq` in row order
  unsigned long long kstar = 0ull;
  unsigned need_eq = 0;
  if (nvalid > n) {
    unsigned long long prefix = 0ull, mask = 0ull;
    unsigned want = (unsigned)n;
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int t = tid; t < 256; t += SEL_THREADS) hist[t] = 0u;
      __syncthreads();
      for (long long v = tid; v < U; v += SEL_THREADS) {
        const unsigned long long k = sim_key(row[v], min_sim);
        if (k && (k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        unsigned acc = 0;
        for (int b = 255; b >= 0; b--) {
          if (acc + hist[b] >= want) {
            prefix |= (unsigned long long)b << shift;
            want -= acc;
            break;
          }
          acc += hist[b];
        }
        bc_prefix = prefix;
        bc_want = want;
      }
      __syncthreads();
      prefix = bc_prefix;
      want = bc_want;
      mask |= 255ull << shift;
      __syncthreads();
    }
    kstar = prefix;
    need_eq = want;
  }
  const int n_out = nvalid < n ? nvalid : n;
  // ordered compaction, ascending rows
  int taken = 0, eq_taken = 0;
  for (long long base = 0; base < U; base += SEL_THREADS) {
    const long long v = base + tid;
    const unsigned long long k = v < U ? sim_key(row[v], min_sim) : 0ull;
    const int eq = k != 0ull && k == kstar;
    int eq_total = 0, tk_total = 0;
    const int eq_before = block_exscan<SEL_THREADS>(eq, scan_sh, &eq_total);
    const int take = (k != 0ull && k > kstar) || (eq && (unsigned)(eq_taken + eq_before) < need_eq);
    const int at = block_exscan<SEL_THREADS>(take, scan_sh, &tk_total);
    if (take) {
      sel_key[taken + at] = k;
      sel_row[taken + at] = (int)v;
    }
    taken += tk_total;
    eq_taken += eq_total;
  }
  int npad = 1;
  while (npad < n_out) npad <<= 1;
  for (int t = n_out + tid; t < npad; t += SEL_THREADS) {
    sel_key[t] = 0ull;
    sel_row[t] = 0x7fffffff;
  }
  __syncthreads();
  // bitonic sort: (key desc, row asc)
  for (int size = 2; size <= npad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < npad; t += SEL_THREADS) {
        const int partner = t ^ stride;
        if (partner > t) {
          const bool desc = (t & size) == 0;
          const unsigned long long x = sel_key[t], y = sel_key[partner];
          const int xr = sel_row[t], yr = sel_row[partner];
          const bool x_first = x > y || (x == y && xr < yr);
          if (desc ? !x_first : x_first) {
            sel_key[t] = y;
            sel_key[partner] = x;
            sel_row[t] = yr;
            sel_row[partner] = xr;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int t = tid; t < n; t += SEL_THREADS) {
    oi[t] = t < n_out ? (long long)sel_row[t] : -1ll;
    os[t] = t < n_out ? row[sel_row[t]] : 0.0;
  }
  if (tid == 0) out_cnt[blockIdx.x] = n_out;
}

// ---------------------------------------------------------------------------------------------------------------
// pair cosine: one CTA per pair, u1 re-sketched at u2's shape in a per-CTA slice
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SZ_THREADS) k_sized_pair(const SizedDev b, const long long* __restrict__ u1,
                                                           const long long* __restrict__ u2, long long n,
                                                           long long* slices, long long slice_cells,
                                                           double* __restrict__ out, unsigned long long* sw) {
  __shared__ double red[2][SZ_THREADS / 32];
  long long* Q = slices + (size_t)blockIdx.x * slice_cells;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned range = 0;
  for (long long p = blockIdx.x; p < n; p += gridDim.x) {
    const long long x = u1[p], y = u2[p];
    if (x < 0 || x >= b.U || y < 0 || y >= b.U) {
      if (threadIdx.x == 0) {
        atomicAdd(&sw[SW_BAD], 1ull);
        out[p] = __longlong_as_double(0x7ff8000000000000ll);
      }
      continue;
    }
    const int w = b.W[y], d = b.D[y];
    const long long cells = (long long)w * d;
    for (long long i = threadIdx.x; i < cells; i += blockDim.x) Q[i] = 0;
    __syncthreads();
    const long long p0 = b.ptr[x], np = b.ptr[x + 1] - p0;
    for (long long k = threadIdx.x; k < np * d; k += blockDim.x) {
      const long long t = p0 + k / d;
      const int r = (int)(k % d);
      const long long q = b.quanta[t];
      if (q != 0)
        atomicAdd(reinterpret_cast<unsigned long long*>(Q + (size_t)r * w + (b.hres[(size_t)r * b.nnz + t] % (unsigned)w)),
                  (unsigned long long)q);
    }
    __syncthreads();
    const long long* C = b.counters + b.off[y];
    double min_cos = DMAX;
    for (int r = 0; r < d; r++) {
      double AA = 0.0, AB = 0.0;
      for (int j = threadIdx.x; j < w; j += blockDim.x) {
        const long long c = Q[(size_t)r * w + j];
        range += c >= (1ll << 53) || c <= -(1ll << 53);
        const double xa = (double)c, xb = (double)C[(size_t)r * w + j];
        AA = __fma_rn(xa, xa, AA);
        AB = __fma_rn(xa, xb, AB);
      }
      AA = warp_sum(AA);
      AB = warp_sum(AB);
      if (lane == 0) {
        red[0][warp] = AA;
        red[1][warp] = AB;
      }
      __syncthreads();
      AA = 0.0;
      AB = 0.0;
      for (int i = 0; i < SZ_THREADS / 32; i++) {
        AA += red[0][i];
        AB += red[1][i];
      }
      range += threadIdx.x == 0 && !(AA < TWO53);
      finish_row(AA, b.sumsq[b.rowoff[y] + r], AB, b.s2, min_cos);
      __syncthreads();
    }
    if (threadIdx.x == 0) out[p] = finish_sim(min_cos);
  }
  range = __reduce_add_sync(0xffffffffu, range);
  if (lane == 0 && range) atomicAdd(&sw[SW_RANGE], (unsigned long long)range);
}

// ---------------------------------------------------------------------------------------------------------------
// doEstimatePreference with each neighbour's own sketch: one thread per query
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(EST_THREADS) k_sized_estimate(
    const SizedDev b, SizedHash hf, int dmax, double inv_q, const long long* __restrict__ nb_idx,
    const double* __restrict__ nb_sim, const int* __restrict__ nb_cnt, long long nb_rows, int ld,
    const long long* __restrict__ user, const long long* __restrict__ nb_row, const long long* __restrict__ item_id,
    long long q, float* __restrict__ out, unsigned long long* sw) {
  extern __shared__ unsigned long long est_s[];  // [dmax][EST_THREADS]
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= q) return;
  unsigned long long* s = est_s + threadIdx.x;
  const long long u = user[t];
  const long long row = nb_row ? nb_row[t] : u;
  const float nanf_ = __int_as_float(0x7fc00000);
  if (u < 0 || u >= b.U || row < 0 || row >= nb_rows) {
    atomicAdd(&sw[SW_BAD], 1ull);
    out[t] = nanf_;
    return;
  }
  const int cnt = nb_cnt[row];
  if (cnt < 0 || cnt > ld) {
    atomicAdd(&sw[SW_BAD], 1ull);
    out[t] = nanf_;
    return;
  }
  const unsigned long long kr = cmh_residue(item_id[t]);
  for (int r = 0; r < dmax; r++) s[r * EST_THREADS] = mod_p(hf.a[r], hf.b[r], kr);
  double pref = 0.0, tot = 0.0;
  int count = 0;
  for (int j = 0; j < cnt; j++) {
    const long long v = nb_idx[row * ld + j];
    if (v == u) continue;
    if (v < 0 || v >= b.U) {
      atomicAdd(&sw[SW_BAD], 1ull);
      continue;
    }
    const unsigned w = (unsigned)b.W[v];
    const int d = b.D[v];
    const long long* sk = b.counters + b.off[v];
    long long mn = __ldg(sk + s[0] % w);
    for (int r = 1; r < d; r++) {
      const long long x = __ldg(sk + (size_t)r * w + s[(size_t)r * EST_THREADS] % w);
      mn = x < mn ? x : mn;
    }
    nb_term(mn, inv_q, clamp_sim(nb_sim[row * ld + j]), pref, tot, count);
  }
  out[t] = nb_result(pref, tot, count);
}

// ---------------------------------------------------------------------------------------------------------------
// recommend(user, how_many): one persistent CTA per SM, one list row at a time (k_recommend's three phases)
// ---------------------------------------------------------------------------------------------------------------
constexpr int SR_THREADS = 512;
constexpr int SR_KMAX = 8;                  // candidates per thread and chunk
constexpr int SR_BITMAP_SMEM_WORDS = 4096;  // 131072 items: larger catalogues use a per-CTA global bitmap
constexpr int SR_RES_BYTES = 64 * 1024;     // the chunk's hash residues (more when d_max leaves < 512 candidates)
constexpr int SR_STAGES = 4;

enum { SR_GATHER = 0, SR_WHOLE, SR_ROWS, SR_TOO_WIDE };
enum { RP_CHUNKS = 0, RP_CAND_SUM, RP_CAND_MAX, RP_STREAM, RP_ROWS, RP_GATHER, RP_TOO_WIDE, RP_STREAM_BYTES, RP_GATHER_LOADS,
       RP_TERMS, RP_BAD, RP_NEXT, RP_WORDS };

struct SrArgs {
  const int* W;
  const int* D;
  const long long* off;
  const long long* counters;
  SizedHash hf;
  int dmax;
  long long U;
  double inv_q;
  const long long* nb_idx;  // [m][ld]: row t belongs to users[t]
  const double* nb_sim;
  const int* nb_cnt;
  int ld;
  const long long* item_ptr;
  const int* item_col;
  long long nnz;
  const long long* item_ids;
  long long num_items;
  const long long* users;
  long long m;
  int how_many, include_known;
  long long* out_item;
  float* out_value;
  int* out_cnt;
  unsigned* ws_bitmap;         // [grid][words] when the bitmap does not fit shared memory
  int* ws_cand;                // [grid][num_items]
  unsigned long long* ws_key;  // [grid][num_items]
  float* ws_val;               // [grid][num_items]
  int words, bitmap_smem;
  int stages;
  long long stage_bytes;  // multiple of 16; 0 when there are no stages
  int ch;                 // candidates per chunk (multiple of SR_THREADS, <= SR_KMAX * SR_THREADS)
  unsigned long long* plan;
};

// how neighbour (w, d) is read for a chunk of cn candidates: streamed when its sketch moves fewer bytes than the
// single counters (8*d*w < cn*d*32) -- whole when the sketch's enclosing 16-byte span fits a stage, else row by row
// -- and gathered otherwise, or when even a row does not fit (the span of n cells is at most 8*n + 8 bytes)
__device__ __forceinline__ int sr_mode(const SrArgs& a, int w, int d, int cn) {
  if ((long long)w >= 4ll * cn) return SR_GATHER;
  if ((long long)d * w * 8 + 8 <= a.stage_bytes) return SR_WHOLE;
  if ((long long)w * 8 + 8 <= a.stage_bytes) return SR_ROWS;
  return SR_TOO_WIDE;
}

// cp.async.bulk wants 16-byte-aligned addresses and sizes: the enclosing span of [src, src + n) is copied, and the
// stage is read at the 8-byte skew of src
__device__ __forceinline__ uint32_t span_bytes(const long long* src, long long n) {
  return (uint32_t)((((uintptr_t)src & 15) + (uintptr_t)n * 8 + 15) & ~(uintptr_t)15);
}
__device__ __forceinline__ int span_skew(const long long* src) { return (int)(((uintptr_t)src & 15) >> 3); }

__global__ void __launch_bounds__(SR_THREADS, 1) k_sized_recommend(const SrArgs a) {
  extern __shared__ __align__(16) unsigned char sr_smem[];
  // layout: [stages][stage_bytes] | full barriers [4] | scratch [8] | sort keys [REC_MAX_N] | residues [dmax][ch] |
  // histogram [256] | scan [32] | bitmap [words] (when it fits)
  unsigned char* p = sr_smem;
  unsigned char* stage_base = p;
  p += (size_t)a.stages * a.stage_bytes;
  unsigned long long* full = reinterpret_cast<unsigned long long*>(p);
  p += 8 * 4;
  long long* bcast = reinterpret_cast<long long*>(p);
  p += 8 * 8;
  unsigned long long* sortbuf = reinterpret_cast<unsigned long long*>(p);
  p += REC_MAX_N * 8;
  unsigned long long* res = reinterpret_cast<unsigned long long*>(p);
  p += (size_t)a.dmax * a.ch * 8;
  unsigned* hist = reinterpret_cast<unsigned*>(p);
  p += 256 * 4;
  int* scan_sh = reinterpret_cast<int*>(p);
  p += 32 * 4;
  unsigned* bitmap_sh = reinterpret_cast<unsigned*>(p);

  unsigned* bitmap = a.bitmap_smem ? bitmap_sh : a.ws_bitmap + (size_t)blockIdx.x * a.words;
  int* cand = a.ws_cand + (size_t)blockIdx.x * a.num_items;
  unsigned long long* keys = a.ws_key + (size_t)blockIdx.x * a.num_items;
  float* vals = a.ws_val + (size_t)blockIdx.x * a.num_items;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0 && a.stages) {
    for (int s = 0; s < a.stages; s++) tc05::mbar_init(tc05::smem_u32(&full[s]), 1);
    tc05::mbar_fence_init();
  }
  __syncthreads();
  uint32_t seq = 0;  // stage loads consumed by this CTA so far: stage = seq % stages, parity = (seq / stages) & 1

  for (;;) {
    if (tid == 0) bcast[0] = (long long)atomicAdd(&a.plan[RP_NEXT], 1ull);
    __syncthreads();
    const long long i = bcast[0];
    __syncthreads();
    if (i >= a.m) break;
    long long* out_item = a.out_item + i * a.how_many;
    float* out_value = a.out_value + i * a.how_many;
    for (int t = tid; t < a.how_many; t += SR_THREADS) {
      out_item[t] = -1;
      out_value[t] = 0.0f;
    }
    const long long u = a.users[i];
    const int cnt = a.nb_cnt[i];
    if (u < 0 || u >= a.U || cnt < 0 || cnt > a.ld) {
      if (tid == 0) {
        atomicAdd(&a.plan[RP_BAD], 1ull);
        a.out_cnt[i] = 0;
      }
      continue;
    }
    const long long* nbi = a.nb_idx + i * a.ld;
    const double* nbs = a.nb_sim + i * a.ld;

    // ---- 1. candidates: every index and range is checked before the load it guards --------------------------
    for (int w = tid; w < a.words; w += SR_THREADS) bitmap[w] = 0u;
    __syncthreads();
    int bad = 0, c_eff = 0;
    for (int j = warp; j < cnt; j += SR_THREADS / 32) {
      const long long v = __ldg(nbi + j);
      if (v < 0 || v >= a.U) {
        bad += lane == 0;
        continue;
      }
      const long long lo = __ldg(a.item_ptr + v), hi = __ldg(a.item_ptr + v + 1);
      if (lo < 0 || hi < lo || hi > a.nnz) {
        bad += lane == 0;
        continue;
      }
      for (long long t = lo + lane; t < hi; t += 32) {
        const int it = __ldg(a.item_col + t);
        if (it < 0 || it >= a.num_items) bad++;
        else atomicOr(&bitmap[it >> 5], 1u << (it & 31));
      }
    }
    for (int j = tid; j < cnt; j += SR_THREADS) c_eff += __ldg(nbi + j) != u;
    __syncthreads();
    if (!a.include_known) {
      const long long lo = a.item_ptr[u], hi = a.item_ptr[u + 1];
      if (lo >= 0 && hi >= lo && hi <= a.nnz) {
        for (long long t = lo + tid; t < hi; t += SR_THREADS) {
          const int it = __ldg(a.item_col + t);
          if (it < 0 || it >= a.num_items) bad++;
          else atomicAnd(&bitmap[it >> 5], ~(1u << (it & 31)));
        }
      } else {
        bad += tid == 0;
      }
    }
    int tot_bad = 0, tot_c = 0;
    block_exscan<SR_THREADS>(bad, scan_sh, &tot_bad);
    block_exscan<SR_THREADS>(c_eff, scan_sh, &tot_c);
    c_eff = tot_c;
    if (tot_bad) {  // the neighbour lists or the data model are malformed: no estimates read through them
      if (tid == 0) {
        atomicAdd(&a.plan[RP_BAD], (unsigned long long)tot_bad);
        a.out_cnt[i] = 0;
      }
      continue;
    }
    // compaction: thread tid owns a contiguous run of words (ascending dense order = ascending itemID)
    const int per = (a.words + SR_THREADS - 1) / SR_THREADS;
    const int w0 = tid * per, w1 = min(a.words, w0 + per);
    int mine = 0;
    for (int w = w0; w < w1; w++) mine += __popc(bitmap[w]);
    int C = 0;
    int at = block_exscan<SR_THREADS>(mine, scan_sh, &C);
    for (int w = w0; w < w1; w++) {
      unsigned b = bitmap[w];
      while (b) {
        const int k = __ffs(b) - 1;
        b &= b - 1;
        cand[at++] = w * 32 + k;
      }
    }
    __syncthreads();  // cand[] is read by other threads below

    // ---- 2. estimates, in chunks of candidates; each neighbour streamed or gathered by bytes ----------------
    long long n_stream = 0, n_rows = 0, n_gather = 0, n_wide = 0, s_bytes = 0, g_loads = 0;  // thread 0's plan tallies
    for (int c0 = 0; c0 < C; c0 += a.ch) {
      const int cn = min(a.ch, C - c0);
      const int kk = (cn + SR_THREADS - 1) / SR_THREADS;
      for (int pos = tid; pos < cn; pos += SR_THREADS) {
        const unsigned long long kr = cmh_residue(__ldg(a.item_ids + cand[c0 + pos]));
        for (int r = 0; r < a.dmax; r++) res[(size_t)r * a.ch + pos] = mod_p(a.hf.a[r], a.hf.b[r], kr);
      }
      double pref[SR_KMAX], tot[SR_KMAX];
      int count[SR_KMAX];
      long long mn[SR_KMAX];
#pragma unroll
      for (int k = 0; k < SR_KMAX; k++) {
        pref[k] = 0.0;
        tot[k] = 0.0;
        count[k] = 0;
        mn[k] = 0;
      }
      __syncthreads();
      // producer (thread 0): the next stage load of this chunk, in list order; nothing once the list is done
      const int S = a.stages;
      int pj = 0, pr = 0;
      auto issue = [&](uint32_t slot_seq) {
        for (; pj < cnt; pj++) {
          const long long v = __ldg(nbi + pj);
          if (v == u) continue;
          const int mode = sr_mode(a, __ldg(a.W + v), __ldg(a.D + v), cn);
          if (mode == SR_WHOLE || mode == SR_ROWS) break;
        }
        if (pj >= cnt) return;
        const long long v = __ldg(nbi + pj);
        const int w = __ldg(a.W + v), d = __ldg(a.D + v);
        const bool whole = sr_mode(a, w, d, cn) == SR_WHOLE;
        const long long* src = a.counters + __ldg(a.off + v) + (whole ? 0 : (size_t)pr * w);
        const uint32_t bytes = span_bytes(src, whole ? (long long)d * w : w);
        const int s = slot_seq % S;
        const uint32_t bar = tc05::smem_u32(&full[s]);
        tc05::mbar_expect_tx(bar, bytes);
        bulk_row(tc05::smem_u32(stage_base + (size_t)s * a.stage_bytes),
                 reinterpret_cast<const void*>((uintptr_t)src & ~(uintptr_t)15), bytes, bar);
        s_bytes += bytes;
        if (whole || ++pr == d) {
          pr = 0;
          pj++;
        }
      };
      if (tid == 0)
        for (int t = 0; t < S; t++) issue(seq + t);
      for (int j = 0; j < cnt; j++) {
        const long long v = __ldg(nbi + j);
        if (v == u) continue;
        const int w = __ldg(a.W + v), d = __ldg(a.D + v);
        const unsigned uw = (unsigned)w;
        const long long* sk = a.counters + __ldg(a.off + v);
        const double sim = clamp_sim(__ldg(nbs + j));
        const int mode = sr_mode(a, w, d, cn);
        if (mode == SR_GATHER || mode == SR_TOO_WIDE) {
#pragma unroll
          for (int k = 0; k < SR_KMAX; k++) {
            const int pos = tid + k * SR_THREADS;
            if (k < kk && pos < cn) {
              long long x = __ldg(sk + res[pos] % uw);
              for (int r = 1; r < d; r++) {
                const long long y = __ldg(sk + (size_t)r * w + res[(size_t)r * a.ch + pos] % uw);
                x = y < x ? y : x;
              }
              nb_term(x, a.inv_q, sim, pref[k], tot[k], count[k]);
            }
          }
          if (tid == 0) {
            n_gather++;
            n_wide += mode == SR_TOO_WIDE;
            g_loads += (long long)cn * d;
          }
          continue;
        }
        const bool whole = mode == SR_WHOLE;
        const int loads = whole ? 1 : d;
        for (int r0 = 0; r0 < loads; r0++) {
          const int s = seq % S;
          tc05::mbar_wait(tc05::smem_u32(&full[s]), (seq / S) & 1u);
          const long long* src = sk + (whole ? 0 : (size_t)r0 * w);
          const long long* st = reinterpret_cast<const long long*>(stage_base + (size_t)s * a.stage_bytes) + span_skew(src);
#pragma unroll
          for (int k = 0; k < SR_KMAX; k++) {
            const int pos = tid + k * SR_THREADS;
            if (k < kk && pos < cn) {
              if (whole) {
                long long x = st[res[pos] % uw];
                for (int r = 1; r < d; r++) {
                  const long long y = st[(size_t)r * w + res[(size_t)r * a.ch + pos] % uw];
                  x = y < x ? y : x;
                }
                mn[k] = x;
              } else {
                const long long x = st[res[(size_t)r0 * a.ch + pos] % uw];
                mn[k] = (r0 == 0 || x < mn[k]) ? x : mn[k];
              }
            }
          }
          __syncthreads();  // every thread is done with stage s
          if (tid == 0) issue(seq + S);
          seq++;
        }
#pragma unroll
        for (int k = 0; k < SR_KMAX; k++)
          if (k < kk && tid + k * SR_THREADS < cn) nb_term(mn[k], a.inv_q, sim, pref[k], tot[k], count[k]);
        n_stream += tid == 0;
        n_rows += tid == 0 && !whole;
      }
#pragma unroll
      for (int k = 0; k < SR_KMAX; k++) {
        const int pos = tid + k * SR_THREADS;
        if (k < kk && pos < cn) {
          const float e = nb_result(pref[k], tot[k], count[k]);
          vals[c0 + pos] = e;
          keys[c0 + pos] = rank_key(e, c0 + pos);
        }
      }
      __syncthreads();  // the residues are rewritten by the next chunk
    }
    if (tid == 0) {
      const int nchunks = (C + a.ch - 1) / a.ch;
      atomicAdd(&a.plan[RP_CHUNKS], (unsigned long long)nchunks);
      atomicAdd(&a.plan[RP_CAND_SUM], (unsigned long long)C);
      atomicMax(&a.plan[RP_CAND_MAX], (unsigned long long)C);
      atomicAdd(&a.plan[RP_STREAM], (unsigned long long)n_stream);
      atomicAdd(&a.plan[RP_ROWS], (unsigned long long)n_rows);
      atomicAdd(&a.plan[RP_GATHER], (unsigned long long)n_gather);
      atomicAdd(&a.plan[RP_TOO_WIDE], (unsigned long long)n_wide);
      atomicAdd(&a.plan[RP_STREAM_BYTES], (unsigned long long)s_bytes);
      atomicAdd(&a.plan[RP_GATHER_LOADS], (unsigned long long)g_loads);
      atomicAdd(&a.plan[RP_TERMS], (unsigned long long)C * (unsigned long long)c_eff);
    }

    // ---- 3. top-N ------------------------------------------------------------------------------------------
    const int n_out = topn_keys<SR_THREADS>(keys, C, a.how_many, hist, scan_sh, bcast, sortbuf);
    for (int t = tid; t < n_out; t += SR_THREADS) {
      const int pos = (int)(0xFFFFFFFFu - (uint32_t)sortbuf[t]);
      out_item[t] = __ldg(a.item_ids + cand[pos]);
      out_value[t] = vals[pos];
    }
    if (tid == 0) a.out_cnt[i] = n_out;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host helpers
// ---------------------------------------------------------------------------------------------------------------
SizedDev dev_view(const mb200_sized_bank* bk) {
  SizedDev v;
  v.W = bk->w;
  v.D = bk->d;
  v.off = bk->off;
  v.rowoff = bk->rowoff;
  v.counters = bk->counters;
  v.sumsq = bk->sumsq;
  v.ptr = bk->ptr;
  v.quanta = bk->quanta;
  v.hres = bk->hres;
  v.nnz = bk->nnz;
  v.U = bk->U;
  v.s2 = ldexp(1.0, -2 * bk->frac_bits);
  return v;
}

SizedHash hash_of(const mb200_sized_bank* bk) {
  SizedHash h;
  for (int i = 0; i < MB200_MAX_DEPTH; i++) {
    h.a[i] = bk->a_res[i];
    h.b[i] = bk->b_res[i];
  }
  return h;
}

void free_bank(mb200_sized_bank* bk) {
  void* ptrs[] = {bk->w, bk->d, bk->off, bk->rowoff, bk->counters, bk->sumsq, bk->ptr, bk->quanta, bk->hres, bk->members};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  delete bk;
}

template <typename T>
int dev_alloc(mb200_ctx* ctx, T** p, size_t n) {
  MB_CUDA(ctx, cudaMalloc((void**)p, (n ? n : 1) * sizeof(T)));
  return MB200_OK;
}

// shared-memory budget for query sketches (MB200_SIZED_QSMEM_BYTES overrides it: tests and A/B runs)
size_t qsmem_budget(mb200_ctx* ctx) {
  const char* e = getenv("MB200_SIZED_QSMEM_BYTES");
  size_t b = e ? (size_t)strtoull(e, nullptr, 10) : SZ_QSMEM_DEFAULT;
  const size_t cap = ctx->smem_optin > (size_t)SZ_TQ * 32 * 8 + 1024 ? ctx->smem_optin - SZ_TQ * 32 * 8 - 1024 : 0;
  return b < cap ? b : cap;
}

int create_impl(mb200_ctx* ctx, int64_t U, const int32_t* width, const int32_t* depth, const int64_t* a,
                const int64_t* b, int32_t frac_bits, const int64_t* user_ptr, const int64_t* item, const float* pref,
                mb200_sized_bank* bk) {
  bk->ctx = ctx;
  bk->U = U;
  bk->frac_bits = frac_bits;
  MB_CHECK(dev_alloc(ctx, &bk->w, (size_t)U));
  MB_CHECK(dev_alloc(ctx, &bk->d, (size_t)U));
  MB_CHECK(dev_alloc(ctx, &bk->ptr, (size_t)U + 1));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->w, width, (size_t)U * 4, cudaMemcpyDefault, ctx->stream));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->d, depth, (size_t)U * 4, cudaMemcpyDefault, ctx->stream));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->ptr, user_ptr, ((size_t)U + 1) * 8, cudaMemcpyDefault, ctx->stream));
  StatusWords sw(ctx, SW_WORDS);
  MB_CHECK(sw.zero(WS_STATUS));
  k_sized_validate<<<(unsigned)std::min<int64_t>(ceil_div64(U + 1, 256), 4096), 256, 0, ctx->stream>>>(
      bk->w, bk->d, bk->ptr, U, sw.dev);
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  unsigned long long h[SW_WORDS];
  MB_CHECK(sw.read(h));
  if (h[SW_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_sized_bank_create: %llu width(s) < 1, depth(s) outside [1, %d] or user_ptr entries not "
                      "starting at 0 / not ascending",
                      h[SW_BAD], MB200_MAX_DEPTH);
  // the shapes are host-side set-up: offsets, shape classes
  bk->w_h.resize((size_t)U);
  bk->d_h.resize((size_t)U);
  std::vector<int64_t> ptr_h((size_t)U + 1);
  MB_CUDA(ctx, cudaMemcpyAsync(bk->w_h.data(), bk->w, (size_t)U * 4, cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->d_h.data(), bk->d, (size_t)U * 4, cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaMemcpyAsync(ptr_h.data(), bk->ptr, ((size_t)U + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  bk->nnz = ptr_h[(size_t)U];
  if (bk->nnz > 0 && (!item || !pref))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_bank_create: NULL array argument");
  bk->off_h.assign((size_t)U + 1, 0);
  std::vector<int64_t> rowoff((size_t)U + 1, 0);
  int64_t longest = 0;
  std::map<std::pair<int64_t, std::pair<int32_t, int32_t>>, std::vector<int32_t>> cls;  // (cells, (w, d)) -> rows
  for (int64_t u = 0; u < U; u++) {
    const int64_t c = (int64_t)bk->w_h[u] * bk->d_h[u];
    bk->off_h[u + 1] = bk->off_h[u] + c;
    rowoff[u + 1] = rowoff[u] + bk->d_h[u];
    bk->dmax = std::max(bk->dmax, bk->d_h[u]);
    bk->max_cells = std::max(bk->max_cells, c);
    longest = std::max(longest, ptr_h[u + 1] - ptr_h[u]);
    cls[{c, {bk->w_h[u], bk->d_h[u]}}].push_back((int32_t)u);
  }
  bk->cells = bk->off_h[(size_t)U];
  bk->rows = rowoff[(size_t)U];
  std::vector<int32_t> members;
  members.reserve((size_t)U);
  bk->cptr.assign(1, 0);
  for (auto& kv : cls) {
    bk->cw.push_back(kv.first.second.first);
    bk->cd.push_back(kv.first.second.second);
    members.insert(members.end(), kv.second.begin(), kv.second.end());
    bk->cptr.push_back((int64_t)members.size());
  }
  for (int i = 0; i < bk->dmax; i++) {
    bk->a_res[i] = cmh_residue(a[i]);
    bk->b_res[i] = cmh_residue(b[i]);
  }
  const int64_t nnz = bk->nnz;
  MB_CHECK(dev_alloc(ctx, &bk->off, (size_t)U + 1));
  MB_CHECK(dev_alloc(ctx, &bk->rowoff, (size_t)U + 1));
  // two cells of padding: k_sized_recommend copies the enclosing 16-byte span of the last sketch
  MB_CHECK(dev_alloc(ctx, &bk->counters, (size_t)bk->cells + 2));
  MB_CHECK(dev_alloc(ctx, &bk->sumsq, (size_t)bk->rows));
  MB_CHECK(dev_alloc(ctx, &bk->quanta, (size_t)nnz));
  MB_CHECK(dev_alloc(ctx, &bk->hres, (size_t)nnz * bk->dmax));
  MB_CHECK(dev_alloc(ctx, &bk->members, (size_t)U));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->off, bk->off_h.data(), ((size_t)U + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->rowoff, rowoff.data(), ((size_t)U + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  MB_CUDA(ctx, cudaMemcpyAsync(bk->members, members.data(), (size_t)U * 4, cudaMemcpyHostToDevice, ctx->stream));
  MB_CUDA(ctx, cudaMemsetAsync(bk->counters, 0, (size_t)bk->cells * 8, ctx->stream));
  // the prefs only pass through workspace slots on their way into quanta / hash residues
  void *ditem = nullptr, *dpref = nullptr;
  MB_CHECK(ws_slot(ctx, WS_SIZED_ITEM, (size_t)(nnz ? nnz : 1) * 8, &ditem));
  MB_CHECK(ws_slot(ctx, WS_SIZED_PREF, (size_t)(nnz ? nnz : 1) * 4, &dpref));
  if (nnz) {
    MB_CUDA(ctx, cudaMemcpyAsync(ditem, item, (size_t)nnz * 8, cudaMemcpyDefault, ctx->stream));
    MB_CUDA(ctx, cudaMemcpyAsync(dpref, pref, (size_t)nnz * 4, cudaMemcpyDefault, ctx->stream));
  }
  MB_CHECK(sw.zero(WS_STATUS));
  if (U > 0) {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_sized_build<<<(unsigned)U, SZ_THREADS, 0, ctx->stream>>>(bk->w, bk->d, bk->off, bk->rowoff, bk->ptr,
                                                               (const long long*)ditem, (const float*)dpref, nnz,
                                                               bk->dmax, hash_of(bk), ldexp(1.0, frac_bits),
                                                               bk->counters, bk->sumsq, bk->quanta, bk->hres, sw.dev);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(sw.read(h));
  if (h[SW_INEXACT])
    return mb200_fail(ctx, MB200_ERR_INEXACT,
                      "%llu increment(s) are not multiples of 2^-%d (or not finite): the bank cannot hold them "
                      "exactly; create the bank with a larger frac_bits",
                      h[SW_INEXACT], frac_bits);
  // conservative: a user's prefs all at the largest magnitude seen, all into one counter
  if (h[SW_RANGE] || (double)longest * (double)h[SW_MAXABS] >= 9.0e18)
    return mb200_fail(ctx, MB200_ERR_RANGE,
                      "%llu counter(s) or sketch row(s) beyond the exact range (|counter| or the row's sum of squared "
                      "quanta >= 2^53): use a smaller frac_bits",
                      h[SW_RANGE]);
  return MB200_OK;
}

}  // namespace

extern "C" {

int mb200_sized_bank_create(mb200_ctx* ctx, int64_t users, const int32_t* width, const int32_t* depth, const int64_t* a,
                            const int64_t* b, int32_t frac_bits, const int64_t* user_ptr, const int64_t* item,
                            const float* pref, int mem, mb200_sized_bank** out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_bank_create: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  *out = nullptr;
  if (users < 0 || users >= (1ll << 31) || frac_bits < 0 || frac_bits > 40 ||
      (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_bank_create: bad shape (users=%lld frac_bits=%d)",
                      (long long)users, frac_bits);
  if (!a || !b || !user_ptr || (users > 0 && (!width || !depth)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_bank_create: NULL array argument");
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  mb200_sized_bank* bk = new mb200_sized_bank();
  const int rc = create_impl(ctx, users, width, depth, a, b, frac_bits, user_ptr, item, pref, bk);
  if (rc != MB200_OK) {
    cudaStreamSynchronize(ctx->stream);
    free_bank(bk);
    return rc;
  }
  *out = bk;
  return MB200_OK;
}

int mb200_sized_bank_destroy(mb200_sized_bank* bk) {
  if (!bk) return MB200_OK;
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  free_bank(bk);
  return MB200_OK;
}

int mb200_sized_bank_read(mb200_sized_bank* bk, int64_t user, double* out) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_bank_read: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (user < 0 || user >= bk->U || !out)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_bank_read: user row %lld outside [0, %lld) or NULL out",
                      (long long)user, (long long)bk->U);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t cells = (size_t)(bk->off_h[user + 1] - bk->off_h[user]);
  std::vector<long long> c(cells);
  MB_CUDA(ctx, cudaMemcpyAsync(c.data(), bk->counters + bk->off_h[user], cells * 8, cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->stat_d2h += (int64_t)(cells * 8);
  const double inv_q = ldexp(1.0, -bk->frac_bits);
  for (size_t i = 0; i < cells; i++) out[i] = (double)c[i] * inv_q;  // |c| < 2^53: checked at creation
  return MB200_OK;
}

int mb200_sized_pair_cosine(mb200_sized_bank* bk, const int64_t* u1, const int64_t* u2, int64_t n, double* out,
                            int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_pair_cosine: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 0 || (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_pair_cosine: bad shape (n=%lld)", (long long)n);
  if (n == 0) return MB200_OK;
  if (!u1 || !u2 || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_pair_cosine: NULL array argument");
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ArgStage st(ctx, mem);
  const long long *d1, *d2;
  double* dout;
  MB_CHECK(st.in((const long long*)u1, (size_t)n, &d1));
  MB_CHECK(st.in((const long long*)u2, (size_t)n, &d2));
  MB_CHECK(st.out(out, (size_t)n, &dout));
  const int64_t slice = bk->max_cells > 0 ? bk->max_cells : 1;
  int64_t grid = std::min<int64_t>(n, (int64_t)ctx->num_sms * 2);
  grid = std::max<int64_t>(1, std::min<int64_t>(grid, (int64_t)(SZ_DENSE / ((size_t)slice * 8))));
  void* slices = nullptr;
  MB_CHECK(ws_slot(ctx, WS_SIZED_SLICE, (size_t)grid * slice * 8, &slices));
  StatusWords sw(ctx, SW_WORDS);
  MB_CHECK(sw.zero(WS_STATUS));
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_sized_pair<<<(unsigned)grid, SZ_THREADS, 0, ctx->stream>>>(dev_view(bk), d1, d2, n, (long long*)slices, slice,
                                                                  dout, sw.dev);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[SW_WORDS];
  MB_CHECK(sw.read(h));
  if (h[SW_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_pair_cosine: %llu user row(s) outside [0, %lld)", h[SW_BAD],
                      (long long)bk->U);
  if (h[SW_RANGE])
    return mb200_fail(ctx, MB200_ERR_RANGE,
                      "mb200_sized_pair_cosine: %llu re-sketched row(s) reach 2^53 quanta^2: the FP64 sums would not "
                      "be exact; use a smaller frac_bits",
                      h[SW_RANGE]);
  return MB200_OK;
}

int mb200_sized_neighborhood(mb200_sized_bank* bk, const int64_t* query_rows, int64_t q, int32_t n,
                             double min_similarity, int64_t* out_idx, double* out_sim, int32_t* out_cnt, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_neighborhood: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (n < 1 || n > SEL_MAX_N)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_neighborhood: n must be in [1, %d] (got %d)", SEL_MAX_N, n);
  if (q < 0 || min_similarity != min_similarity || (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_neighborhood: bad shape (q=%lld) or NaN min_similarity",
                      (long long)q);
  if (q == 0) return MB200_OK;
  if (!query_rows || !out_idx || !out_sim || !out_cnt)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_neighborhood: NULL array argument");
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ArgStage st(ctx, mem);
  const long long* dq;
  long long* didx;
  double* dsim;
  int* dcnt;
  MB_CHECK(st.in((const long long*)query_rows, (size_t)q, &dq));
  MB_CHECK(st.out((long long*)out_idx, (size_t)q * n, &didx));
  MB_CHECK(st.out(out_sim, (size_t)q * n, &dsim));
  MB_CHECK(st.out((int*)out_cnt, (size_t)q, &dcnt));
  StatusWords sw(ctx, SW_WORDS);
  MB_CHECK(sw.zero(WS_STATUS));
  k_sized_check_rows<<<(unsigned)std::min<int64_t>(ceil_div64(q, 256), 4096), 256, 0, ctx->stream>>>(dq, q, bk->U,
                                                                                                       sw.dev);
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  unsigned long long h[SW_WORDS];
  MB_CHECK(sw.read(h));
  if (h[SW_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_neighborhood: %llu query row(s) outside [0, %lld)", h[SW_BAD],
                      (long long)bk->U);

  // per class: query tile, accumulator path, members per work item
  const int C = (int)bk->cw.size();
  const size_t qbudget = qsmem_budget(ctx);
  std::vector<int> ctile(C), cglob(C), cmem(C);
  int64_t slice_cells = 1, pair_fmas = 0, smem_classes = 0, global_classes = 0;
  int tile_max = 0;
  size_t qsmem_used = 0;
  for (int c = 0; c < C; c++) {
    const int64_t cells = (int64_t)bk->cw[c] * bk->cd[c];
    int64_t t = (int64_t)(qbudget / ((size_t)cells * 8));
    if (t >= 1) {
      ctile[c] = (int)std::min<int64_t>(t, SZ_TQ);
      cglob[c] = 0;
      smem_classes++;
      qsmem_used = std::max(qsmem_used, (size_t)ctile[c] * cells * 8);
    } else {
      ctile[c] = (int)std::max<int64_t>(1, std::min<int64_t>(SZ_TQ, (int64_t)(SZ_GSLICE / ((size_t)cells * 8))));
      cglob[c] = 1;
      global_classes++;
      slice_cells = std::max(slice_cells, (int64_t)ctile[c] * cells);
    }
    tile_max = std::max(tile_max, ctile[c]);
    const int64_t m = ((1ll << 21) / ((int64_t)ctile[c] * cells) + SZ_MQ - 1) / SZ_MQ * SZ_MQ;
    cmem[c] = (int)std::max<int64_t>(SZ_MQ, std::min<int64_t>(m, 4096));
    pair_fmas += q * (bk->cptr[c + 1] - bk->cptr[c]) * cells;
  }
  const int64_t U = bk->U;
  const int64_t qb = std::max<int64_t>(1, std::min<int64_t>(q, (int64_t)(SZ_DENSE / ((size_t)std::max<int64_t>(U, 1) * 8))));
  const int grid = ctx->num_sms * 2;
  const size_t smem = (size_t)SZ_TQ * 32 * 8 + qsmem_used;
  void *wsims = nullptr, *wslice = nullptr, *wcls = nullptr, *witems = nullptr;
  MB_CHECK(ws_slot(ctx, WS_SIZED_SIMS, (size_t)qb * std::max<int64_t>(U, 1) * 8, &wsims));
  MB_CHECK(ws_slot(ctx, WS_SIZED_SLICE, global_classes ? (size_t)grid * slice_cells * 8 : 8, &wslice));
  MB_CHECK(ws_slot(ctx, WS_SIZED_CLASSES, (size_t)std::max(C, 1) * 4 * 4, &wcls));
  std::vector<int> hcls((size_t)std::max(C, 1) * 4);
  for (int c = 0; c < C; c++) {
    hcls[c] = bk->cw[c];
    hcls[(size_t)C + c] = bk->cd[c];
    hcls[(size_t)2 * C + c] = ctile[c];
    hcls[(size_t)3 * C + c] = cglob[c];
  }
  MB_CUDA(ctx, cudaMemcpyAsync(wcls, hcls.data(), hcls.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  MB_CUDA(ctx, cudaFuncSetAttribute(k_sized_score, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  std::vector<SzItem> items;
  int64_t batches = 0, n_items_total = 0;
  for (int64_t q0 = 0; q0 < q; q0 += qb) {
    const int64_t nq = std::min<int64_t>(qb, q - q0);
    items.clear();
    for (int c = 0; c < C; c++)
      for (int64_t m0 = bk->cptr[c]; m0 < bk->cptr[c + 1]; m0 += cmem[c])
        for (int64_t t0 = 0; t0 < nq; t0 += ctile[c])
          items.push_back({c, (int)m0, (int)std::min<int64_t>(cmem[c], bk->cptr[c + 1] - m0), (int)t0});
    // the staging slot of the items is refilled per batch: the previous batch must be done with it
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    MB_CHECK(ws_slot(ctx, WS_SIZED_ITEMS, std::max<size_t>(items.size(), 1) * sizeof(SzItem), &witems));
    MB_CUDA(ctx, cudaMemcpyAsync(witems, items.data(), items.size() * sizeof(SzItem), cudaMemcpyHostToDevice,
                                 ctx->stream));
    MB_CUDA(ctx, cudaMemsetAsync(sw.dev + SW_NEXT, 0, 8, ctx->stream));
    ScoreArgs a;
    a.b = dev_view(bk);
    a.members = bk->members;
    a.cw = (const int*)wcls;
    a.cd = a.cw + C;
    a.ctile = a.cw + 2 * C;
    a.cglobal = a.cw + 3 * C;
    a.items = (const SzItem*)witems;
    a.n_items = (long long)items.size();
    a.queries = dq + q0;
    a.nq = nq;
    a.sims = (double*)wsims;
    a.gslice = (long long*)wslice;
    a.slice_cells = slice_cells;
    a.sw = sw.dev;
    {
      ProfScope prof(ctx, MB200_K_RECOMMEND);
      k_sized_score<<<grid, SZ_THREADS, smem, ctx->stream>>>(a);
    }
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
    {
      ProfScope prof(ctx, MB200_K_RECOMMEND);
      k_sized_select<<<(unsigned)nq, SEL_THREADS, 0, ctx->stream>>>((const double*)wsims, U, n, min_similarity,
                                                                    didx + q0 * n, dsim + q0 * n, dcnt + q0);
    }
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
    batches++;
    n_items_total += (int64_t)items.size();
  }
  MB_CHECK(st.finish());
  MB_CHECK(sw.read(h));
  mb200_sized_plan& pl = ctx->last_sized_plan;
  pl.queries = q;
  pl.classes = C;
  pl.smem_classes = smem_classes;
  pl.global_classes = global_classes;
  pl.pair_fmas = pair_fmas;
  pl.batches = batches;
  pl.items = n_items_total;
  pl.query_tile_max = tile_max;
  pl.smem_bytes = (int32_t)qbudget;
  if (getenv("MB200_TRACE"))
    fprintf(stderr,
            "[mb200 trace] sized plan: queries=%lld classes=%d smem_classes=%lld global_classes=%lld pair_fmas=%lld "
            "batches=%lld items=%lld tile_max=%d qsmem=%zu users=%lld\n",
            (long long)q, C, (long long)smem_classes, (long long)global_classes, (long long)pair_fmas,
            (long long)batches, (long long)n_items_total, tile_max, qbudget, (long long)U);
  if (h[SW_RANGE])
    return mb200_fail(ctx, MB200_ERR_RANGE,
                      "mb200_sized_neighborhood: %llu re-sketched row(s) reach 2^53 quanta^2: the FP64 sums would not "
                      "be exact; use a smaller frac_bits",
                      h[SW_RANGE]);
  return MB200_OK;
}

int mb200_sized_estimate_prefs(mb200_sized_bank* bk, const int64_t* nb_idx, const double* nb_sim,
                               const int32_t* nb_cnt, int64_t nb_rows, int32_t nb_ld, const int64_t* user,
                               const int64_t* nb_row, const int64_t* item_id, int64_t q, float* out, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_estimate_prefs: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (q < 0 || nb_rows < 0 || nb_ld < 1 || (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_estimate_prefs: bad shape (q=%lld nb_rows=%lld nb_ld=%d)",
                      (long long)q, (long long)nb_rows, nb_ld);
  if (q == 0) return MB200_OK;
  if (!user || !item_id || !out || (nb_rows > 0 && (!nb_idx || !nb_sim || !nb_cnt)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_estimate_prefs: NULL array argument");
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  ArgStage st(ctx, mem);
  const long long *d_idx, *d_user, *d_row, *d_item;
  const double* d_sim;
  const int* d_cnt;
  float* d_out;
  const size_t nbc = (size_t)nb_rows * nb_ld;
  MB_CHECK(st.in((const long long*)nb_idx, nbc, &d_idx));
  MB_CHECK(st.in(nb_sim, nbc, &d_sim));
  MB_CHECK(st.in((const int*)nb_cnt, (size_t)nb_rows, &d_cnt));
  MB_CHECK(st.in((const long long*)user, (size_t)q, &d_user));
  MB_CHECK(st.in((const long long*)nb_row, nb_row ? (size_t)q : 0, &d_row));
  MB_CHECK(st.in((const long long*)item_id, (size_t)q, &d_item));
  MB_CHECK(st.out(out, (size_t)q, &d_out));
  StatusWords sw(ctx, SW_WORDS);
  MB_CHECK(sw.zero(WS_STATUS));
  const int dmax = bk->dmax > 0 ? bk->dmax : 1;
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_sized_estimate<<<(unsigned)ceil_div64(q, EST_THREADS), EST_THREADS, (size_t)dmax * EST_THREADS * 8, ctx->stream>>>(
        dev_view(bk), hash_of(bk), bk->dmax, ldexp(1.0, -bk->frac_bits), d_idx, d_sim, d_cnt, nb_rows, nb_ld, d_user,
        d_row, d_item, q, d_out, sw.dev);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[SW_WORDS];
  MB_CHECK(sw.read(h));
  if (h[SW_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_sized_estimate_prefs: %llu user row(s), neighbourhood row(s), counts or neighbour "
                      "index(es) out of range (users %lld, neighbourhood rows %lld, nb_ld %d)",
                      h[SW_BAD], (long long)bk->U, (long long)nb_rows, nb_ld);
  return MB200_OK;
}

int mb200_sized_recommend(mb200_sized_bank* bk, const int64_t* nb_idx, const double* nb_sim, const int32_t* nb_cnt,
                          int32_t nb_ld, const int64_t* item_ptr, const int32_t* item_col, int64_t nnz,
                          const int64_t* item_ids, int64_t num_items, const int64_t* users, int64_t m,
                          int32_t how_many, int include_known, int64_t* out_item, float* out_value, int32_t* out_cnt,
                          int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_recommend: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (how_many < 1 || how_many > REC_MAX_N)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_recommend: how_many must be in [1, %d] (got %d)", REC_MAX_N,
                      how_many);
  if (m < 0 || nb_ld < 1 || nnz < 0 || num_items < 0 || num_items >= (1LL << 31) ||
      (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_sized_recommend: bad shape (m=%lld nb_ld=%d nnz=%lld num_items=%lld)", (long long)m, nb_ld,
                      (long long)nnz, (long long)num_items);
  if (m == 0) return MB200_OK;
  if (!nb_idx || !nb_sim || !nb_cnt || !item_ptr || (nnz > 0 && !item_col) || (num_items > 0 && !item_ids) || !users ||
      !out_item || !out_value || !out_cnt)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_recommend: NULL array argument");
  const int64_t U = bk->U;
  if (mem == MB200_MEM_HOST) {
    // the data model is host memory: its shape can be checked here
    if (item_ptr[0] != 0 || item_ptr[U] != nnz)
      return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                        "mb200_sized_recommend: item_ptr[0] must be 0 and item_ptr[users] = nnz (%lld)", (long long)nnz);
    for (int64_t t = 1; t < num_items; t++)
      if (item_ids[t] <= item_ids[t - 1])
        return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_recommend: item_ids must be strictly ascending");
  }
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const int dmax = bk->dmax > 0 ? bk->dmax : 1;
  const long long words = (num_items + 31) / 32;
  const bool bitmap_smem = words <= SR_BITMAP_SMEM_WORDS;
  int ch = SR_RES_BYTES / (8 * dmax) / SR_THREADS * SR_THREADS;
  ch = std::max(SR_THREADS, std::min(ch, SR_KMAX * SR_THREADS));
  const size_t fixed = 8 * 4 + 8 * 8 + REC_MAX_N * 8 + (size_t)dmax * ch * 8 + 256 * 4 + 32 * 4 +
                       (bitmap_smem ? (size_t)words * 4 : 0);
  // the ring takes what shared memory is left, in SR_STAGES equal stages (MB200_SIZED_REC_STAGE_BYTES caps a stage:
  // tests and A/B runs)
  long long stage_bytes = ctx->smem_optin > fixed ? (long long)((ctx->smem_optin - fixed) / SR_STAGES) & ~15ll : 0;
  if (const char* e = getenv("MB200_SIZED_REC_STAGE_BYTES"))
    stage_bytes = std::min<long long>(stage_bytes, strtoll(e, nullptr, 10) & ~15ll);
  const int stages = stage_bytes >= 32 ? SR_STAGES : 0;
  if (!stages) stage_bytes = 0;
  const size_t smem = fixed + (size_t)stages * stage_bytes;
  const int grid = (int)std::min<int64_t>(m, ctx->num_sms);

  ArgStage st(ctx, mem);
  SrArgs a;
  a.W = bk->w;
  a.D = bk->d;
  a.off = bk->off;
  a.counters = bk->counters;
  a.hf = hash_of(bk);
  a.dmax = dmax;
  a.U = U;
  a.inv_q = ldexp(1.0, -bk->frac_bits);
  a.ld = nb_ld;
  a.nnz = nnz;
  a.num_items = num_items;
  a.m = m;
  a.how_many = how_many;
  a.include_known = include_known != 0;
  a.words = (int)words;
  a.bitmap_smem = bitmap_smem;
  a.stages = stages;
  a.stage_bytes = stage_bytes;
  a.ch = ch;
  const size_t nbc = (size_t)m * nb_ld;
  MB_CHECK(st.in((const long long*)nb_idx, nbc, &a.nb_idx));
  MB_CHECK(st.in(nb_sim, nbc, &a.nb_sim));
  MB_CHECK(st.in((const int*)nb_cnt, (size_t)m, &a.nb_cnt));
  MB_CHECK(st.in((const long long*)item_ptr, (size_t)U + 1, &a.item_ptr));
  MB_CHECK(st.in((const int*)item_col, (size_t)nnz, &a.item_col));
  MB_CHECK(st.in((const long long*)item_ids, (size_t)num_items, &a.item_ids));
  MB_CHECK(st.in((const long long*)users, (size_t)m, &a.users));
  MB_CHECK(st.out((long long*)out_item, (size_t)m * how_many, &a.out_item));
  MB_CHECK(st.out(out_value, (size_t)m * how_many, &a.out_value));
  MB_CHECK(st.out((int*)out_cnt, (size_t)m, &a.out_cnt));
  void *wb = nullptr, *wc = nullptr, *wk = nullptr, *wv = nullptr;
  const size_t per = (size_t)(num_items > 0 ? num_items : 1);
  MB_CHECK(ws_slot(ctx, WS_REC_BITMAP, bitmap_smem ? 4 : (size_t)grid * words * 4, &wb));
  MB_CHECK(ws_slot(ctx, WS_REC_CAND, (size_t)grid * per * 4, &wc));
  MB_CHECK(ws_slot(ctx, WS_REC_KEY, (size_t)grid * per * 8, &wk));
  MB_CHECK(ws_slot(ctx, WS_REC_VAL, (size_t)grid * per * 4, &wv));
  StatusWords plan(ctx, RP_WORDS);
  MB_CHECK(plan.zero(WS_STATUS));
  a.ws_bitmap = (unsigned*)wb;
  a.ws_cand = (int*)wc;
  a.ws_key = (unsigned long long*)wk;
  a.ws_val = (float*)wv;
  a.plan = plan.dev;
  MB_CUDA(ctx, cudaFuncSetAttribute(k_sized_recommend, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_sized_recommend<<<grid, SR_THREADS, smem, ctx->stream>>>(a);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[RP_WORDS];
  MB_CHECK(plan.read(h));
  mb200_sized_recommend_plan& pl = ctx->last_sized_recommend_plan;
  pl.users = m;
  pl.chunks = (int64_t)h[RP_CHUNKS];
  pl.candidates = (int64_t)h[RP_CAND_SUM];
  pl.candidates_max = (int64_t)h[RP_CAND_MAX];
  pl.stream_visits = (int64_t)h[RP_STREAM];
  pl.row_visits = (int64_t)h[RP_ROWS];
  pl.gather_visits = (int64_t)h[RP_GATHER];
  pl.too_wide_visits = (int64_t)h[RP_TOO_WIDE];
  pl.stream_bytes = (int64_t)h[RP_STREAM_BYTES];
  pl.gather_loads = (int64_t)h[RP_GATHER_LOADS];
  pl.terms = (int64_t)h[RP_TERMS];
  pl.stages = stages;
  pl.stage_bytes = (int32_t)stage_bytes;
  pl.chunk_candidates = ch;
  if (getenv("MB200_TRACE"))
    fprintf(stderr,
            "[mb200 trace] sized recommend plan: users=%lld chunks=%lld candidates=%lld max=%lld stream=%lld "
            "rows=%lld gather=%lld too_wide=%lld stream_bytes=%lld gather_loads=%lld terms=%lld stages=%d stage_bytes=%lld "
            "chunk=%d bitmap=%s\n",
            (long long)m, (long long)pl.chunks, (long long)pl.candidates, (long long)pl.candidates_max,
            (long long)pl.stream_visits, (long long)pl.row_visits, (long long)pl.gather_visits, (long long)pl.too_wide_visits,
            (long long)pl.stream_bytes, (long long)pl.gather_loads, (long long)pl.terms, stages, stage_bytes, ch,
            bitmap_smem ? "smem" : "global");
  if (h[RP_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_sized_recommend: %llu user row(s), neighbour count(s) or index(es), item_ptr range(s) or "
                      "item_col entr(ies) out of range (users %lld, num_items %lld, nnz %lld, nb_ld %d)",
                      h[RP_BAD], (long long)U, (long long)num_items, (long long)nnz, nb_ld);
  return MB200_OK;
}

int mb200_sized_recommend_last_plan(mb200_ctx* ctx, mb200_sized_recommend_plan* out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_recommend_last_plan: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  *out = ctx->last_sized_recommend_plan;
  return MB200_OK;
}

int mb200_sized_last_plan(mb200_ctx* ctx, mb200_sized_plan* out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_sized_last_plan: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  *out = ctx->last_sized_plan;
  return MB200_OK;
}

}  // extern "C"
