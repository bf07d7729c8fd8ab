// recommend.cu -- GenericUserBasedRecommender on the sketch bank: doEstimatePreference for (user, item) queries and
// recommend(user, howMany) for many users, over the neighbourhood lists of mb200_bank_cosine_topk.
//
// Reference semantics (GenericUserBasedRecommender.java:134-184 with CosineCM's point query, restated in DESIGN.md
// section 7): for user row u and item i, the listed neighbours v != u are visited in list order;
//   p = (float) min_r C[v][r][h_r(i)] * 2^-frac_bits,  s = clamp(sim, -1, 1) (NaN stays NaN)
//   if p != 0 and s is not NaN: pref += s * (double) p; tot += s; count++      (product and sum rounded separately)
//   estimate = count <= 1 ? NaN : (float) (pref / tot)
// recommend: candidates = items of the listed neighbours (minus the user's own unless include_known), NaN estimates
// dropped, ranked by (value desc, itemID asc), the first how_many kept.
//
// K_RECOMMEND is one persistent CTA per SM, one user at a time:
//   1. candidates: the neighbours' item rows OR-ed into a bitmap (shared memory, or a per-CTA global slice), the own
//      items cleared, compacted in ascending dense order (= ascending itemID);
//   2. estimates, in chunks of up to CH candidates (d hash columns each, cached in shared memory):
//      STREAM  every neighbour's sketch row (W x 8 bytes) is staged into shared memory with cp.async.bulk through an
//              mbarrier ring of 2..4 stages and read at the candidates' columns;
//      GATHER  d 8-byte loads per (candidate, neighbour) from HBM -- the loop of k_estimate_prefs (nb_term);
//      the cheaper by bytes (c*d*W*8 per chunk against C*c*d*32) is taken per user; rows that do not fit twice in
//      shared memory always gather;
//   3. top-N by radix select on (value, position) keys + a bitonic sort of the survivors in shared memory.
//
// k_itembased: RecommenderJob's aggregate-and-recommend phase over the item top-k lists (DESIGN.md section 3) --
// per user, the considered prefs' lists are summed into an open-addressing table in shared memory or a dense
// per-CTA slice (chosen from the entry count), then the same top-N as k_recommend.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "nb_terms.cuh"
#include "rec_topn.cuh"
#include "tc05.cuh"

namespace {

constexpr int REC_THREADS = 512;
constexpr int REC_KMAX = 8;                  // candidates per thread and chunk
constexpr int REC_BITMAP_SMEM_WORDS = 4096;  // 131072 items: larger catalogues use a per-CTA global bitmap
constexpr int REC_COLS_BYTES = 64 * 1024;    // shared memory for the candidates' hash columns
constexpr int EST_THREADS = 128;

// plan / error words of one call
enum { PL_STREAM = 0, PL_GATHER, PL_CHUNKS, PL_CAND_SUM, PL_CAND_MAX, PL_STREAM_ROWS, PL_GATHER_LOADS, PL_BAD,
       PL_NEXT, PL_WORDS };

struct RecArgs {
  const long long* counters;
  HashFamily hf;
  long long E;
  double inv_q;
  const long long* nb_idx;
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
  unsigned* ws_bitmap;   // [grid][words] when the bitmap does not fit shared memory
  int* ws_cand;          // [grid][num_items]
  unsigned long long* ws_key;  // [grid][num_items]
  float* ws_val;         // [grid][num_items]
  int words, bitmap_smem;
  int stages;            // 0: rows cannot be staged (gather only)
  int ch;                // candidates per chunk (multiple of REC_THREADS, <= REC_KMAX * REC_THREADS)
  unsigned long long* plan;
};

// min over the d rows of sketch `sk` at the columns cols[r * stride] -- DoubleCountMinSketch.get on int64 quanta
// (the conversion to double is exact and monotone, so the min commutes with it)
__device__ __forceinline__ long long gather_min(const long long* __restrict__ sk, const uint32_t* cols, int stride,
                                                int d, uint32_t W) {
  long long mn = __ldg(sk + cols[0]);
  for (int r = 1; r < d; r++) {
    const long long x = __ldg(sk + (size_t)r * W + cols[(size_t)r * stride]);
    mn = x < mn ? x : mn;
  }
  return mn;
}

__device__ __forceinline__ uint32_t item_column(const HashFamily& hf, int r, uint64_t kr) {
  return cmh_column(hf.a[r], hf.b[r], kr, hf.w, hf.wmask);
}

// ---------------------------------------------------------------------------------------------------------------
// doEstimatePreference for q (user row, itemID) pairs: one thread per query, the d columns of the item computed once
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(EST_THREADS) k_estimate_prefs(
    const long long* __restrict__ counters, HashFamily hf, long long E, double inv_q,
    const long long* __restrict__ nb_idx, const double* __restrict__ nb_sim, const int* __restrict__ nb_cnt,
    long long nb_rows, int ld, const long long* __restrict__ user, const long long* __restrict__ nb_row,
    const long long* __restrict__ item_id, long long q, float* __restrict__ out, unsigned long long* plan) {
  extern __shared__ uint32_t est_cols[];  // [d][EST_THREADS]
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= q) return;
  uint32_t* cols = est_cols + threadIdx.x;
  const long long u = user[t];
  const long long row = nb_row ? nb_row[t] : u;
  const float nanf_ = __int_as_float(0x7fc00000);
  if (u < 0 || u >= E || row < 0 || row >= nb_rows) {
    atomicAdd(&plan[PL_BAD], 1ull);
    out[t] = nanf_;
    return;
  }
  const int cnt = nb_cnt[row];
  if (cnt < 0 || cnt > ld) {
    atomicAdd(&plan[PL_BAD], 1ull);
    out[t] = nanf_;
    return;
  }
  const uint64_t kr = cmh_residue(item_id[t]);
  for (int r = 0; r < hf.d; r++) cols[r * EST_THREADS] = item_column(hf, r, kr);
  const size_t cells = (size_t)hf.d * hf.w;
  double pref = 0.0, tot = 0.0;
  int count = 0;
  for (int j = 0; j < cnt; j++) {
    const long long v = nb_idx[row * ld + j];
    if (v == u) continue;
    if (v < 0 || v >= E) {
      atomicAdd(&plan[PL_BAD], 1ull);
      continue;
    }
    const long long mn = gather_min(counters + (size_t)v * cells, cols, EST_THREADS, hf.d, hf.w);
    nb_term(mn, inv_q, clamp_sim(nb_sim[row * ld + j]), pref, tot, count);
  }
  out[t] = nb_result(pref, tot, count);
}

// ---------------------------------------------------------------------------------------------------------------
// K_RECOMMEND
// ---------------------------------------------------------------------------------------------------------------
// the listed neighbour slot j of user u: its row, or -1 when it is skipped (the user itself, or out of range)
__device__ __forceinline__ long long nb_at(const RecArgs& a, long long u, int j) {
  const long long v = __ldg(a.nb_idx + u * a.ld + j);
  return (v == u || v < 0 || v >= a.E) ? -1 : v;
}

__global__ void __launch_bounds__(REC_THREADS, 1) k_recommend(const RecArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int d = a.hf.d;
  const uint32_t W = a.hf.w;
  const uint32_t row_bytes = W * 8u;
  // layout: [stages][row] | full barriers [4] | scratch [8] | sort keys [REC_MAX_N] | cols [d][ch] | histogram [256] |
  // scan [32] | bitmap [words] (when it fits)
  unsigned char* p = smem;
  unsigned char* stage_base = p;
  p += (size_t)a.stages * row_bytes;
  unsigned long long* full = reinterpret_cast<unsigned long long*>(p);
  p += 8 * 4;
  long long* bcast = reinterpret_cast<long long*>(p);
  p += 8 * 8;
  unsigned long long* sortbuf = reinterpret_cast<unsigned long long*>(p);
  p += REC_MAX_N * 8;
  uint32_t* cols = reinterpret_cast<uint32_t*>(p);
  p += (size_t)d * a.ch * 4;
  unsigned* hist = reinterpret_cast<unsigned*>(p);
  p += 256 * 4;
  int* scan_sh = reinterpret_cast<int*>(p);
  p += 32 * 4;
  unsigned* bitmap_sh = reinterpret_cast<unsigned*>(p);

  unsigned* bitmap = a.bitmap_smem ? bitmap_sh : a.ws_bitmap + (size_t)blockIdx.x * a.words;
  int* cand = a.ws_cand + (size_t)blockIdx.x * a.num_items;
  unsigned long long* keys = a.ws_key + (size_t)blockIdx.x * a.num_items;
  float* vals = a.ws_val + (size_t)blockIdx.x * a.num_items;
  const size_t cells = (size_t)d * W;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0 && a.stages) {
    for (int s = 0; s < a.stages; s++) tc05::mbar_init(tc05::smem_u32(&full[s]), 1);
    tc05::mbar_fence_init();
  }
  __syncthreads();
  uint32_t seq = 0;  // rows consumed by this CTA so far: stage = seq % stages, parity = (seq / stages) & 1

  for (;;) {
    if (tid == 0) bcast[0] = (long long)atomicAdd(&a.plan[PL_NEXT], 1ull);
    __syncthreads();
    const long long i = bcast[0];
    __syncthreads();
    if (i >= a.m) break;
    long long* out_item = a.out_item + i * a.how_many;
    float* out_value = a.out_value + i * a.how_many;
    for (int t = tid; t < a.how_many; t += REC_THREADS) {
      out_item[t] = -1;
      out_value[t] = 0.0f;
    }
    const long long u = a.users[i];
    int cnt = (u >= 0 && u < a.E) ? a.nb_cnt[u] : -1;
    if (cnt < 0 || cnt > a.ld) {
      if (tid == 0) {
        atomicAdd(&a.plan[PL_BAD], 1ull);
        a.out_cnt[i] = 0;
      }
      continue;
    }

    // ---- 1. candidates -------------------------------------------------------------------------------------
    for (int w = tid; w < a.words; w += REC_THREADS) bitmap[w] = 0u;
    __syncthreads();
    int bad = 0, c_eff = 0;
    for (int j = warp; j < cnt; j += REC_THREADS / 32) {
      const long long v = __ldg(a.nb_idx + u * a.ld + j);
      if (v < 0 || v >= a.E) {
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
    for (int j = tid; j < cnt; j += REC_THREADS) c_eff += nb_at(a, u, j) >= 0;
    __syncthreads();
    if (!a.include_known) {
      const long long lo = a.item_ptr[u], hi = a.item_ptr[u + 1];
      if (lo >= 0 && hi >= lo && hi <= a.nnz) {
        for (long long t = lo + tid; t < hi; t += REC_THREADS) {
          const int it = __ldg(a.item_col + t);
          if (it < 0 || it >= a.num_items) bad++;
          else atomicAnd(&bitmap[it >> 5], ~(1u << (it & 31)));
        }
      } else {
        bad += tid == 0;
      }
    }
    __syncthreads();
    // compaction: thread tid owns a contiguous run of words
    const int per = (a.words + REC_THREADS - 1) / REC_THREADS;
    const int w0 = tid * per, w1 = min(a.words, w0 + per);
    int mine = 0;
    for (int w = w0; w < w1; w++) mine += __popc(bitmap[w]);
    int C = 0;
    int at = block_exscan<REC_THREADS>(mine, scan_sh, &C);
    for (int w = w0; w < w1; w++) {
      unsigned b = bitmap[w];
      while (b) {
        const int k = __ffs(b) - 1;
        b &= b - 1;
        cand[at++] = w * 32 + k;
      }
    }
    int tot_bad = 0, tot_c = 0;
    block_exscan<REC_THREADS>(bad, scan_sh, &tot_bad);
    block_exscan<REC_THREADS>(c_eff, scan_sh, &tot_c);
    c_eff = tot_c;
    if (tot_bad && tid == 0) atomicAdd(&a.plan[PL_BAD], (unsigned long long)tot_bad);
    // cand[] is written by other threads of the block: ordered by the barriers of the scans above

    // ---- 2. estimates -------------------------------------------------------------------------------------
    const int nchunks = (C + a.ch - 1) / a.ch;
    const bool stream = a.stages > 0 && c_eff > 0 && (unsigned long long)W * nchunks < 4ull * (unsigned long long)C;
    if (tid == 0) {
      atomicAdd(&a.plan[stream ? PL_STREAM : PL_GATHER], 1ull);
      atomicAdd(&a.plan[PL_CHUNKS], (unsigned long long)nchunks);
      atomicAdd(&a.plan[PL_CAND_SUM], (unsigned long long)C);
      atomicMax(&a.plan[PL_CAND_MAX], (unsigned long long)C);
      if (stream) atomicAdd(&a.plan[PL_STREAM_ROWS], (unsigned long long)c_eff * d * nchunks);
      else atomicAdd(&a.plan[PL_GATHER_LOADS], (unsigned long long)C * c_eff * d);
    }
    for (int c0 = 0; c0 < C; c0 += a.ch) {
      const int cn = min(a.ch, C - c0);
      const int kk = (cn + REC_THREADS - 1) / REC_THREADS;
      for (int pos = tid; pos < cn; pos += REC_THREADS) {
        const uint64_t kr = cmh_residue(__ldg(a.item_ids + cand[c0 + pos]));
        for (int r = 0; r < d; r++) cols[r * a.ch + pos] = item_column(a.hf, r, kr);
      }
      double pref[REC_KMAX], tot[REC_KMAX];
      int count[REC_KMAX];
      long long mn[REC_KMAX];
#pragma unroll
      for (int k = 0; k < REC_KMAX; k++) {
        pref[k] = 0.0;
        tot[k] = 0.0;
        count[k] = 0;
        mn[k] = 0;
      }
      __syncthreads();
      if (stream) {
        const int S = a.stages;
        const uint32_t T = (uint32_t)c_eff * d;
        // producer cursor (thread 0 only): neighbour slot and depth row of the next row to issue
        int pj = 0, pr = 0;
        auto issue = [&](uint32_t slot_seq) {
          while (nb_at(a, u, pj) < 0) pj++;
          const long long v = nb_at(a, u, pj);
          const int s = slot_seq % S;
          const uint32_t bar = tc05::smem_u32(&full[s]);
          tc05::mbar_expect_tx(bar, row_bytes);
          bulk_row(tc05::smem_u32(stage_base + (size_t)s * row_bytes), a.counters + (size_t)v * cells + (size_t)pr * W,
                   row_bytes, bar);
          if (++pr == d) {
            pr = 0;
            pj++;
          }
        };
        if (tid == 0)
          for (uint32_t t = 0; t < T && t < (uint32_t)S; t++) issue(seq + t);
        int j = 0, r = 0;
        for (uint32_t t = 0; t < T; t++) {
          if (r == 0)
            while (nb_at(a, u, j) < 0) j++;
          const uint32_t sq = seq + t;
          const int s = sq % S;
          tc05::mbar_wait(tc05::smem_u32(&full[s]), (sq / S) & 1u);
          const long long* row = reinterpret_cast<const long long*>(stage_base + (size_t)s * row_bytes);
          const uint32_t* cr = cols + r * a.ch;
#pragma unroll
          for (int k = 0; k < REC_KMAX; k++) {
            const int pos = tid + k * REC_THREADS;
            if (k < kk && pos < cn) {
              const long long x = row[cr[pos]];
              mn[k] = (r == 0 || x < mn[k]) ? x : mn[k];
            }
          }
          if (r == d - 1) {
            const double sim = clamp_sim(__ldg(a.nb_sim + u * a.ld + j));
#pragma unroll
            for (int k = 0; k < REC_KMAX; k++)
              if (k < kk && tid + k * REC_THREADS < cn) nb_term(mn[k], a.inv_q, sim, pref[k], tot[k], count[k]);
          }
          __syncthreads();  // every thread is done with stage s
          if (tid == 0 && t + S < T) issue(sq + S);
          if (++r == d) {
            r = 0;
            j++;
          }
        }
        seq += T;
      } else {
        for (int j = 0; j < cnt; j++) {
          const long long v = nb_at(a, u, j);
          if (v < 0) continue;
          const double sim = clamp_sim(__ldg(a.nb_sim + u * a.ld + j));
          const long long* sk = a.counters + (size_t)v * cells;
#pragma unroll
          for (int k = 0; k < REC_KMAX; k++) {
            const int pos = tid + k * REC_THREADS;
            if (k < kk && pos < cn) nb_term(gather_min(sk, cols + pos, a.ch, d, W), a.inv_q, sim, pref[k], tot[k], count[k]);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < REC_KMAX; k++) {
        const int pos = tid + k * REC_THREADS;
        if (k < kk && pos < cn) {
          const float e = nb_result(pref[k], tot[k], count[k]);
          vals[c0 + pos] = e;
          keys[c0 + pos] = rank_key(e, c0 + pos);
        }
      }
      __syncthreads();  // cols are rewritten by the next chunk
    }

    // ---- 3. top-N ------------------------------------------------------------------------------------------
    const int n_out = topn_keys<REC_THREADS>(keys, C, a.how_many, hist, scan_sh, bcast, sortbuf);
    for (int t = tid; t < n_out; t += REC_THREADS) {
      const int pos = (int)(0xFFFFFFFFu - (uint32_t)sortbuf[t]);
      out_item[t] = __ldg(a.item_ids + cand[pos]);
      out_value[t] = vals[pos];
    }
    if (tid == 0) a.out_cnt[i] = n_out;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// K_RECOMMEND, item-based: RecommenderJob's aggregate-and-recommend phase over the item top-k lists
// ---------------------------------------------------------------------------------------------------------------
constexpr int IB_THREADS = 128;
constexpr int IB_TABLE_LOG2 = 11;
constexpr int IB_TABLE = 1 << IB_TABLE_LOG2;  // open-addressing slots per CTA
constexpr int IB_TABLE_MAX = IB_TABLE / 2;    // users with more list entries than this take a dense slice
constexpr int IB_SORT_TILE = 2048;            // itemID rank sort: elements per shared-memory tile
constexpr size_t IB_SMEM = (size_t)IB_TABLE * (8 + 8 + 4 + 4) + REC_MAX_N * 8 + 8 * 8 + 32 * 8 + 256 * 4 + 32 * 4;
constexpr size_t IB_DENSE_MAX_BYTES = 4ull << 30;  // dense slices of one call, all CTAs together

enum { IP_SMEM = 0, IP_DENSE, IP_ENTRIES, IP_ENTRIES_MAX, IP_PRUNED, IP_CAND_MAX, IP_BAD, IP_NEXT, IP_WORDS };

struct IbArgs {
  const long long* sim_idx;
  const double* sim_val;
  const int* sim_cnt;
  long long num_items;
  int ld;
  const long long* user_ptr;
  const int* pref_row;
  const float* pref_val;
  long long num_users, nnz;
  const long long* item_ids;
  const int* rank_of;  // [num_items] row -> rank of its itemID among all itemIDs
  const int* row_at;   // [num_items] rank -> row
  const unsigned* allowed;
  const long long* users;
  long long m;
  int how_many, max_prefs, boolean_data;
  long long* out_item;
  float* out_value;
  int* out_cnt;
  // dense slices [slices][num_items] each; num / den / cnt are all zero between users
  double* d_num;
  double* d_den;
  int* d_cnt;
  int* d_touched;
  unsigned long long* d_key;
  int* d_lock;  // [slices]
  int slices;
  unsigned long long* plan;
};

template <int NT>
__device__ __forceinline__ long long block_sum(long long x, long long* sh) {
  for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = x;
  __syncthreads();
  long long t = 0;
  for (int w = 0; w < NT / 32; w++) t += sh[w];
  __syncthreads();
  return t;
}

__device__ __forceinline__ uint32_t ib_hash(int key) { return ((uint32_t)key * 0x9E3779B1u) >> (32 - IB_TABLE_LOG2); }

// slot of `key` in the table, inserted if absent (the table never fills: at most IB_TABLE_MAX keys)
__device__ __forceinline__ int ib_insert(int* tkey, int key) {
  uint32_t h = ib_hash(key);
  for (;;) {
    const int k = *(volatile int*)&tkey[h];
    if (k == key) return (int)h;
    if (k == -1) {
      const int old = atomicCAS(&tkey[h], -1, key);
      if (old == -1 || old == key) return (int)h;
    }
    h = (h + 1) & (IB_TABLE - 1);
  }
}

__device__ __forceinline__ int ib_find(const int* tkey, int key) {
  uint32_t h = ib_hash(key);
  for (;;) {
    const int k = tkey[h];
    if (k == key) return (int)h;
    if (k == -1) return -1;
    h = (h + 1) & (IB_TABLE - 1);
  }
}

// AggregateAndRecommendReducer's prediction of item row `row` as a ranking key: order-preserving float bits, then
// 2^32-1-rank(itemID), so that (value desc, itemID asc) is one descending order; 0 = no recommendation
__device__ __forceinline__ unsigned long long ib_key(const IbArgs& a, int row, double num, double den, int cnt) {
  float v;
  if (a.boolean_data) {
    v = __double2float_rn(num);
  } else {
    if (cnt < 2) return 0ull;  // "preference estimations must be based on at least 2 datapoints"
    v = __double2float_rn(num / den);
  }
  if (!(v > __int_as_float(1))) return 0ull;  // NaN, and TopItemsQueue's sentinel Float.MIN_VALUE
  if (a.allowed && !((__ldg(a.allowed + (row >> 5)) >> (row & 31)) & 1u)) return 0ull;
  return ((unsigned long long)(__float_as_uint(v) | 0x80000000u) << 32) |
         (unsigned long long)(0xFFFFFFFFu - (uint32_t)__ldg(a.rank_of + row));
}

__global__ void __launch_bounds__(IB_THREADS) k_itembased(const IbArgs a) {
  extern __shared__ __align__(16) unsigned char ib_smem[];
  double* tnum = reinterpret_cast<double*>(ib_smem);  // [IB_TABLE]; holds the keys after the accumulation
  double* tden = tnum + IB_TABLE;
  int* tkey = reinterpret_cast<int*>(tden + IB_TABLE);  // item row, -1 = empty
  int* tcnt = tkey + IB_TABLE;
  unsigned long long* sortbuf = reinterpret_cast<unsigned long long*>(tcnt + IB_TABLE);  // [REC_MAX_N]
  long long* bcast = reinterpret_cast<long long*>(sortbuf + REC_MAX_N);                   // [8]
  long long* red = bcast + 8;                                                              // [32]
  unsigned* hist = reinterpret_cast<unsigned*>(red + 32);                                  // [256]
  int* scan_sh = reinterpret_cast<int*>(hist + 256);                                       // [32]
  const int tid = threadIdx.x;
  for (int s = tid; s < IB_TABLE; s += IB_THREADS) {
    tkey[s] = -1;
    tnum[s] = 0.0;
    tden[s] = 0.0;
    tcnt[s] = 0;
  }
  __syncthreads();

  for (;;) {
    if (tid == 0) bcast[0] = (long long)atomicAdd(&a.plan[IP_NEXT], 1ull);
    __syncthreads();
    const long long i = bcast[0];
    __syncthreads();
    if (i >= a.m) break;
    long long* out_item = a.out_item + i * a.how_many;
    float* out_value = a.out_value + i * a.how_many;
    for (int t = tid; t < a.how_many; t += IB_THREADS) {
      out_item[t] = -1;
      out_value[t] = 0.0f;
    }

    // ---- (a) the user vector, checked before anything depends on it ----------------------------------------
    const long long u = a.users[i];
    long long lo = 0, hi = 0;
    bool bad_user = u < 0 || u >= a.num_users;
    if (!bad_user) {
      lo = a.user_ptr[u];
      hi = a.user_ptr[u + 1];
      bad_user = lo < 0 || hi < lo || hi > a.nnz;
    }
    long long bad = 0, nz = 0;
    if (!bad_user) {
      for (long long t = lo + tid; t < hi; t += IB_THREADS) {
        const int r = a.pref_row[t];
        bad += r < 0 || r >= a.num_items || (t > lo && a.pref_row[t - 1] >= r);
        nz += a.pref_val[t] != 0.0f;  // RandomAccessSparseVector.set(i, 0) stores nothing
      }
    }
    bad = block_sum<IB_THREADS>(bad, red);
    nz = block_sum<IB_THREADS>(nz, red);
    if (bad_user || bad) {
      if (tid == 0) {
        atomicAdd(&a.plan[IP_BAD], (unsigned long long)(bad_user ? 1 : bad));
        a.out_cnt[i] = 0;
      }
      continue;
    }
    // pruning (UserVectorSplitterMapper.maybePruneUserVector): T = the P-th largest |pref|, as float bits
    uint32_t T = 0;
    const bool pruned = nz > a.max_prefs;
    if (pruned) {
      uint32_t prefix = 0, mask = 0;
      unsigned want = (unsigned)a.max_prefs;
      for (int shift = 24; shift >= 0; shift -= 8) {
        for (int t = tid; t < 256; t += IB_THREADS) hist[t] = 0u;
        __syncthreads();
        for (long long t = lo + tid; t < hi; t += IB_THREADS) {
          const float p = a.pref_val[t];
          const uint32_t b = __float_as_uint(fabsf(p));
          if (p != 0.0f && (b & mask) == prefix) atomicAdd(&hist[(b >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid == 0) {
          unsigned acc = 0;
          for (int b = 255; b >= 0; b--) {
            if (acc + hist[b] >= want) {
              prefix |= (uint32_t)b << shift;
              want -= acc;
              break;
            }
            acc += hist[b];
          }
          bcast[1] = (long long)prefix;
          bcast[2] = (long long)want;
        }
        __syncthreads();
        prefix = (uint32_t)bcast[1];
        want = (unsigned)bcast[2];
        mask |= 255u << shift;
        __syncthreads();
      }
      T = prefix;
    }
    // considered: non-zero, and |pref| >= T (ties at T all kept; below it upstream sets the pref to NaN)
    auto considered = [&](float p) { return p != 0.0f && __float_as_uint(fabsf(p)) >= T; };

    // ---- (b) B = entries of the considered lists --------------------------------------------------------------
    long long B = 0;
    for (long long t = lo + tid; t < hi; t += IB_THREADS) {
      if (!considered(a.pref_val[t])) continue;
      const int c = a.sim_cnt[a.pref_row[t]];
      if (c < 0 || c > a.ld) bad++;
      else B += c;
    }
    bad = block_sum<IB_THREADS>(bad, red);
    B = block_sum<IB_THREADS>(B, red);
    if (bad) {
      if (tid == 0) {
        atomicAdd(&a.plan[IP_BAD], (unsigned long long)bad);
        a.out_cnt[i] = 0;
      }
      continue;
    }
    const bool dense = B > IB_TABLE_MAX;
    double *num = tnum, *den = tden;
    int* cnt = tcnt;
    int* touched = nullptr;
    unsigned long long* dkeys = nullptr;
    int slice = -1;
    if (dense) {
      if (tid == 0) {
        for (int s = 0;; s = s + 1 == a.slices ? 0 : s + 1)
          if (atomicCAS(&a.d_lock[s], 0, 1) == 0) {
            bcast[3] = s;
            break;
          }
        __threadfence();
        bcast[4] = 0;  // touched items
      }
      __syncthreads();
      slice = (int)bcast[3];
      const size_t off = (size_t)slice * a.num_items;
      num = a.d_num + off;
      den = a.d_den + off;
      cnt = a.d_cnt + off;
      touched = a.d_touched + off;
      dkeys = a.d_key + off;
    }

    // ---- (c) partial products: one pass per considered list in ascending item row, lanes split its entries ----
    for (long long t = lo; t < hi; t++) {
      const float p = a.pref_val[t];
      if (!considered(p)) continue;  // the same t on every thread: uniform
      const long long j = a.pref_row[t];
      const int c = a.sim_cnt[j];
      const double pd = (double)p;
      for (int e = tid; e < c; e += IB_THREADS) {
        const long long it = __ldg(a.sim_idx + j * a.ld + e);
        const double s = __ldg(a.sim_val + j * a.ld + e);
        if (it < 0 || it >= a.num_items) {
          bad++;
          continue;
        }
        int at;
        double n0, d0;
        if (dense) {
          // the counts are updated at L2 (atomics): dense slices are read past L1
          at = (int)it;
          if (atomicAdd(&cnt[at], 1) == 0) touched[atomicAdd(reinterpret_cast<unsigned long long*>(&bcast[4]), 1ull)] = at;
          n0 = __ldcg(num + at);
          d0 = __ldcg(den + at);
        } else {
          at = ib_insert(tkey, (int)it);
          cnt[at]++;
          n0 = num[at];
          d0 = den[at];
        }
        num[at] = a.boolean_data ? __dadd_rn(n0, s) : __dadd_rn(n0, __dmul_rn(s, pd));
        den[at] = __dadd_rn(d0, fabs(s));
      }
      __syncthreads();
    }
    // known items: upstream's NaN diagonal gives every considered item a NaN prediction
    for (long long t = lo + tid; t < hi; t += IB_THREADS) {
      if (!considered(a.pref_val[t])) continue;
      const int j = a.pref_row[t];
      const int at = dense ? (__ldcg(cnt + j) ? j : -1) : ib_find(tkey, j);
      if (at >= 0) num[at] = __longlong_as_double(0x7ff8000000000000ll);
    }
    __syncthreads();

    // ---- (d) ranking keys, top-N ------------------------------------------------------------------------------
    int C;
    unsigned long long* keys;
    long long cand = 0;
    if (dense) {
      C = (int)bcast[4];
      keys = dkeys;
      for (int t = tid; t < C; t += IB_THREADS) {
        const int it = touched[t];
        keys[t] = ib_key(a, it, __ldcg(num + it), __ldcg(den + it), __ldcg(cnt + it));
      }
      cand = C;
    } else {
      C = IB_TABLE;
      keys = reinterpret_cast<unsigned long long*>(tnum);  // in place: each slot read, then written, by one thread
      for (int s = tid; s < IB_TABLE; s += IB_THREADS) {
        const int it = tkey[s];
        keys[s] = it >= 0 ? ib_key(a, it, tnum[s], tden[s], tcnt[s]) : 0ull;
        cand += it >= 0;
      }
      cand = block_sum<IB_THREADS>(cand, red);
    }
    __syncthreads();
    const int n_out = topn_keys<IB_THREADS>(keys, C, a.how_many, hist, scan_sh, bcast, sortbuf);
    for (int t = tid; t < n_out; t += IB_THREADS) {
      const unsigned long long k = sortbuf[t];
      const int row = __ldg(a.row_at + (0xFFFFFFFFu - (uint32_t)k));
      out_item[t] = __ldg(a.item_ids + row);
      out_value[t] = __uint_as_float((uint32_t)(k >> 32) & 0x7FFFFFFFu);
    }
    bad = block_sum<IB_THREADS>(bad, red);
    if (tid == 0) {
      a.out_cnt[i] = n_out;
      if (bad) atomicAdd(&a.plan[IP_BAD], (unsigned long long)bad);
      atomicAdd(&a.plan[dense ? IP_DENSE : IP_SMEM], 1ull);
      atomicAdd(&a.plan[IP_ENTRIES], (unsigned long long)B);
      atomicMax(&a.plan[IP_ENTRIES_MAX], (unsigned long long)B);
      if (pruned) atomicAdd(&a.plan[IP_PRUNED], 1ull);
      atomicMax(&a.plan[IP_CAND_MAX], (unsigned long long)cand);
    }

    // ---- reset the accumulators for the next user -------------------------------------------------------------
    if (dense) {
      for (int t = tid; t < C; t += IB_THREADS) {
        const int it = touched[t];
        num[it] = 0.0;
        den[it] = 0.0;
        cnt[it] = 0;
      }
      __syncthreads();
      if (tid == 0) {
        __threadfence();
        atomicExch(&a.d_lock[slice], 0);
      }
    } else {
      for (int s = tid; s < IB_TABLE; s += IB_THREADS) {
        tkey[s] = -1;
        tnum[s] = 0.0;
        tden[s] = 0.0;
        tcnt[s] = 0;
      }
    }
    __syncthreads();
  }
}

// itemID rank table: (itemID, row) pairs sorted ascending by a bitonic sort; keys are itemID ^ 2^63 (signed order
// as unsigned), padding keys ~0.  One tile of IB_SORT_TILE elements per CTA: every size up to the tile (k_fixed = 0)
// or the strides below the tile of one size k_fixed.
__device__ __forceinline__ void rank_cmp(unsigned long long* key, int* row, long long t, long long j, long long k) {
  const long long p = t + j;
  const bool asc = (t & k) == 0;
  const unsigned long long x = key[t], y = key[p];
  if (asc ? x > y : x < y) {
    key[t] = y;
    key[p] = x;
    const int r = row[t];
    row[t] = row[p];
    row[p] = r;
  }
}

__global__ void __launch_bounds__(IB_SORT_TILE / 2) k_rank_tile(unsigned long long* key, int* row, long long npad,
                                                                 long long k_fixed) {
  __shared__ unsigned long long sk[IB_SORT_TILE];
  __shared__ int sr[IB_SORT_TILE];
  const long long tile = npad < IB_SORT_TILE ? npad : IB_SORT_TILE;
  const long long base = (long long)blockIdx.x * tile;
  for (long long t = threadIdx.x; t < tile; t += blockDim.x) {
    sk[t] = key[base + t];
    sr[t] = row[base + t];
  }
  __syncthreads();
  const long long k0 = k_fixed ? k_fixed : 2, k1 = k_fixed ? k_fixed : tile;
  for (long long k = k0; k <= k1; k <<= 1) {
    for (long long j = (k >> 1) < tile ? (k >> 1) : (tile >> 1); j > 0; j >>= 1) {
      for (long long c = threadIdx.x; c < tile / 2; c += blockDim.x) {
        const long long t = (c / j) * 2 * j + (c % j);
        // direction from the global position
        const long long p = t + j;
        const bool asc = ((base + t) & k) == 0;
        const unsigned long long x = sk[t], y = sk[p];
        if (asc ? x > y : x < y) {
          sk[t] = y;
          sk[p] = x;
          const int r = sr[t];
          sr[t] = sr[p];
          sr[p] = r;
        }
      }
      __syncthreads();
    }
  }
  for (long long t = threadIdx.x; t < tile; t += blockDim.x) {
    key[base + t] = sk[t];
    row[base + t] = sr[t];
  }
}

__global__ void k_rank_global(unsigned long long* key, int* row, long long npad, long long j, long long k) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= npad / 2) return;
  rank_cmp(key, row, (c / j) * 2 * j + (c % j), j, k);
}

__global__ void k_rank_init(const long long* __restrict__ item_ids, long long n, long long npad,
                            unsigned long long* key, int* row) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= npad) return;
  key[t] = t < n ? ((unsigned long long)item_ids[t] ^ 0x8000000000000000ull) : ~0ull;
  row[t] = t < n ? (int)t : -1;
}

__global__ void k_rank_scatter(const int* __restrict__ row_at, long long n, int* rank_of) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) rank_of[row_at[t]] = (int)t;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
extern "C" {

int mb200_bank_estimate_prefs(mb200_bank* bk, const int64_t* nb_idx, const double* nb_sim, const int32_t* nb_cnt,
                              int64_t nb_rows, int32_t nb_ld, const int64_t* user, const int64_t* nb_row,
                              const int64_t* item_id, int64_t q, float* out, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_estimate_prefs: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (q < 0 || nb_rows < 0 || nb_ld < 1 || (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_estimate_prefs: bad shape (q=%lld nb_rows=%lld nb_ld=%d)",
                      (long long)q, (long long)nb_rows, nb_ld);
  if (q == 0) return MB200_OK;
  if (!user || !item_id || !out || (nb_rows > 0 && (!nb_idx || !nb_sim || !nb_cnt)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_estimate_prefs: NULL array argument");
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
  StatusWords plan(ctx, PL_WORDS);
  MB_CHECK(plan.zero(WS_STATUS));
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_estimate_prefs<<<(unsigned)ceil_div64(q, EST_THREADS), EST_THREADS, (size_t)bk->d * EST_THREADS * 4, ctx->stream>>>(
        bk->counters, bk->hf, bk->E, ldexp(1.0, -bk->frac_bits), d_idx, d_sim, d_cnt, nb_rows, nb_ld, d_user, d_row,
        d_item, q, d_out, plan.dev);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[PL_WORDS];
  MB_CHECK(plan.read(h));
  if (h[PL_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_bank_estimate_prefs: %llu user row(s), neighbourhood row(s), counts or neighbour index(es) "
                      "out of range (entities %lld, neighbourhood rows %lld, nb_ld %d)",
                      h[PL_BAD], (long long)bk->E, (long long)nb_rows, nb_ld);
  return MB200_OK;
}

int mb200_bank_recommend(mb200_bank* bk, const int64_t* nb_idx, const double* nb_sim, const int32_t* nb_cnt,
                         int32_t nb_ld, const int64_t* item_ptr, const int32_t* item_col, int64_t nnz,
                         const int64_t* item_ids, int64_t num_items, const int64_t* users, int64_t m, int32_t how_many,
                         int include_known, int64_t* out_item, float* out_value, int32_t* out_cnt, int mem) {
  if (!bk) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_bank_recommend: bank is NULL");
  mb200_ctx* ctx = bk->ctx;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (how_many < 1 || how_many > REC_MAX_N)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_recommend: how_many must be in [1, %d] (got %d)", REC_MAX_N,
                      how_many);
  if (m < 0 || nb_ld < 1 || nnz < 0 || num_items < 0 || num_items >= (1LL << 31) ||
      (mem != MB200_MEM_HOST && mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_bank_recommend: bad shape (m=%lld nb_ld=%d nnz=%lld num_items=%lld)", (long long)m, nb_ld,
                      (long long)nnz, (long long)num_items);
  if (m == 0) return MB200_OK;
  if (!nb_idx || !nb_sim || !nb_cnt || !item_ptr || (nnz > 0 && !item_col) || (num_items > 0 && !item_ids) || !users ||
      !out_item || !out_value || !out_cnt)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_recommend: NULL array argument");
  if (mem == MB200_MEM_HOST) {
    // the data model is host memory: its shape can be checked here
    if (item_ptr[0] != 0 || item_ptr[bk->E] != nnz)
      return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_recommend: item_ptr[0] must be 0 and item_ptr[E] = nnz (%lld)",
                        (long long)nnz);
    for (int64_t t = 1; t < num_items; t++)
      if (item_ids[t] <= item_ids[t - 1])
        return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_bank_recommend: item_ids must be strictly ascending");
  }
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const int d = bk->d;
  const long long W = bk->W;
  const long long words = (num_items + 31) / 32;
  const bool bitmap_smem = words <= REC_BITMAP_SMEM_WORDS;
  int ch = REC_COLS_BYTES / (4 * d);
  ch = ch > REC_KMAX * REC_THREADS ? REC_KMAX * REC_THREADS : ch;
  ch = (ch / REC_THREADS) * REC_THREADS;
  const size_t fixed = 8 * 4 + 8 * 8 + REC_MAX_N * 8 + (size_t)d * ch * 4 + 256 * 4 + 32 * 4 +
                       (bitmap_smem ? (size_t)words * 4 : 0);
  const size_t row_bytes = (size_t)W * 8;
  int stages = 0;
  if ((W & 1) == 0 && ctx->smem_optin > fixed) {
    const size_t s = (ctx->smem_optin - fixed) / row_bytes;
    stages = s >= 2 ? (s > 4 ? 4 : (int)s) : 0;
  }
  const size_t smem = fixed + (size_t)stages * row_bytes;
  const int grid = (int)(m < ctx->num_sms ? m : ctx->num_sms);

  ArgStage st(ctx, mem);
  RecArgs a;
  a.counters = bk->counters;
  a.hf = bk->hf;
  a.E = bk->E;
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
  a.ch = ch;
  const size_t nbc = (size_t)bk->E * nb_ld;
  MB_CHECK(st.in((const long long*)nb_idx, nbc, &a.nb_idx));
  MB_CHECK(st.in(nb_sim, nbc, &a.nb_sim));
  MB_CHECK(st.in((const int*)nb_cnt, (size_t)bk->E, &a.nb_cnt));
  MB_CHECK(st.in((const long long*)item_ptr, (size_t)bk->E + 1, &a.item_ptr));
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
  a.ws_bitmap = (unsigned*)wb;
  a.ws_cand = (int*)wc;
  a.ws_key = (unsigned long long*)wk;
  a.ws_val = (float*)wv;
  StatusWords plan(ctx, PL_WORDS);
  MB_CHECK(plan.zero(WS_STATUS));
  a.plan = plan.dev;
  MB_CUDA(ctx, cudaFuncSetAttribute(k_recommend, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_recommend<<<grid, REC_THREADS, smem, ctx->stream>>>(a);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[PL_WORDS];
  MB_CHECK(plan.read(h));
  mb200_recommend_plan& pl = ctx->last_recommend_plan;
  pl.stream_users = (int64_t)h[PL_STREAM];
  pl.gather_users = (int64_t)h[PL_GATHER];
  pl.chunks = (int64_t)h[PL_CHUNKS];
  pl.candidates = (int64_t)h[PL_CAND_SUM];
  pl.candidates_max = (int64_t)h[PL_CAND_MAX];
  pl.stream_rows = (int64_t)h[PL_STREAM_ROWS];
  pl.gather_loads = (int64_t)h[PL_GATHER_LOADS];
  pl.stages = stages;
  pl.chunk_candidates = ch;
  if (getenv("MB200_TRACE"))
    fprintf(stderr,
            "[mb200 trace] recommend plan: users=%lld stream=%lld gather=%lld chunks=%lld stages=%d chunk=%d "
            "candidates=%lld max=%lld W=%lld d=%d\n",
            (long long)m, (long long)pl.stream_users, (long long)pl.gather_users, (long long)pl.chunks, stages, ch,
            (long long)pl.candidates, (long long)pl.candidates_max, W, d);
  if (h[PL_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_bank_recommend: %llu user row(s), neighbour count(s) or index(es), item_ptr range(s) or "
                      "item_col entr(ies) out of range (entities %lld, num_items %lld, nnz %lld)",
                      h[PL_BAD], (long long)bk->E, (long long)num_items, (long long)nnz);
  return MB200_OK;
}

int mb200_recommend_last_plan(mb200_ctx* ctx, mb200_recommend_plan* out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_recommend_last_plan: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  *out = ctx->last_recommend_plan;
  return MB200_OK;
}

}  // extern "C"

int mb200_itembased_call(mb200_ctx* ctx, const mb200_itembased_args* args, bool data_on_device) {
  if (!ctx || !args) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_recommend_item_based: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  const mb200_itembased_args& x = *args;
  if (x.how_many < 1 || x.how_many > REC_MAX_N)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_recommend_item_based: how_many must be in [1, %d] (got %d)",
                      REC_MAX_N, x.how_many);
  if (x.max_prefs_per_user < 1)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_recommend_item_based: max_prefs_per_user must be >= 1 (got %d)",
                      x.max_prefs_per_user);
  if (x.m < 0 || x.sim_ld < 1 || x.num_items < 0 || x.num_items >= (1LL << 31) || x.num_users < 0 || x.nnz < 0 ||
      (x.mem != MB200_MEM_HOST && x.mem != MB200_MEM_DEVICE))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_recommend_item_based: bad shape (m=%lld sim_ld=%d num_items=%lld num_users=%lld nnz=%lld)",
                      (long long)x.m, x.sim_ld, (long long)x.num_items, (long long)x.num_users, (long long)x.nnz);
  if (x.m == 0) return MB200_OK;
  if (!x.user_ptr || !x.users || !x.out_item || !x.out_value || !x.out_cnt ||
      (x.num_items > 0 && (!x.sim_idx || !x.sim_val || !x.sim_cnt || !x.item_ids)) ||
      (x.nnz > 0 && (!x.pref_row || !x.pref_val)))
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_recommend_item_based: NULL array argument");
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long n = x.num_items;
  const long long words = (n + 31) / 32;

  ArgStage st(ctx, x.mem);
  IbArgs a;
  a.num_items = n;
  a.ld = x.sim_ld;
  a.num_users = x.num_users;
  a.nnz = x.nnz;
  a.m = x.m;
  a.how_many = x.how_many;
  a.max_prefs = x.max_prefs_per_user;
  a.boolean_data = x.boolean_data != 0;
  const size_t lists = (size_t)n * x.sim_ld;
  // the lists, the user CSR and the itemIDs: staged with the rest, or already on the device
  ArgStage data(ctx, data_on_device ? MB200_MEM_DEVICE : x.mem);
  ArgStage& dst = data_on_device ? data : st;
  MB_CHECK(dst.in((const long long*)x.sim_idx, lists, &a.sim_idx));
  MB_CHECK(dst.in(x.sim_val, lists, &a.sim_val));
  MB_CHECK(dst.in((const int*)x.sim_cnt, (size_t)n, &a.sim_cnt));
  MB_CHECK(dst.in((const long long*)x.user_ptr, (size_t)x.num_users + 1, &a.user_ptr));
  MB_CHECK(dst.in((const int*)x.pref_row, (size_t)x.nnz, &a.pref_row));
  MB_CHECK(dst.in(x.pref_val, (size_t)x.nnz, &a.pref_val));
  MB_CHECK(dst.in((const long long*)x.item_ids, (size_t)n, &a.item_ids));
  MB_CHECK(st.in((const unsigned*)x.allowed, x.allowed ? (size_t)words : 0, &a.allowed));
  MB_CHECK(st.in((const long long*)x.users, (size_t)x.m, &a.users));
  MB_CHECK(st.out((long long*)x.out_item, (size_t)x.m * x.how_many, &a.out_item));
  MB_CHECK(st.out(x.out_value, (size_t)x.m * x.how_many, &a.out_value));
  MB_CHECK(st.out((int*)x.out_cnt, (size_t)x.m, &a.out_cnt));

  // the itemID rank table: (itemID, row) sorted on the device, rank -> row and row -> rank
  long long npad = 1;
  while (npad < n) npad <<= 1;
  void *wk = nullptr, *wr = nullptr, *wo = nullptr;
  MB_CHECK(ws_slot(ctx, WS_IB_RANK_KEY, (size_t)npad * 8, &wk));
  MB_CHECK(ws_slot(ctx, WS_IB_RANK_ROW, (size_t)npad * 4, &wr));
  MB_CHECK(ws_slot(ctx, WS_IB_RANK_OF, (size_t)(n > 0 ? n : 1) * 4, &wo));
  StatusWords plan(ctx, IP_WORDS);
  MB_CHECK(plan.zero(WS_STATUS));
  a.row_at = (const int*)wr;
  a.rank_of = (const int*)wo;
  a.plan = plan.dev;
  if (n > 0) {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    unsigned long long* key = (unsigned long long*)wk;
    int* row = (int*)wr;
    k_rank_init<<<(unsigned)ceil_div64(npad, 256), 256, 0, ctx->stream>>>(a.item_ids, n, npad, key, row);
    const long long tile = npad < IB_SORT_TILE ? npad : IB_SORT_TILE;
    k_rank_tile<<<(unsigned)(npad / tile), IB_SORT_TILE / 2, 0, ctx->stream>>>(key, row, npad, 0);
    ctx->launches += 2;
    for (long long k = 2 * IB_SORT_TILE; k <= npad; k <<= 1) {
      for (long long j = k >> 1; j >= IB_SORT_TILE; j >>= 1) {
        k_rank_global<<<(unsigned)ceil_div64(npad / 2, 256), 256, 0, ctx->stream>>>(key, row, npad, j, k);
        ctx->launches++;
      }
      k_rank_tile<<<(unsigned)(npad / IB_SORT_TILE), IB_SORT_TILE / 2, 0, ctx->stream>>>(key, row, npad, k);
      ctx->launches++;
    }
    k_rank_scatter<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(row, n, (int*)wo);
    ctx->launches++;
    MB_CUDA(ctx, cudaGetLastError());
  }

  // persistent CTAs, as many as fit; dense slices for as many of them as 4 GiB allow
  MB_CUDA(ctx, cudaFuncSetAttribute(k_itembased, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IB_SMEM));
  int per_sm = 0;
  MB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_itembased, IB_THREADS, IB_SMEM));
  per_sm = per_sm < 1 ? 1 : per_sm;
  const long long grid = x.m < (long long)ctx->num_sms * per_sm ? x.m : (long long)ctx->num_sms * per_sm;
  const size_t slice_bytes = (size_t)(n > 0 ? n : 1) * (8 + 8 + 4 + 4 + 8);
  long long slices = (long long)(IB_DENSE_MAX_BYTES / slice_bytes);
  slices = slices < 1 ? 1 : (slices > grid ? grid : slices);
  // num / den / cnt of the slices are kept zero by the kernel, so they are cleared only when the slot is (re)allocated
  // or its layout changes
  const size_t dense_bytes = (size_t)slices * slice_bytes;
  void *wd = nullptr, *wl = nullptr;
  bool fresh = false;
  MB_CHECK(ws_slot(ctx, WS_IB_DENSE, dense_bytes, &wd, &fresh));
  if (fresh || ctx->itembased_dense_items != n || ctx->itembased_dense_slices != slices) {
    MB_CUDA(ctx, cudaMemsetAsync(wd, 0, dense_bytes, ctx->stream));
    ctx->itembased_dense_items = n;
    ctx->itembased_dense_slices = slices;
  }
  MB_CHECK(ws_slot(ctx, WS_IB_LOCKS, (size_t)slices * 4, &wl));
  MB_CUDA(ctx, cudaMemsetAsync(wl, 0, (size_t)slices * 4, ctx->stream));
  const size_t per = (size_t)slices * (n > 0 ? n : 1);
  a.d_num = (double*)wd;
  a.d_den = a.d_num + per;
  a.d_key = (unsigned long long*)(a.d_den + per);
  a.d_cnt = (int*)(a.d_key + per);
  a.d_touched = a.d_cnt + per;
  a.d_lock = (int*)wl;
  a.slices = (int)slices;
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_itembased<<<(unsigned)grid, IB_THREADS, IB_SMEM, ctx->stream>>>(a);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[IP_WORDS];
  MB_CHECK(plan.read(h));
  mb200_itembased_plan& pl = ctx->last_itembased_plan;
  pl.users = x.m;
  pl.smem_users = (int64_t)h[IP_SMEM];
  pl.dense_users = (int64_t)h[IP_DENSE];
  pl.entries = (int64_t)h[IP_ENTRIES];
  pl.entries_max = (int64_t)h[IP_ENTRIES_MAX];
  pl.pruned_users = (int64_t)h[IP_PRUNED];
  pl.candidates_max = (int64_t)h[IP_CAND_MAX];
  pl.table_slots = IB_TABLE;
  pl.dense_slices = (int32_t)slices;
  if (getenv("MB200_TRACE"))
    fprintf(stderr,
            "[mb200 trace] itembased plan: users=%lld smem=%lld dense=%lld entries=%lld entries_max=%lld pruned=%lld "
            "candidates_max=%lld table=%d slices=%lld grid=%lld\n",
            (long long)pl.users, (long long)pl.smem_users, (long long)pl.dense_users, (long long)pl.entries,
            (long long)pl.entries_max, (long long)pl.pruned_users, (long long)pl.candidates_max, IB_TABLE, slices, grid);
  if (h[IP_BAD])
    return mb200_fail(ctx, MB200_ERR_BAD_ARG,
                      "mb200_recommend_item_based: %llu user row(s), user_ptr range(s), pref_row entr(ies) (out of range "
                      "or not ascending), list count(s) or list entr(ies) out of range (num_users %lld, num_items %lld, "
                      "nnz %lld, sim_ld %d)",
                      h[IP_BAD], (long long)x.num_users, (long long)n, (long long)x.nnz, x.sim_ld);
  return MB200_OK;
}

extern "C" {

int mb200_recommend_item_based(mb200_ctx* ctx, const mb200_itembased_args* args) {
  return mb200_itembased_call(ctx, args, false);
}

int mb200_itembased_last_plan(mb200_ctx* ctx, mb200_itembased_plan* out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_itembased_last_plan: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  *out = ctx->last_itembased_plan;
  return MB200_OK;
}

}  // extern "C"
