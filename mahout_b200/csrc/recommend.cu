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
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc05.cuh"

namespace {

constexpr int REC_THREADS = 512;
constexpr int REC_KMAX = 8;                  // candidates per thread and chunk
constexpr int REC_MAX_N = 1024;              // largest how_many
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

__device__ __forceinline__ double clamp_sim(double s) {
  // AbstractSimilarity.normalizeWeightResult: clamp to [-1, 1], NaN stays NaN
  return s != s ? s : (s < -1.0 ? -1.0 : (s > 1.0 ? 1.0 : s));
}

// one neighbour's term of doEstimatePreference, FP64 with the product and the sum rounded separately (Java does not
// fuse them)
__device__ __forceinline__ void nb_term(long long mn, double inv_q, double s, double& pref, double& tot, int& count) {
  const float p = __double2float_rn((double)mn * inv_q);
  if (p != 0.0f && s == s) {
    pref = __dadd_rn(pref, __dmul_rn(s, (double)p));
    tot = __dadd_rn(tot, s);
    count++;
  }
}

__device__ __forceinline__ float nb_result(double pref, double tot, int count) {
  return count <= 1 ? __int_as_float(0x7fc00000) : __double2float_rn(pref / tot);
}

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
__device__ __forceinline__ void bulk_row(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// the listed neighbour slot j of user u: its row, or -1 when it is skipped (the user itself, or out of range)
__device__ __forceinline__ long long nb_at(const RecArgs& a, long long u, int j) {
  const long long v = __ldg(a.nb_idx + u * a.ld + j);
  return (v == u || v < 0 || v >= a.E) ? -1 : v;
}

// block-wide exclusive scan of one int per thread (REC_THREADS); returns the total through *total
__device__ __forceinline__ int block_exscan(int x, int* sh, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = x;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) sh[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = lane < REC_THREADS / 32 ? sh[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < REC_THREADS / 32) sh[lane] = w;  // inclusive per warp
  }
  __syncthreads();
  const int before = (warp ? sh[warp - 1] : 0) + inc - x;
  *total = sh[REC_THREADS / 32 - 1];
  __syncthreads();
  return before;
}

// order-preserving key: (value desc, position asc) == key desc; 0 = no estimate
__device__ __forceinline__ unsigned long long rank_key(float v, int pos) {
  if (v != v) return 0ull;
  uint32_t b = __float_as_uint(v == 0.0f ? 0.0f : v);  // -0.0 ranks as 0.0
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)b << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)pos);
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
    int at = block_exscan(mine, scan_sh, &C);
    for (int w = w0; w < w1; w++) {
      unsigned b = bitmap[w];
      while (b) {
        const int k = __ffs(b) - 1;
        b &= b - 1;
        cand[at++] = w * 32 + k;
      }
    }
    int tot_bad = 0, tot_c = 0;
    block_exscan(bad, scan_sh, &tot_bad);
    block_exscan(c_eff, scan_sh, &tot_c);
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
    int valid = 0, nvalid = 0;
    for (int pos = tid; pos < C; pos += REC_THREADS) valid += keys[pos] != 0ull;
    block_exscan(valid, scan_sh, &nvalid);
    unsigned long long thr = 1ull;  // keys >= thr are kept
    if (nvalid > a.how_many) {
      unsigned long long prefix = 0ull, mask = 0ull;
      unsigned want = (unsigned)a.how_many;
      for (int shift = 56; shift >= 0; shift -= 8) {
        if (tid < 256) hist[tid] = 0u;
        __syncthreads();
        for (int pos = tid; pos < C; pos += REC_THREADS) {
          const unsigned long long k = keys[pos];
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
          bcast[1] = (long long)prefix;
          bcast[2] = (long long)want;
        }
        __syncthreads();
        prefix = (unsigned long long)bcast[1];
        want = (unsigned)bcast[2];
        mask |= 255ull << shift;
        __syncthreads();
      }
      thr = prefix;  // keys are distinct: exactly how_many keys are >= the how_many-th largest
    }
    const int n_out = nvalid < a.how_many ? nvalid : a.how_many;
    int npad = 1;
    while (npad < n_out) npad <<= 1;
    for (int t = tid; t < npad; t += REC_THREADS) sortbuf[t] = 0ull;
    if (tid == 0) bcast[3] = 0;
    __syncthreads();
    for (int pos = tid; pos < C; pos += REC_THREADS) {
      const unsigned long long k = keys[pos];
      if (k && k >= thr) sortbuf[atomicAdd(reinterpret_cast<unsigned long long*>(&bcast[3]), 1ull)] = k;
    }
    __syncthreads();
    // bitonic sort, descending
    for (int size = 2; size <= npad; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = tid; t < npad; t += REC_THREADS) {
          const int partner = t ^ stride;
          if (partner > t) {
            const bool desc = (t & size) == 0;
            const unsigned long long x = sortbuf[t], y = sortbuf[partner];
            if (desc ? (x < y) : (x > y)) {
              sortbuf[t] = y;
              sortbuf[partner] = x;
            }
          }
        }
        __syncthreads();
      }
    }
    for (int t = tid; t < n_out; t += REC_THREADS) {
      const int pos = (int)(0xFFFFFFFFu - (uint32_t)sortbuf[t]);
      out_item[t] = __ldg(a.item_ids + cand[pos]);
      out_value[t] = vals[pos];
    }
    if (tid == 0) a.out_cnt[i] = n_out;
    __syncthreads();
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// host-memory arguments are staged through grow-only slots of the context (mb200_group_ws; slots 40.. are this file's)
namespace {
struct Staged {
  mb200_ctx* ctx;
  int mem;
  int next_slot = 40;
  std::vector<std::pair<void*, std::pair<void*, size_t>>> outs;  // (device, (user, bytes))
  Staged(mb200_ctx* c, int m) : ctx(c), mem(m) {}
  template <typename T>
  int in(const T* user, size_t n, const T** dev) {
    if (mem == MB200_MEM_DEVICE || !user) {
      *dev = user;
      next_slot++;
      return MB200_OK;
    }
    void* p = nullptr;
    MB_CHECK(mb200_group_ws(ctx, next_slot++, n * sizeof(T), &p));
    if (n) MB_CUDA(ctx, cudaMemcpyAsync(p, user, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    ctx->stat_h2d += (int64_t)(n * sizeof(T));
    *dev = (const T*)p;
    return MB200_OK;
  }
  template <typename T>
  int out(T* user, size_t n, T** dev) {
    if (mem == MB200_MEM_DEVICE) {
      *dev = user;
      next_slot++;
      return MB200_OK;
    }
    void* p = nullptr;
    MB_CHECK(mb200_group_ws(ctx, next_slot++, n * sizeof(T), &p));
    outs.push_back({p, {(void*)user, n * sizeof(T)}});
    *dev = (T*)p;
    return MB200_OK;
  }
  int finish() {
    for (auto& o : outs) {
      if (o.second.second)
        MB_CUDA(ctx, cudaMemcpyAsync(o.second.first, o.first, o.second.second, cudaMemcpyDeviceToHost, ctx->stream));
      ctx->stat_d2h += (int64_t)o.second.second;
    }
    MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return MB200_OK;
  }
};

// the plan / error words live in a slot of their own; read back after the launch
int plan_words(mb200_ctx* ctx, unsigned long long** plan) {
  void* p = nullptr;
  MB_CHECK(mb200_group_ws(ctx, 39, PL_WORDS * sizeof(unsigned long long), &p));
  MB_CUDA(ctx, cudaMemsetAsync(p, 0, PL_WORDS * sizeof(unsigned long long), ctx->stream));
  *plan = (unsigned long long*)p;
  return MB200_OK;
}

int read_plan(mb200_ctx* ctx, const unsigned long long* plan, unsigned long long* h) {
  MB_CUDA(ctx, cudaMemcpyAsync(h, plan, PL_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MB200_OK;
}
}  // namespace

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
  Staged st(ctx, mem);
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
  unsigned long long* plan = nullptr;
  MB_CHECK(plan_words(ctx, &plan));
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_estimate_prefs<<<(unsigned)ceil_div64(q, EST_THREADS), EST_THREADS, (size_t)bk->d * EST_THREADS * 4, ctx->stream>>>(
        bk->counters, bk->hf, bk->E, ldexp(1.0, -bk->frac_bits), d_idx, d_sim, d_cnt, nb_rows, nb_ld, d_user, d_row,
        d_item, q, d_out, plan);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[PL_WORDS];
  MB_CHECK(read_plan(ctx, plan, h));
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

  Staged st(ctx, mem);
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
  MB_CHECK(mb200_group_ws(ctx, 36, bitmap_smem ? 4 : (size_t)grid * words * 4, &wb));
  MB_CHECK(mb200_group_ws(ctx, 37, (size_t)grid * per * 4, &wc));
  MB_CHECK(mb200_group_ws(ctx, 38, (size_t)grid * per * 8, &wk));
  MB_CHECK(mb200_group_ws(ctx, 35, (size_t)grid * per * 4, &wv));
  a.ws_bitmap = (unsigned*)wb;
  a.ws_cand = (int*)wc;
  a.ws_key = (unsigned long long*)wk;
  a.ws_val = (float*)wv;
  MB_CHECK(plan_words(ctx, &a.plan));
  MB_CUDA(ctx, cudaFuncSetAttribute(k_recommend, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  {
    ProfScope prof(ctx, MB200_K_RECOMMEND);
    k_recommend<<<grid, REC_THREADS, smem, ctx->stream>>>(a);
  }
  ctx->launches++;
  MB_CUDA(ctx, cudaGetLastError());
  MB_CHECK(st.finish());
  unsigned long long h[PL_WORDS];
  MB_CHECK(read_plan(ctx, a.plan, h));
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
