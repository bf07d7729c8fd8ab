// rec_topn.cuh -- the block scan, the ranking keys, the top-N and the bulk row copy of the recommendation kernels,
// shared by recommend.cu (k_recommend, k_itembased) and cmsized.cu (k_sized_recommend, k_sized_select).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

constexpr int REC_MAX_N = 1024;  // largest how_many

static __device__ __forceinline__ void bulk_row(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

// block-wide exclusive scan of one int per thread (NT threads); returns the total through *total
template <int NT>
static __device__ __forceinline__ int block_exscan(int x, int* sh, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = x;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) sh[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = lane < NT / 32 ? sh[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < NT / 32) sh[lane] = w;  // inclusive per warp
  }
  __syncthreads();
  const int before = (warp ? sh[warp - 1] : 0) + inc - x;
  *total = sh[NT / 32 - 1];
  __syncthreads();
  return before;
}

// order-preserving key: (value desc, position asc) == key desc; 0 = no estimate.  -inf ranks below every finite
// value and +inf above, like any other float.
static __device__ __forceinline__ unsigned long long rank_key(float v, int pos) {
  if (v != v) return 0ull;
  uint32_t b = __float_as_uint(v == 0.0f ? 0.0f : v);  // -0.0 ranks as 0.0
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)b << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)pos);
}

// top-N of C 64-bit keys (0 = none; the others distinct): the keys >= the how_many-th largest, sorted descending into
// sortbuf[0, n_out) (REC_MAX_N entries); returns n_out.  A radix select (8 passes of 8 bits) finds the how_many-th
// key, a bitonic sort in shared memory orders the survivors.  Uses bcast[1..3].
template <int NT>
static __device__ int topn_keys(const unsigned long long* keys, int C, int how_many, unsigned* hist, int* scan_sh,
                                long long* bcast, unsigned long long* sortbuf) {
  const int tid = threadIdx.x;
  int valid = 0, nvalid = 0;
  for (int pos = tid; pos < C; pos += NT) valid += keys[pos] != 0ull;
  block_exscan<NT>(valid, scan_sh, &nvalid);
  unsigned long long thr = 1ull;  // keys >= thr are kept
  if (nvalid > how_many) {
    unsigned long long prefix = 0ull, mask = 0ull;
    unsigned want = (unsigned)how_many;
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int t = tid; t < 256; t += NT) hist[t] = 0u;
      __syncthreads();
      for (int pos = tid; pos < C; pos += NT) {
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
  const int n_out = nvalid < how_many ? nvalid : how_many;
  int npad = 1;
  while (npad < n_out) npad <<= 1;
  for (int t = tid; t < npad; t += NT) sortbuf[t] = 0ull;
  if (tid == 0) bcast[3] = 0;
  __syncthreads();
  for (int pos = tid; pos < C; pos += NT) {
    const unsigned long long k = keys[pos];
    if (k && k >= thr) {
      const unsigned long long at = atomicAdd(reinterpret_cast<unsigned long long*>(&bcast[3]), 1ull);
      if (at < (unsigned long long)npad) sortbuf[at] = k;
    }
  }
  __syncthreads();
  // bitonic sort, descending
  for (int size = 2; size <= npad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < npad; t += NT) {
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
  return n_out;
}
