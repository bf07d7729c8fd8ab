// k1_dev.cuh -- device helpers shared by the K1 kernels (sketch.cu: direct scatter; group.cu: grouped
// shared-memory-tile update): increment -> fixed-point quanta, the d scattered RMWs of one event
// (DoubleCountMinSketch.update, DoubleCountMinSketch.java:72-80), status-word publication.
#pragma once
#include <math.h>

#include "common.cuh"

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
// T: increment type (float / double preference values, or uint8_t quanta of the narrow wire format);
// K: key / entity type (long long, or uint32_t in the narrow wire format)
template <typename T, typename K = long long>
struct UpdateArgs {
  long long* counters;
  const K* entity;  // may be null
  const K* key;
  const T* inc;
  long long n;
  long long E;
  double qscale;  // 2^frac_bits
  unsigned long long* flags;
  HashFamily hf;
};

template <typename T>
__device__ __forceinline__ long long inc_to_quanta(T inc, double qscale, unsigned int& bad,
                                                   unsigned long long& maxabs) {
  double qd = (double)inc * qscale;
  long long q = __double2ll_rn(qd);
  bool ok = ((double)q == qd) && (fabs(qd) < 4.0e18);
  if (!ok) {
    bad++;
    q = 0;
  }
  unsigned long long aq = q < 0 ? (unsigned long long)(-q) : (unsigned long long)q;
  maxabs = aq > maxabs ? aq : maxabs;
  return q;
}

// narrow wire format: the byte IS the number of quanta -- nothing to round, nothing to reject
__device__ __forceinline__ long long inc_to_quanta(unsigned char inc, double, unsigned int&, unsigned long long& maxabs) {
  maxabs = (unsigned long long)inc > maxabs ? (unsigned long long)inc : maxabs;
  return (long long)inc;
}

// the d scattered RMWs of one event: RED.ADD.64 into HBM/L2-resident counter rows
template <int D>
__device__ __forceinline__ void scatter_event(long long* __restrict__ sketch, const HashFamily& hf,
                                              long long key, long long q) {
  const uint64_t kr = cmh_residue(key);
  if (D > 0) {
#pragma unroll
    for (int i = 0; i < D; i++) {
      uint32_t col = cmh_column(hf.a[i], hf.b[i], kr, hf.w, hf.wmask);
      atomicAdd(reinterpret_cast<unsigned long long*>(sketch + (size_t)i * hf.w + col),
                (unsigned long long)q);
    }
  } else {
#pragma unroll 1
    for (int i = 0; i < hf.d; i++) {
      uint32_t col = cmh_column(hf.a[i], hf.b[i], kr, hf.w, hf.wmask);
      atomicAdd(reinterpret_cast<unsigned long long*>(sketch + (size_t)i * hf.w + col),
                (unsigned long long)q);
    }
  }
}

__device__ __forceinline__ void publish_flags(unsigned long long* flags, unsigned int bad,
                                              unsigned int bad_entity, unsigned long long maxabs) {
  bad = __reduce_add_sync(0xffffffffu, bad);
  bad_entity = __reduce_add_sync(0xffffffffu, bad_entity);
  unsigned int mhi = __reduce_max_sync(0xffffffffu, (unsigned int)(maxabs >> 32));
  unsigned int mlo = __reduce_max_sync(0xffffffffu, (unsigned int)(maxabs >> 32) == mhi
                                                       ? (unsigned int)maxabs : 0u);
  if ((threadIdx.x & 31) == 0) {
    if (bad) atomicAdd(&flags[FLAG_INEXACT], (unsigned long long)bad);
    if (bad_entity) atomicAdd(&flags[FLAG_BAD_ENTITY], (unsigned long long)bad_entity);
    unsigned long long m = ((unsigned long long)mhi << 32) | mlo;
    if (m) atomicMax(&flags[FLAG_MAXABS], m);
  }
}

