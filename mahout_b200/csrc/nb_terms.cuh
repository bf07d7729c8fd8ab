// nb_terms.cuh -- the per-neighbour arithmetic of GenericUserBasedRecommender.doEstimatePreference
// (GenericUserBasedRecommender.java:134-184), shared by the estimate kernels of recommend.cu (one sketch shape) and
// cmsized.cu (per-user sketch shapes).
#pragma once
#include <cuda_runtime.h>

static __device__ __forceinline__ double clamp_sim(double s) {
  // AbstractSimilarity.normalizeWeightResult: clamp to [-1, 1], NaN stays NaN
  return s != s ? s : (s < -1.0 ? -1.0 : (s > 1.0 ? 1.0 : s));
}

// one neighbour's term of doEstimatePreference, FP64 with the product and the sum rounded separately (Java does not
// fuse them)
static __device__ __forceinline__ void nb_term(long long mn, double inv_q, double s, double& pref, double& tot,
                                               int& count) {
  const float p = __double2float_rn((double)mn * inv_q);
  if (p != 0.0f && s == s) {
    pref = __dadd_rn(pref, __dmul_rn(s, (double)p));
    tot = __dadd_rn(tot, s);
    count++;
  }
}

static __device__ __forceinline__ float nb_result(double pref, double tot, int count) {
  return count <= 1 ? __int_as_float(0x7fc00000) : __double2float_rn(pref / tot);
}
