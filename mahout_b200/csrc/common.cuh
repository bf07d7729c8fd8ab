// common.cuh -- context / bank structures and error plumbing shared by the .cu files.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/mahout_b200.h"
#include "cm_hash.cuh"

struct HashFamily {
  uint64_t a[MB200_MAX_DEPTH];  // residues mod p
  uint64_t b[MB200_MAX_DEPTH];
  uint32_t w;
  uint32_t wmask;  // w-1 when w is a power of two, else 0
  int32_t d;
};

// device-side status words (one set per bank)
enum { FLAG_INEXACT = 0, FLAG_MAXABS = 1, FLAG_BAD_ENTITY = 2, FLAG_RANGE = 3,
       FLAG_MIXED = 4,  // K2 saw a negative counter or a row norm >= 2^36 quanta (see mb200_bank_sign_info)
       FLAG_WORDS = 5 };

struct ProfSpan {
  int kernel_id;
  cudaEvent_t beg, end;
};

struct mb200_ctx {
  int device = 0;
  int num_sms = 0;
  size_t smem_optin = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t stream = nullptr;  // stream in use (own_stream or the caller's)
  std::mutex mu;
  std::string err;
  int64_t launches = 0;
  bool profiling = false;
  std::vector<ProfSpan> spans;
  std::vector<cudaEvent_t> event_pool;
  double prof_ms[MB200_K_COUNT] = {};
  int64_t prof_n[MB200_K_COUNT] = {};
  // host-path staging (device) buffers, grown on demand
  void* stage[2] = {nullptr, nullptr};
  size_t stage_bytes = 0;
  cudaEvent_t stage_free[2] = {nullptr, nullptr};
  cudaEvent_t stage_full[2] = {nullptr, nullptr};
  // grow-only device workspaces of the cosine stage (slot i = i-th request of a call); cudaMalloc /
  // cudaFree of a few hundred MB per call would otherwise cost more than the kernels
  std::vector<std::pair<void*, size_t>> ws;
  // grow-only workspaces of the grouped K1 path (group.cu) and of the event router (route.cu)
  std::vector<std::pair<void*, size_t>> ws_group;
  int64_t group_min_events = 1 << 16;  // MB200_OPT_GROUP_MIN_EVENTS
  int group_prefetch = 0;              // MB200_OPT_GROUP_PREFETCH
  int single_kernel = 1;               // MB200_OPT_SINGLE_KERNEL
  int64_t max_fallback_rows = -1;      // MB200_OPT_MAX_FALLBACK_ROWS
  // grow-only device staging of host-memory arguments (see io_slot in sketch.cu)
  std::pair<void*, size_t> io[3] = {{nullptr, 0}, {nullptr, 0}, {nullptr, 0}};
  // pull-gather: per-block arrival flags written by the copy stream, read by K3 (+ 1 abort word)
  uint32_t* gather_flags = nullptr;
  uint32_t* gather_abort = nullptr;
  uint32_t gather_epoch = 0;
  cudaEvent_t gather_ev = nullptr;
  cudaEvent_t fence_ev = nullptr;  // mb200_gather_fence
  int64_t last_fallback_rows = 0;
  int64_t last_band_rows = 0, stat_band = 0;
  int64_t stat_events = 0, stat_rows = 0, stat_fallback = 0, stat_h2d = 0, stat_d2h = 0;
  struct mb200_cosine_job* active_job = nullptr;  // the cosine stage's workspaces serve one job at a time
  mb200_recommend_plan last_recommend_plan = {};  // mb200_recommend_last_plan
  mb200_itembased_plan last_itembased_plan = {};  // mb200_itembased_last_plan
  mb200_sized_plan last_sized_plan = {};          // mb200_sized_last_plan
  mb200_sized_recommend_plan last_sized_recommend_plan = {};  // mb200_sized_recommend_last_plan
  int64_t itembased_dense_items = -1, itembased_dense_slices = -1;  // layout of the zeroed dense slices (slot 62)
};

// borrows workspace slots from the context in request order; nothing is freed on return
struct Workspace {
  mb200_ctx* ctx;
  size_t next = 0;
  explicit Workspace(mb200_ctx* c) : ctx(c) {}
  int get(size_t bytes, void** out);
};

struct mb200_bank {
  mb200_ctx* ctx = nullptr;
  int64_t E = 0;
  int32_t d = 0, W = 0, frac_bits = 0;
  HashFamily hf;
  int64_t a_raw[MB200_MAX_DEPTH], b_raw[MB200_MAX_DEPTH];
  long long* counters = nullptr;  // [E][d][W] fixed point
  unsigned long long* flags = nullptr;  // FLAG_WORDS
  double events_total = 0;  // for the conservative range bound
  bool virgin = true;       // nothing has been added since creation / clear: the counters are all zero
};

int mb200_fail(mb200_ctx* ctx, int code, const char* fmt, ...);
// group.cu: bank-mode K1 through device-side grouping (called with ctx->mu held)
bool mb200_group_applicable(const mb200_bank* bk, int64_t n);
int mb200_group_ws(mb200_ctx* ctx, size_t slot, size_t bytes, void** out);  // grow-only slot of ctx->ws_group
template <typename T>
int mb200_group_update(mb200_bank* bk, const long long* entity, const long long* key, const T* inc, int64_t n);
extern "C" void mb200_job_release(struct mb200_cosine_job* job);  // cosine.cu (internal)
void mb200_set_global_error(const char* msg);

#define MB_CUDA(ctx, expr)                                                                   \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return mb200_fail((ctx), _e == cudaErrorMemoryAllocation ? MB200_ERR_OOM : MB200_ERR_CUDA, \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define MB_CHECK(call)          \
  do {                          \
    int _rc = (call);           \
    if (_rc != MB200_OK) return _rc; \
  } while (0)

// profiling helpers: bracket a kernel launch with events when profiling is on
struct ProfScope {
  mb200_ctx* ctx;
  int idx = -1;
  ProfScope(mb200_ctx* c, int kernel_id);
  ~ProfScope();
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
