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

// Named grow-only device workspaces of the context (ws_slot).  Two buffers live in the same call have different
// names; buffers of the same role in calls that never run together share one.
enum WsSlot {
  WS_GROUP_SMALL,     // group.cu: histogram, segment offsets, cursors and ticket of one sub-batch
  WS_GROUP_KQ2,       // group.cu: (key, quanta) records in entity order
  WS_GROUP_KQ1,       // group.cu: (key, quanta) records after the coarse level
  WS_GROUP_ENT1,      // group.cu: entities after the coarse level
  WS_GROUP_WINDOWS,   // group.cu: first record of each K1 window
  WS_GROUP_TILES,     // group.cu: tile descriptors of the second scatter level
  WS_GROUP_TICKET,    // group.cu: work ticket of mb200_bank_update_grouped
  WS_ROUTE,           // route.cu: per-shard counts and cursors
  WS_WIDEN_ENTITY,    // sketch.cu: entity column of widened u8 events
  WS_WIDEN_KEY,       // sketch.cu: key column of widened u8 events
  WS_WIDEN_INC,       // sketch.cu: increment column of widened u8 events
  WS_KEYTAB,          // sketch.cu: the K1 key table, all zero between calls
  WS_K1_STATS,        // sketch.cu: MB200_TRACE counters of K1
  WS_STATUS,          // recommend.cu, cmsized.cu: plan and status words of a call (StatusWords)
  WS_REC_BITMAP,      // recommend.cu, cmsized.cu: per-CTA candidate bitmaps of k_recommend / k_sized_recommend
  WS_REC_CAND,        // recommend.cu, cmsized.cu: per-CTA candidate lists
  WS_REC_KEY,         // recommend.cu, cmsized.cu: per-CTA top-N keys
  WS_REC_VAL,         // recommend.cu, cmsized.cu: per-CTA estimates
  WS_IB_RANK_KEY,     // recommend.cu: (itemID, row) sort keys of the item-based rank table
  WS_IB_RANK_ROW,     // recommend.cu: rank -> row
  WS_IB_RANK_OF,      // recommend.cu: row -> rank
  WS_IB_DENSE,        // recommend.cu: item-based dense slices, kept zero by k_itembased
  WS_IB_LOCKS,        // recommend.cu: locks of the dense slices
  WS_SIZED_ITEM,      // cmsized.cu: item column of the prefs while a sized bank is built
  WS_SIZED_PREF,      // cmsized.cu: pref column of the prefs while a sized bank is built
  WS_SIZED_SIMS,      // cmsized.cu: similarities of a query batch
  WS_SIZED_SLICE,     // cmsized.cu: per-CTA global sketch slices (pair cosine, neighbourhood)
  WS_SIZED_CLASSES,   // cmsized.cu: shape-class table of a neighbourhood call
  WS_SIZED_ITEMS,     // cmsized.cu: work items of a neighbourhood batch
  WS_SLOT_COUNT
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
  // named grow-only workspaces (WsSlot)
  std::pair<void*, size_t> ws_slots[WS_SLOT_COUNT] = {};
  int64_t group_min_events = 1 << 16;  // MB200_OPT_GROUP_MIN_EVENTS
  int group_prefetch = 0;              // MB200_OPT_GROUP_PREFETCH
  int64_t max_fallback_rows = -1;      // MB200_OPT_MAX_FALLBACK_ROWS
  // grow-only device staging of host-memory arguments, in request order within a call (ArgStage)
  std::vector<std::pair<void*, size_t>> io;
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
  int64_t itembased_dense_items = -1, itembased_dense_slices = -1;  // layout of the zeroed dense slices (WS_IB_DENSE)
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
// the named workspace `slot`, (re)allocated when smaller than `bytes`; *fresh tells that it just was
int ws_slot(mb200_ctx* ctx, WsSlot slot, size_t bytes, void** out, bool* fresh = nullptr);
// group.cu: bank-mode K1 through device-side grouping (called with ctx->mu held)
bool mb200_group_applicable(const mb200_bank* bk, int64_t n);
template <typename T>
int mb200_group_update(mb200_bank* bk, const long long* entity, const long long* key, const T* inc, int64_t n);
extern "C" void mb200_job_release(struct mb200_cosine_job* job);  // cosine.cu (internal)
void mb200_set_global_error(const char* msg);
// recommend.cu: mb200_recommend_item_based, except that with data_on_device the lists, the user CSR and the itemIDs
// are device pointers whatever args->mem says (itembased_multi.cu's replicas); the other arrays follow args->mem
int mb200_itembased_call(mb200_ctx* ctx, const mb200_itembased_args* args, bool data_on_device);

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

// A call's array arguments.  Under MB200_MEM_DEVICE, and for a NULL input, the caller's pointer passes through;
// otherwise in() copies the host array into ctx->io and out() lends a buffer there that finish() copies back.
// ctx->io is taken in request order, so no staged call may run while another is in progress.  The caller's host
// buffers are only borrowed for the call: finish() synchronises when anything was staged, and the destructor does
// when inputs were staged and finish() did not run.
struct ArgStage {
  mb200_ctx* ctx;
  int mem;
  ArgStage(mb200_ctx* c, int m) : ctx(c), mem(m) {}
  ~ArgStage();
  template <typename T>
  int in(const T* user, size_t n, const T** dev) {
    *dev = user;
    if (mem == MB200_MEM_DEVICE || !user) return MB200_OK;
    void* p = nullptr;
    MB_CHECK(buffer(n * sizeof(T), &p));
    if (n) MB_CUDA(ctx, cudaMemcpyAsync(p, user, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    ctx->stat_h2d += (int64_t)(n * sizeof(T));
    inputs = true;
    *dev = (const T*)p;
    return MB200_OK;
  }
  template <typename T>
  int out(T* user, size_t n, T** dev) {
    *dev = user;
    if (mem == MB200_MEM_DEVICE) return MB200_OK;
    void* p = nullptr;
    MB_CHECK(buffer(n * sizeof(T), &p));
    outs.push_back({p, user, n * sizeof(T)});
    *dev = (T*)p;
    return MB200_OK;
  }
  int finish();

 private:
  struct Out {
    void* dev;
    void* user;
    size_t bytes;
  };
  size_t next = 0;
  bool inputs = false;  // staged inputs not yet synchronised
  std::vector<Out> outs;
  int buffer(size_t bytes, void** out);
};

// `n` status / plan words in a named workspace: zero() clears them on the stream before the launch, read() copies
// them to the host with one synchronise
struct StatusWords {
  mb200_ctx* ctx;
  size_t n;
  unsigned long long* dev = nullptr;
  StatusWords(mb200_ctx* c, size_t words) : ctx(c), n(words) {}
  int zero(WsSlot slot);
  int read(unsigned long long* h);
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
