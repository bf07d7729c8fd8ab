// runtime.cu -- context lifetime, error reporting, profiling spans, host-side hash parameters.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

static thread_local std::string g_last_error;

void mb200_set_global_error(const char* msg) { g_last_error = msg; }

int mb200_fail(mb200_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  if (ctx) ctx->err = buf;
  return code;
}

// Grow-only device buffer: reallocated only when smaller than `bytes`, never freed on return.  cudaMalloc / cudaFree
// synchronise the device and were measured at 1 ms .. 1 s each on a process holding tens of GB.
static int grow(mb200_ctx* ctx, std::pair<void*, size_t>& slot, size_t bytes, void** out, bool* fresh = nullptr) {
  if (fresh) *fresh = false;
  if (slot.second < bytes || !slot.first) {
    if (slot.first) cudaFree(slot.first);
    slot.first = nullptr;
    slot.second = 0;
    const size_t want = bytes ? bytes : 1;
    cudaError_t e = cudaMalloc(&slot.first, want);
    if (e != cudaSuccess) {
      slot.first = nullptr;
      return mb200_fail(ctx, MB200_ERR_OOM, "cannot allocate %zu bytes of workspace: %s", want, cudaGetErrorString(e));
    }
    slot.second = want;
    if (fresh) *fresh = true;
  }
  *out = slot.first;
  return MB200_OK;
}

// the next buffer of a request-order pool (a cosine job may start its requests past the pool's end)
static int grow_next(mb200_ctx* ctx, std::vector<std::pair<void*, size_t>>& pool, size_t& next, size_t bytes,
                     void** out) {
  while (next >= pool.size()) pool.emplace_back(nullptr, 0);
  return grow(ctx, pool[next++], bytes, out);
}

int Workspace::get(size_t bytes, void** out) { return grow_next(ctx, ctx->ws, next, bytes, out); }

int ws_slot(mb200_ctx* ctx, WsSlot slot, size_t bytes, void** out, bool* fresh) {
  return grow(ctx, ctx->ws_slots[slot], bytes, out, fresh);
}

int ArgStage::buffer(size_t bytes, void** out) { return grow_next(ctx, ctx->io, next, bytes, out); }

int ArgStage::finish() {
  if (!inputs && outs.empty()) return MB200_OK;
  for (auto& o : outs) {
    if (o.bytes) MB_CUDA(ctx, cudaMemcpyAsync(o.user, o.dev, o.bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stat_d2h += (int64_t)o.bytes;
  }
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  inputs = false;
  outs.clear();
  return MB200_OK;
}

ArgStage::~ArgStage() {
  // pageable inputs are already copied when cudaMemcpyAsync returns; pinned ones are read asynchronously
  if (inputs) cudaStreamSynchronize(ctx->stream);
}

int StatusWords::zero(WsSlot slot) {
  void* p = nullptr;
  MB_CHECK(ws_slot(ctx, slot, n * sizeof(unsigned long long), &p));
  MB_CUDA(ctx, cudaMemsetAsync(p, 0, n * sizeof(unsigned long long), ctx->stream));
  dev = (unsigned long long*)p;
  return MB200_OK;
}

int StatusWords::read(unsigned long long* h) {
  MB_CUDA(ctx, cudaMemcpyAsync(h, dev, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MB200_OK;
}

ProfScope::ProfScope(mb200_ctx* c, int kernel_id) : ctx(c) {
  if (!ctx->profiling) return;
  ProfSpan s;
  s.kernel_id = kernel_id;
  cudaEvent_t ev[2];
  for (int i = 0; i < 2; i++) {
    if (!ctx->event_pool.empty()) {
      ev[i] = ctx->event_pool.back();
      ctx->event_pool.pop_back();
    } else if (cudaEventCreate(&ev[i]) != cudaSuccess) {
      return;
    }
  }
  s.beg = ev[0];
  s.end = ev[1];
  cudaEventRecord(s.beg, ctx->stream);
  ctx->spans.push_back(s);
  idx = (int)ctx->spans.size() - 1;
}

ProfScope::~ProfScope() {
  if (idx >= 0) cudaEventRecord(ctx->spans[idx].end, ctx->stream);
}

static int resolve_spans(mb200_ctx* ctx) {
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& s : ctx->spans) {
    float ms = 0.f;
    MB_CUDA(ctx, cudaEventElapsedTime(&ms, s.beg, s.end));
    ctx->prof_ms[s.kernel_id] += ms;
    ctx->prof_n[s.kernel_id] += 1;
    ctx->event_pool.push_back(s.beg);
    ctx->event_pool.push_back(s.end);
  }
  ctx->spans.clear();
  return MB200_OK;
}

extern "C" {

int mb200_create(int device, mb200_ctx** out) {
  if (!out) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return mb200_fail(nullptr, MB200_ERR_NO_DEVICE,
                      "mb200_create: no CUDA device (%s); this library has no CPU fallback",
                      e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= n)
    return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_create: device %d out of range [0,%d)", device, n);
  cudaDeviceProp prop;
  MB_CUDA(nullptr, cudaSetDevice(device));
  MB_CUDA(nullptr, cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return mb200_fail(nullptr, MB200_ERR_NO_DEVICE,
                      "mb200_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                      device, prop.major, prop.minor);
  mb200_ctx* ctx = new mb200_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  MB_CUDA(nullptr, cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
  MB_CUDA(nullptr, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) {
    MB_CUDA(nullptr, cudaEventCreateWithFlags(&ctx->stage_free[i], cudaEventDisableTiming));
    MB_CUDA(nullptr, cudaEventCreateWithFlags(&ctx->stage_full[i], cudaEventDisableTiming));
  }
  ctx->stream = ctx->own_stream;
  *out = ctx;
  return MB200_OK;
}

int mb200_destroy(mb200_ctx* ctx) {
  if (!ctx) return MB200_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->copy_stream);
  if (ctx->active_job) mb200_job_release(ctx->active_job);
  for (auto& s : ctx->spans) {
    cudaEventDestroy(s.beg);
    cudaEventDestroy(s.end);
  }
  for (auto ev : ctx->event_pool) cudaEventDestroy(ev);
  for (auto& w : ctx->ws)
    if (w.first) cudaFree(w.first);
  for (auto& w : ctx->io)
    if (w.first) cudaFree(w.first);
  for (auto& w : ctx->ws_slots)
    if (w.first) cudaFree(w.first);
  if (ctx->gather_flags) cudaFree(ctx->gather_flags);
  if (ctx->gather_ev) cudaEventDestroy(ctx->gather_ev);
  if (ctx->fence_ev) cudaEventDestroy(ctx->fence_ev);
  for (int i = 0; i < 2; i++) {
    if (ctx->stage[i]) cudaFree(ctx->stage[i]);
    cudaEventDestroy(ctx->stage_free[i]);
    cudaEventDestroy(ctx->stage_full[i]);
  }
  cudaStreamDestroy(ctx->own_stream);
  cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
  return MB200_OK;
}

const char* mb200_last_error(mb200_ctx* ctx) {
  if (ctx && !ctx->err.empty()) return ctx->err.c_str();
  return g_last_error.c_str();
}

int mb200_get_stats(mb200_ctx* ctx, mb200_stats* out) {
  if (!ctx || !out) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_get_stats: NULL argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  memset(out, 0, sizeof(*out));
  out->device = ctx->device;
  out->num_sms = ctx->num_sms;
  out->launches = ctx->launches;
  for (auto& w : ctx->ws) out->workspace_bytes += (int64_t)w.second;
  for (auto& w : ctx->ws_slots) out->workspace_bytes += (int64_t)w.second;
  for (auto& w : ctx->io) out->staging_bytes += (int64_t)w.second;
  out->staging_bytes += 2 * (int64_t)ctx->stage_bytes;
  out->last_fallback_rows = ctx->last_fallback_rows;
  out->cosine_job_active = ctx->active_job ? 1 : 0;
  out->events_updated = ctx->stat_events;
  out->rows_scored = ctx->stat_rows;
  out->fallback_rows_total = ctx->stat_fallback;
  out->band_rows_total = ctx->stat_band;
  out->h2d_bytes = ctx->stat_h2d;
  out->d2h_bytes = ctx->stat_d2h;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, ctx->device) == cudaSuccess) {
    strncpy(out->device_name, prop.name, sizeof(out->device_name) - 1);
  }
  return MB200_OK;
}

int mb200_release_workspace(mb200_ctx* ctx) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_release_workspace: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->active_job)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_release_workspace: a cosine job is active on this context");
  for (auto& w : ctx->ws)
    if (w.first) cudaFree(w.first);
  ctx->ws.clear();
  for (auto& w : ctx->ws_slots) {
    if (w.first) cudaFree(w.first);
    w = {nullptr, 0};
  }
  for (auto& w : ctx->io)
    if (w.first) cudaFree(w.first);
  ctx->io.clear();
  return MB200_OK;
}

int mb200_set_stream(mb200_ctx* ctx, void* cuda_stream) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_set_stream: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return MB200_OK;
}

int mb200_set_option(mb200_ctx* ctx, int option, int64_t value) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_set_option: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  switch (option) {
    case MB200_OPT_GROUP_MIN_EVENTS:
      if (value < 0) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_set_option: GROUP_MIN_EVENTS must be >= 0");
      ctx->group_min_events = value;
      return MB200_OK;
    case MB200_OPT_MAX_FALLBACK_ROWS:
      ctx->max_fallback_rows = value;
      return MB200_OK;
    case MB200_OPT_GROUP_PREFETCH:
      ctx->group_prefetch = value ? 1 : 0;
      return MB200_OK;
    default:
      return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_set_option: unknown option %d", option);
  }
}

int mb200_sync(mb200_ctx* ctx) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sync: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return MB200_OK;
}

int mb200_set_profiling(mb200_ctx* ctx, int on) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_set_profiling: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  ctx->profiling = on != 0;
  return MB200_OK;
}

int mb200_kernel_time(mb200_ctx* ctx, int kernel_id, double* total_ms, int64_t* launches) {
  if (!ctx || kernel_id < 0 || kernel_id >= MB200_K_COUNT)
    return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_kernel_time: bad arguments");
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CHECK(resolve_spans(ctx));
  if (total_ms) *total_ms = ctx->prof_ms[kernel_id];
  if (launches) *launches = ctx->prof_n[kernel_id];
  return MB200_OK;
}

int mb200_reset_profile(mb200_ctx* ctx) {
  if (!ctx) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_reset_profile: ctx is NULL");
  std::lock_guard<std::mutex> g(ctx->mu);
  MB_CUDA(ctx, cudaSetDevice(ctx->device));
  MB_CHECK(resolve_spans(ctx));
  for (int i = 0; i < MB200_K_COUNT; i++) {
    ctx->prof_ms[i] = 0;
    ctx->prof_n[i] = 0;
  }
  return MB200_OK;
}

int mb200_launch_count(mb200_ctx* ctx, int64_t* launches) {
  if (!ctx || !launches) return mb200_fail(ctx, MB200_ERR_BAD_ARG, "mb200_launch_count: bad arguments");
  *launches = ctx->launches;
  return MB200_OK;
}

int mb200_host_alloc(int64_t bytes, void** out) {
  if (!out || bytes < 0) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_host_alloc: bad arguments");
  *out = nullptr;
  cudaError_t e = cudaHostAlloc(out, bytes > 0 ? (size_t)bytes : 1, cudaHostAllocPortable);
  if (e != cudaSuccess)
    return mb200_fail(nullptr, MB200_ERR_OOM, "mb200_host_alloc(%lld): %s", (long long)bytes, cudaGetErrorString(e));
  return MB200_OK;
}

int mb200_host_free(void* ptr) {
  if (!ptr) return MB200_OK;
  cudaError_t e = cudaFreeHost(ptr);
  if (e != cudaSuccess) return mb200_fail(nullptr, MB200_ERR_CUDA, "mb200_host_free: %s", cudaGetErrorString(e));
  return MB200_OK;
}

int mb200_host_register(void* ptr, int64_t bytes) {
  if (!ptr || bytes <= 0) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_host_register: bad arguments");
  cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable);
  if (e != cudaSuccess) return mb200_fail(nullptr, MB200_ERR_CUDA, "mb200_host_register: %s", cudaGetErrorString(e));
  return MB200_OK;
}

int mb200_host_unregister(void* ptr) {
  if (!ptr) return MB200_OK;
  cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) return mb200_fail(nullptr, MB200_ERR_CUDA, "mb200_host_unregister: %s", cudaGetErrorString(e));
  return MB200_OK;
}

// ---- host-side set-up arithmetic (not the hot path) -------------------------------------------
// java.util.Random as specified by Java SE; HashFunctionBuilder.java:23-28,40-60 draws
// ra = Math.abs(nextLong()), rb = Math.abs(nextLong()) per iteration index, in that order.
static inline int32_t jrand_next(uint64_t& s, int bits) {
  s = (s * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
  return (int32_t)((int64_t)s >> (48 - bits));
}
static inline int64_t jrand_long(uint64_t& s) {
  int64_t hi = jrand_next(s, 32);
  int64_t lo = jrand_next(s, 32);
  return (int64_t)(((uint64_t)hi << 32) + (uint64_t)lo);
}

int mb200_hash_params(int64_t seed, int depth, int64_t* a, int64_t* b) {
  if (depth < 0 || (depth > 0 && (!a || !b)))
    return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_hash_params: bad arguments");
  uint64_t s = ((uint64_t)seed ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1);
  for (int i = 0; i < depth; i++) {
    int64_t ra = jrand_long(s), rb = jrand_long(s);
    a[i] = ra < 0 ? (int64_t)(0ULL - (uint64_t)ra) : ra;  // Math.abs: Long.MIN_VALUE stays negative
    b[i] = rb < 0 ? (int64_t)(0ULL - (uint64_t)rb) : rb;
  }
  return MB200_OK;
}

int mb200_cm_dims(double delta, double epsilon, int32_t* width, int32_t* depth) {
  if (!width || !depth) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_cm_dims: NULL output");
  // AbstractCountMinSketch.java:71-76 (message text kept)
  if (!(delta > 0) || delta > exp(-1.0))
    return mb200_fail(nullptr, MB200_ERR_CM_DELTA, "CountMinSketch: delta must be between 0 and 1, exclusive");
  if (!(epsilon > 0) || epsilon > exp(1.0))
    return mb200_fail(nullptr, MB200_ERR_CM_EPSILON, "CountMinSketch: epsilon must be between 0 and 1, exclusive");
  *width = (int32_t)ceil(exp(1.0) / epsilon);
  *depth = (int32_t)ceil(log(1.0 / delta));
  return MB200_OK;
}

}  // extern "C"
