// multi.cuh -- the one-process multi-GPU handle (mb200_create_multi, csrc/job.cu) and the host helpers shared by
// the calls that drive it: the item-similarity job (job.cu), the replicated sized bank (sized_multi.cu) and the
// replicated item-based recommender (itembased_multi.cu).
#pragma once

#include <stdarg.h>
#include <stdio.h>

#include <chrono>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

struct mb200_multi {
  int n = 0;
  std::vector<int> devices;
  std::vector<mb200_ctx*> ctx;
  std::string err;
  std::mutex mu;  // one call at a time per handle
};

static inline double multi_now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static inline int multi_fail(mb200_multi* m, int code, const std::string& msg) {
  if (m) m->err = msg;
  mb200_set_global_error(msg.c_str());
  return code;
}

static inline int multi_bad_arg(mb200_multi* m, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
static inline int multi_bad_arg(mb200_multi* m, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  return multi_fail(m, MB200_ERR_BAD_ARG, buf);
}

// the last call of a replicated handle: per-GPU work and worker wall clock, the call's wall clock
struct MultiStats {
  std::vector<int64_t> work;
  std::vector<double> seconds;
  double wall_s = 0;
};

// one GPU's part of a call: the first failure, and the device buffers it allocated
struct Part {
  mb200_ctx* ctx = nullptr;
  int rc = MB200_OK;
  std::string msg;
  std::vector<void*> dev;

  bool ok() const { return rc == MB200_OK; }
  void take(int code) {  // a single-context call's status
    if (code != MB200_OK && ok()) {
      rc = code;
      msg = mb200_last_error(ctx);
    }
  }
  void cuda(cudaError_t e, const char* what) {
    if (e != cudaSuccess && ok()) {
      rc = e == cudaErrorMemoryAllocation ? MB200_ERR_OOM : MB200_ERR_CUDA;
      msg = std::string(what) + " failed: " + cudaGetErrorString(e);
    }
  }
  template <typename T>
  T* alloc(size_t n) {
    void* p = nullptr;
    if (!ok()) return nullptr;
    cuda(cudaMalloc(&p, (n ? n : 1) * sizeof(T)), "cudaMalloc");
    if (!ok()) return nullptr;
    dev.push_back(p);
    return (T*)p;
  }
  template <typename T>
  T* upload(const T* h, size_t n) {
    T* d = alloc<T>(n);
    if (ok() && n) cuda(cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream), "cudaMemcpyAsync H2D");
    return d;
  }
  template <typename T>
  void download(std::vector<T>& h, const T* d, size_t n) {
    h.resize(n);
    if (ok() && n) cuda(cudaMemcpyAsync(h.data(), d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream), "cudaMemcpyAsync D2H");
  }
  void finish() {
    if (ok()) cuda(cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize");
  }
  void release() {
    for (void* p : dev) cudaFree(p);
    dev.clear();
  }
};

// the positions t = l * G + g of [0, q) that go to GPU g
static inline int64_t multi_share(int64_t q, int g, int G) { return q > g ? (q - g + G - 1) / G : 0; }

// v[g], v[g + G], ... : GPU g's share of [0, q)
static inline std::vector<int64_t> multi_gather(const int64_t* v, int64_t q, int g, int G) {
  std::vector<int64_t> out((size_t)multi_share(q, g, G));
  for (size_t l = 0; l < out.size(); l++) out[l] = v[(int64_t)l * G + g];
  return out;
}

// runs fn(g, part) on one worker thread per GPU of m (GPU 0 on the caller's), records the per-GPU and wall times in
// st, and returns the first failing GPU's status with "GPU d: <message>".  Buffers a part allocated are freed when
// its worker ends.
template <typename F>
int run_parts(mb200_multi* m, MultiStats& st, F&& fn) {
  const int G = m->n;
  std::vector<Part> parts(G);
  st.work.assign(G, 0);
  st.seconds.assign(G, 0.0);
  int caller_device = 0;
  cudaGetDevice(&caller_device);
  const double t0 = multi_now_s();
  auto one = [&](int g) {
    const double s = multi_now_s();
    Part& p = parts[g];
    p.ctx = m->ctx[g];
    p.cuda(cudaSetDevice(p.ctx->device), "cudaSetDevice");
    if (p.ok()) fn(g, p);
    if (!p.ok()) cudaStreamSynchronize(p.ctx->stream);  // nothing may still use the buffers freed below
    p.release();
    st.seconds[g] = multi_now_s() - s;
  };
  std::vector<std::thread> th;
  for (int g = 1; g < G; g++) th.emplace_back(one, g);
  one(0);
  for (auto& t : th) t.join();
  st.wall_s = multi_now_s() - t0;
  cudaSetDevice(caller_device);  // GPU 0's worker ran on the caller's thread
  for (int g = 0; g < G; g++)
    if (!parts[g].ok()) return multi_fail(m, parts[g].rc, "GPU " + std::to_string(m->devices[g]) + ": " + parts[g].msg);
  return MB200_OK;
}

static inline void multi_last_stats(const MultiStats& st, int64_t* work, double* seconds, double* wall_s) {
  for (size_t g = 0; g < st.work.size(); g++) {
    if (work) work[g] = st.work[g];
    if (seconds) seconds[g] = st.seconds[g];
  }
  if (wall_s) *wall_s = st.wall_s;
}
