// job.cu -- the whole item-similarity phase behind one C call, on one GPU or on all GPUs of the box.
//
// Replaces phase 1 of ItemSimilarityJob.run (cf/taste/hadoop/similarity/item/ItemSimilarityJob.java:146-162,
// the RowSimilarityJob invocation) for a JVM that holds the prepared preference events: ONE process, one
// mb200_ctx and one host worker thread per GPU (SURVEY.md 8b), no torch, no NCCL -- inside one process the
// GPUs reach each other's memory directly (cudaDeviceEnablePeerAccess), so the cross-GPU steps are the same
// peer stores and copy-engine pulls the one-process-per-GPU path uses:
//
//   slice      GPU g takes events [g*n/G, (g+1)*n/G) of the caller's host columns (H2D)
//   route      mb200_route_count -> host G x G count matrix -> mb200_route_scatter: partition by owner
//              (row mod G) + NVLink stores straight into the owners' receive columns (route.cu)
//   build      mb200_bank_update on the owner: grouped K1 (group.cu)
//   normalise  K2 into a peer-readable row buffer
//   cosine     mb200_gather_pull (copy engines pull the shards; arrival flags) + ONE K3 launch per GPU that
//              consumes the blocks in order of arrival, top-k fused; CERTIFIED reads the undecided
//              candidates from the owners' banks through the peer mappings, RESCORED from peer copies
//   results    every GPU returns the top-k of its own rows; the caller's arrays are in global row order
//
// Host threads meet at barriers between the steps that read another GPU's memory.
#include <string.h>

#include <condition_variable>
#include <thread>

#include "multi.cuh"

namespace {

struct HostBarrier {
  std::mutex m;
  std::condition_variable cv;
  int n, waiting = 0, generation = 0;
  explicit HostBarrier(int n_) : n(n_) {}
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    const int gen = generation;
    if (++waiting == n) {
      waiting = 0;
      generation++;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return gen != generation; });
    }
  }
};

struct Shared {
  mb200_multi* m;
  const mb200_job_params* p;
  const int64_t *row, *key;
  const float* inc;
  int64_t n, num_items, E_loc;
  int G;
  HostBarrier bar;
  std::vector<std::vector<int64_t>> counts;  // [src][dst]
  std::vector<void*> r_row, r_key, r_inc;    // receive columns per GPU
  std::vector<void*> rows16, valid, counters, n32, gathered;
  std::vector<int64_t> recv;
  std::vector<int> rc;
  std::vector<std::string> msg;
  std::vector<int64_t> fallback;
  std::vector<int32_t> pull_retries;  // 1 = this GPU repeated its cosine phase without arrival flags
  std::vector<int32_t> mixed;
  int64_t* out_idx;
  double* out_sim;
  int32_t* out_cnt;
  double t_route = 0, t_build = 0, t_cosine = 0;
  Shared(int g) : bar(g) {}
  bool failed() const {
    for (int r : rc)
      if (r != MB200_OK) return true;
    return false;
  }
};

#define JOB_TRY(call)                                  \
  do {                                                 \
    int rc_ = (call);                                  \
    if (rc_ != MB200_OK && sh.rc[g] == MB200_OK) {     \
      sh.rc[g] = rc_;                                  \
      sh.msg[g] = mb200_last_error(ctx);               \
    }                                                  \
  } while (0)
#define JOB_CUDA(expr)                                                                       \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess && sh.rc[g] == MB200_OK) {                                         \
      sh.rc[g] = e_ == cudaErrorMemoryAllocation ? MB200_ERR_OOM : MB200_ERR_CUDA;           \
      sh.msg[g] = std::string(#expr) + " failed: " + cudaGetErrorString(e_);                 \
    }                                                                                        \
  } while (0)
// every thread passes every barrier even after a failure: nobody may be left waiting
#define OK_SO_FAR (sh.rc[g] == MB200_OK)

void worker(Shared& sh, int g) {
  mb200_ctx* ctx = sh.m->ctx[g];
  const mb200_job_params& P = *sh.p;
  const int G = sh.G;
  cudaSetDevice(ctx->device);
  const int64_t s0 = sh.n * g / G, s1 = sh.n * (g + 1) / G, ns = s1 - s0;
  void *d_row = nullptr, *d_key = nullptr, *d_inc = nullptr;
  const double t0 = multi_now_s();
  // ---- slice + count
  if (ns > 0) {
    JOB_CUDA(cudaMalloc(&d_row, (size_t)ns * 8));
    JOB_CUDA(cudaMalloc(&d_key, (size_t)ns * 8));
    JOB_CUDA(cudaMalloc(&d_inc, (size_t)ns * 4));
    if (OK_SO_FAR) {
      JOB_CUDA(cudaMemcpyAsync(d_row, sh.row + s0, (size_t)ns * 8, cudaMemcpyHostToDevice, ctx->stream));
      JOB_CUDA(cudaMemcpyAsync(d_key, sh.key + s0, (size_t)ns * 8, cudaMemcpyHostToDevice, ctx->stream));
      JOB_CUDA(cudaMemcpyAsync(d_inc, sh.inc + s0, (size_t)ns * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
  }
  sh.counts[g].assign(G, 0);
  if (OK_SO_FAR && G > 1) JOB_TRY(mb200_route_count(ctx, (const int64_t*)d_row, ns, G, sh.counts[g].data()));
  if (G == 1) sh.counts[g][0] = ns;
  sh.bar.wait();
  // ---- receive columns
  int64_t recv = 0;
  for (int s = 0; s < G; s++) recv += sh.counts[s][g];
  sh.recv[g] = recv;
  if (G > 1 && !sh.failed()) {
    JOB_CUDA(cudaMalloc(&sh.r_row[g], (size_t)(recv > 0 ? recv : 1) * 8));
    JOB_CUDA(cudaMalloc(&sh.r_key[g], (size_t)(recv > 0 ? recv : 1) * 8));
    JOB_CUDA(cudaMalloc(&sh.r_inc[g], (size_t)(recv > 0 ? recv : 1) * 4));
  }
  sh.bar.wait();
  // ---- route: partition by owner + peer stores
  if (G > 1 && !sh.failed()) {
    std::vector<int64_t> off(G, 0);
    for (int d = 0; d < G; d++)
      for (int s = 0; s < g; s++) off[d] += sh.counts[s][d];
    JOB_TRY(mb200_route_scatter(ctx, (const int64_t*)d_row, (const int64_t*)d_key, (const float*)d_inc, ns, G,
                                sh.r_row.data(), sh.r_key.data(), sh.r_inc.data(), off.data()));
    JOB_TRY(mb200_sync(ctx));
  }
  sh.bar.wait();
  if (g == 0) sh.t_route = multi_now_s() - t0;
  const double t1 = multi_now_s();
  // ---- build the shard bank
  mb200_bank* bank = nullptr;
  if (!sh.failed()) {
    if (P.hash_a && P.hash_b)
      JOB_TRY(mb200_bank_create_params(ctx, sh.E_loc, P.depth, P.width, P.hash_a, P.hash_b, P.frac_bits, &bank));
    else
      JOB_TRY(mb200_bank_create(ctx, sh.E_loc, P.depth, P.width, P.seed, P.frac_bits, &bank));
    if (OK_SO_FAR && recv > 0) {
      if (G > 1)
        JOB_TRY(mb200_bank_update(bank, (const int64_t*)sh.r_row[g], (const int64_t*)sh.r_key[g], (const float*)sh.r_inc[g],
                                  recv, MB200_MEM_DEVICE));
      else
        JOB_TRY(mb200_bank_update(bank, (const int64_t*)d_row, (const int64_t*)d_key, (const float*)d_inc, ns, MB200_MEM_DEVICE));
    }
    if (OK_SO_FAR) JOB_TRY(mb200_bank_check(bank));
  }
  cudaFree(d_row);
  cudaFree(d_key);
  cudaFree(d_inc);
  if (G > 1) {
    cudaFree(sh.r_row[g]);
    cudaFree(sh.r_key[g]);
    cudaFree(sh.r_inc[g]);
  }
  mb200_release_workspace(ctx);  // the grouping workspaces: 20 B per event
  if (g == 0) sh.t_build = multi_now_s() - t1;
  const double t2 = multi_now_s();
  const int k = P.k;
  const int64_t E = sh.E_loc;
  void *o_idx = nullptr, *o_sim = nullptr, *o_cnt = nullptr;
  JOB_CUDA(cudaMalloc(&o_idx, (size_t)E * k * 8));
  JOB_CUDA(cudaMalloc(&o_sim, (size_t)E * k * 8));
  JOB_CUDA(cudaMalloc(&o_cnt, (size_t)E * 4));
  if (G == 1) {
    if (OK_SO_FAR)
      JOB_TRY(mb200_bank_cosine_topk(bank, k, P.threshold, 1, P.dtype, P.precision, (int64_t*)o_idx, (double*)o_sim,
                                     (int32_t*)o_cnt, MB200_MEM_DEVICE));
    if (OK_SO_FAR) JOB_TRY(mb200_cosine_last_fallback_rows(ctx, &sh.fallback[g]));
  } else {
    // ---- K2 into peer-readable rows; peers' counters for the exact-set precisions
    const int64_t ld = mb200_row_ld(P.width), vw = mb200_valid_words(E);
    const int64_t rows_bytes = (int64_t)P.depth * E * ld * 2, valid_bytes = (int64_t)P.depth * vw * 4;
    const int64_t cells = E * (int64_t)P.depth * P.width;
    void *staging = nullptr, *staging_v = nullptr;
    if (!sh.failed()) {
      JOB_CUDA(cudaMalloc(&sh.rows16[g], (size_t)rows_bytes));
      JOB_CUDA(cudaMalloc(&sh.valid[g], (size_t)valid_bytes));
      JOB_CUDA(cudaMalloc(&staging, (size_t)rows_bytes * G));
      JOB_CUDA(cudaMalloc(&staging_v, (size_t)valid_bytes * G));
      if (OK_SO_FAR) JOB_TRY(mb200_bank_normalize(bank, P.dtype, sh.rows16[g], (uint32_t*)sh.valid[g]));
      if (OK_SO_FAR && P.precision != MB200_PRECISION_TENSOR) JOB_TRY(mb200_bank_sign_info(bank, &sh.mixed[g]));
      int64_t got_cells = 0;
      if (OK_SO_FAR) JOB_TRY(mb200_bank_counters(bank, &sh.counters[g], &got_cells));
      if (OK_SO_FAR && P.precision == MB200_PRECISION_CERTIFIED) {
        JOB_CUDA(cudaMalloc(&sh.n32[g], (size_t)cells * 4));
        if (OK_SO_FAR) JOB_TRY(mb200_bank_narrow32(bank, (int32_t*)sh.n32[g]));
      }
      if (OK_SO_FAR) JOB_TRY(mb200_sync(ctx));
    }
    sh.bar.wait();  // every GPU's rows and counters are final
    if (!sh.failed()) {
      int mixed = 0;
      for (int s = 0; s < G; s++) mixed |= sh.mixed[s];
      if (P.precision == MB200_PRECISION_RESCORED) {
        // the exact re-score reads arbitrary peers' counters: pulled whole (G x the shard) -- fine at the sizes
        // where bit-equal similarities are asked for; CERTIFIED reads only the undecided candidates remotely
        JOB_CUDA(cudaMalloc(&sh.gathered[g], (size_t)cells * 8 * G));
        for (int s = 0; s < G && OK_SO_FAR; s++)
          JOB_CUDA(cudaMemcpyAsync((char*)sh.gathered[g] + (size_t)s * cells * 8, sh.counters[s], (size_t)cells * 8,
                                   cudaMemcpyDeviceToDevice, ctx->stream));
      }
      const uint32_t* flags = nullptr;
      uint32_t epoch = 0;
      if (OK_SO_FAR)
        JOB_TRY(mb200_gather_pull(ctx, staging, (uint32_t*)staging_v, sh.rows16.data(), (const uint32_t* const*)sh.valid.data(),
                                  G, g, rows_bytes, valid_bytes, &flags, &epoch));
      mb200_cosine_args a;
      memset(&a, 0, sizeof(a));
      a.a_rows = sh.rows16[g];
      a.a_valid = (const uint32_t*)sh.valid[g];
      a.a_count = E;
      a.a_id_mul = G;
      a.a_id_off = g;
      a.depth = P.depth;
      a.width = P.width;
      a.dtype = P.dtype;
      a.precision = P.precision;
      a.k = k;
      a.threshold = P.threshold;
      a.exclude_self = 1;
      a.mixed_sign = mixed;
      // Attempt 0: K3 starts at once and waits block by block on the arrival flags.  If a pull has not landed when
      // K3 gives up (~4 s: MB200_ERR_PULL_TIMEOUT from finish), attempt 1 waits for the copy stream and sweeps the fully
      // staged operand without flags -- a local decision: the peers' rows and counters stay alive until the barrier
      // below, so no other worker needs to know.
      for (int attempt = 0; attempt < 2 && OK_SO_FAR; attempt++) {
        if (attempt == 1) JOB_TRY(mb200_gather_wait(ctx));
        mb200_cosine_job* job = nullptr;
        int rc = mb200_cosine_begin(ctx, &a, &job);
        if (rc == MB200_OK) {
          mb200_cosine_piece pc;
          memset(&pc, 0, sizeof(pc));
          pc.b_rows = staging;
          pc.b_valid = (const uint32_t*)staging_v;
          pc.b_count = E;
          pc.b_blocks = G;
          pc.b_id_mul = G;
          pc.b_id_add = 1;
          pc.ready_flags = attempt == 0 ? flags : nullptr;
          pc.ready_epoch = attempt == 0 ? epoch : 0;
          pc.first_block = g;
          rc = mb200_cosine_push(job, &pc);
          mb200_cosine_args fin;
          memset(&fin, 0, sizeof(fin));
          fin.out_idx = (int64_t*)o_idx;
          fin.out_sim = (double*)o_sim;
          fin.out_cnt = (int32_t*)o_cnt;
          fin.b_rows = staging;  // still resident: uncertified rows may take the band pass
          fin.b_valid = (const uint32_t*)staging_v;
          if (P.precision != MB200_PRECISION_TENSOR) {
            fin.a_counters = (const int64_t*)sh.counters[g];
            fin.b_blocks = G;
            fin.b_count = E;
            fin.b_id_mul = G;
            fin.b_id_add = 1;
            if (P.precision == MB200_PRECISION_CERTIFIED) {
              fin.b_counter_blocks = (const int64_t* const*)sh.counters.data();
              fin.b_counter_blocks32 = (const int32_t* const*)sh.n32.data();
            } else {
              fin.b_counters = (const int64_t*)sh.gathered[g];
            }
          }
          if (rc == MB200_OK) rc = mb200_cosine_finish(job, &fin);
          else mb200_cosine_abort(job);
        }
        const bool lost_block = rc == MB200_ERR_PULL_TIMEOUT && attempt == 0;
        if (lost_block) {
          sh.pull_retries[g] = 1;
          continue;
        }
        JOB_TRY(rc);
        if (OK_SO_FAR) JOB_TRY(mb200_cosine_last_fallback_rows(ctx, &sh.fallback[g]));
        break;
      }
      JOB_TRY(mb200_sync(ctx));
      mb200_gather_wait(ctx);
    }
    sh.bar.wait();  // nobody reads my rows / counters any more
    cudaFree(staging);
    cudaFree(staging_v);
    cudaFree(sh.rows16[g]);
    cudaFree(sh.valid[g]);
    cudaFree(sh.n32[g]);
    cudaFree(sh.gathered[g]);
  }
  // ---- results: local row l of shard g is global row l * G + g
  if (!sh.failed()) {
    const int64_t mine = sh.num_items > g ? (sh.num_items - g + G - 1) / G : 0;
    std::vector<int64_t> h_idx((size_t)E * k);
    std::vector<double> h_sim((size_t)E * k);
    std::vector<int32_t> h_cnt((size_t)E);
    JOB_CUDA(cudaMemcpyAsync(h_idx.data(), o_idx, (size_t)E * k * 8, cudaMemcpyDeviceToHost, ctx->stream));
    JOB_CUDA(cudaMemcpyAsync(h_sim.data(), o_sim, (size_t)E * k * 8, cudaMemcpyDeviceToHost, ctx->stream));
    JOB_CUDA(cudaMemcpyAsync(h_cnt.data(), o_cnt, (size_t)E * 4, cudaMemcpyDeviceToHost, ctx->stream));
    JOB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int64_t l = 0; l < mine && OK_SO_FAR; l++) {
      const int64_t r = l * G + g;
      memcpy(sh.out_idx + r * k, h_idx.data() + l * k, (size_t)k * 8);
      memcpy(sh.out_sim + r * k, h_sim.data() + l * k, (size_t)k * 8);
      sh.out_cnt[r] = h_cnt[(size_t)l];
    }
  }
  cudaFree(o_idx);
  cudaFree(o_sim);
  cudaFree(o_cnt);
  if (bank) mb200_bank_destroy(bank);
  mb200_release_workspace(ctx);
  sh.bar.wait();
  if (g == 0) sh.t_cosine = multi_now_s() - t2;
}

}  // namespace

extern "C" {

int mb200_create_multi(int32_t n_gpus, const int32_t* devices, mb200_multi** out) {
  if (!out) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_create_multi: out is NULL");
  *out = nullptr;
  int have = 0;
  cudaError_t e = cudaGetDeviceCount(&have);
  if (e != cudaSuccess || have <= 0)
    return mb200_fail(nullptr, MB200_ERR_NO_DEVICE, "mb200_create_multi: no CUDA device (%s); this library has no CPU fallback",
                      e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (n_gpus == 0) n_gpus = have;  // all GPUs of the box
  // an explicit list may name a device more than once (several contexts on it); without one, GPUs 0 .. n_gpus-1
  if (n_gpus < 0 || (!devices && n_gpus > have) || n_gpus > MB200_MAX_BLOCKS)
    return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_create_multi: %d GPUs asked for, %d visible", n_gpus, have);
  for (int g = 0; devices && g < n_gpus; g++)
    if (devices[g] < 0 || devices[g] >= have)
      return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_create_multi: device %d out of range [0, %d)", devices[g], have);
  mb200_multi* m = new mb200_multi();
  m->n = n_gpus;
  for (int g = 0; g < n_gpus; g++) m->devices.push_back(devices ? devices[g] : g);
  for (int g = 0; g < n_gpus; g++) {
    mb200_ctx* c = nullptr;
    int rc = mb200_create(m->devices[g], &c);
    if (rc != MB200_OK) {
      for (auto* x : m->ctx) mb200_destroy(x);
      delete m;
      return rc;
    }
    m->ctx.push_back(c);
  }
  // one process: the GPUs map each other's memory directly (NVLink / NVSwitch)
  for (int a = 0; a < n_gpus; a++) {
    cudaSetDevice(m->devices[a]);
    for (int b = 0; b < n_gpus; b++) {
      if (m->devices[a] == m->devices[b]) continue;  // a device listed twice reaches its own memory
      int can = 0;
      cudaDeviceCanAccessPeer(&can, m->devices[a], m->devices[b]);
      if (!can) {
        for (auto* x : m->ctx) mb200_destroy(x);
        delete m;
        return mb200_fail(nullptr, MB200_ERR_UNSUPPORTED, "mb200_create_multi: device %d cannot access device %d's memory",
                          m->devices[a], m->devices[b]);
      }
      cudaError_t pe = cudaDeviceEnablePeerAccess(m->devices[b], 0);
      if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) {
        for (auto* x : m->ctx) mb200_destroy(x);
        delete m;
        return mb200_fail(nullptr, MB200_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", m->devices[a], m->devices[b],
                          cudaGetErrorString(pe));
      }
      cudaGetLastError();
    }
  }
  *out = m;
  return MB200_OK;
}

int mb200_multi_destroy(mb200_multi* m) {
  if (!m) return MB200_OK;
  for (auto* c : m->ctx) mb200_destroy(c);
  delete m;
  return MB200_OK;
}

int mb200_multi_gpus(mb200_multi* m, int32_t* n_gpus) {
  if (!m || !n_gpus) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_multi_gpus: NULL argument");
  *n_gpus = m->n;
  return MB200_OK;
}

int mb200_multi_ctx(mb200_multi* m, int32_t g, mb200_ctx** out) {
  if (!m || !out || g < 0 || g >= m->n) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_multi_ctx: bad arguments");
  *out = m->ctx[g];
  return MB200_OK;
}

const char* mb200_multi_last_error(mb200_multi* m) { return m && !m->err.empty() ? m->err.c_str() : mb200_last_error(nullptr); }

int mb200_job_item_similarity(mb200_multi* m, const int64_t* row, const int64_t* key, const float* inc, int64_t n,
                              int64_t num_items, const mb200_job_params* p, int64_t* out_idx, double* out_sim,
                              int32_t* out_cnt, mb200_job_stats* stats) {
  if (!m) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_job_item_similarity: handle is NULL");
  std::lock_guard<std::mutex> lock(m->mu);
  if (!p || n < 0 || num_items <= 0 || (n > 0 && (!row || !key || !inc)) || !out_idx || !out_sim || !out_cnt)
    return multi_fail(m, MB200_ERR_BAD_ARG, "mb200_job_item_similarity: bad arguments");
  if (p->k <= 0 || p->depth <= 0 || p->depth > MB200_MAX_DEPTH || p->width <= 0)
    return multi_fail(m, MB200_ERR_BAD_ARG, "mb200_job_item_similarity: need k > 0, 0 < depth <= 32, width > 0");
  if (p->precision != MB200_PRECISION_TENSOR && p->precision != MB200_PRECISION_RESCORED &&
      p->precision != MB200_PRECISION_CERTIFIED)
    return multi_fail(m, MB200_ERR_BAD_ARG, "mb200_job_item_similarity: unknown precision");
  const int G = m->n;
  Shared sh(G);
  sh.m = m;
  sh.p = p;
  sh.row = row;
  sh.key = key;
  sh.inc = inc;
  sh.n = n;
  sh.num_items = num_items;
  sh.E_loc = (num_items + G - 1) / G;
  sh.G = G;
  sh.counts.resize(G);
  for (auto* v : {&sh.r_row, &sh.r_key, &sh.r_inc, &sh.rows16, &sh.valid, &sh.counters, &sh.n32, &sh.gathered}) v->assign(G, nullptr);
  sh.recv.assign(G, 0);
  sh.rc.assign(G, MB200_OK);
  sh.msg.assign(G, "");
  sh.fallback.assign(G, 0);
  sh.pull_retries.assign(G, 0);
  sh.mixed.assign(G, 0);
  sh.out_idx = out_idx;
  sh.out_sim = out_sim;
  sh.out_cnt = out_cnt;
  for (int64_t r = 0; r < num_items; r++) out_cnt[r] = 0;
  std::vector<std::thread> th;
  for (int g = 1; g < G; g++) th.emplace_back(worker, std::ref(sh), g);
  worker(sh, 0);
  for (auto& t : th) t.join();
  for (int g = 0; g < G; g++)
    if (sh.rc[g] != MB200_OK) return multi_fail(m, sh.rc[g], "GPU " + std::to_string(m->devices[g]) + ": " + sh.msg[g]);
  for (int g = 0; g < G; g++)
    if (sh.pull_retries[g])
      fprintf(stderr, "mb200_job_item_similarity: GPU %d repeated its cosine phase over the fully staged operand "
                      "(a peer block had not arrived within K3's time-out)\n", m->devices[g]);
  if (stats) {
    memset(stats, 0, sizeof(*stats));
    stats->n_gpus = G;
    stats->events = n;
    stats->rows = num_items;
    for (int g = 0; g < G; g++) {
      stats->fallback_rows += sh.fallback[g];
      if (sh.recv[g] > stats->events_busiest_gpu) stats->events_busiest_gpu = sh.recv[g];
    }
    for (int64_t r = 0; r < num_items; r++) stats->similarities_kept += out_cnt[r];
    stats->route_s = sh.t_route;
    stats->build_s = sh.t_build;
    stats->cosine_s = sh.t_cosine;
  }
  return MB200_OK;
}

}  // extern "C"
