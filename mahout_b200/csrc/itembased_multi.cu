// itembased_multi.cu -- item-based recommendation (RecommenderJob's aggregate-and-recommend phase) on all GPUs of an
// mb200_multi: one replica of the item top-k lists, the user CSR and the itemIDs per GPU, the query users split
// between them.  Host code only: the kernels are recommend.cu's k_itembased and the itemID rank table kernels.
//
// One user's recommendations depend only on that user's vector, the lists and the call's parameters, so the call
// splits by user with no traffic between GPUs:
//
//   create     one worker thread per GPU copies the caller's host arrays to that GPU once (I * ld * 16 B of lists,
//              12 B per item, 8 B per pref, 8 B per user); the replicas live until destroy
//   split      query position t goes to GPU t mod G
//   run        each worker hands its share of the users, the allowed mask and its output slots to the single-context
//              call on its replica (mb200_itembased_call with the data on the device): the context stages them in
//              its grow-only buffers, so a repeated call of the same or a smaller shape allocates nothing; the host
//              scatters the results to the caller's positions
//
// Every user row is computed by the same kernel on the same data whatever its neighbours in the launch, so the
// results are the single-context call's byte for byte for any G.  Host-side argument errors fail with
// MB200_ERR_BAD_ARG before any GPU work; a GPU's failure fails the call with the first failing GPU's code and
// "GPU d: <message>".
#include <string.h>

#include "multi.cuh"

namespace {

constexpr int IB_MAX_HOW = 1024;  // mb200_recommend_item_based's how_many

// one GPU's copy of the call-independent arrays, in one allocation
struct Replica {
  int device = 0;
  void* base = nullptr;
  const int64_t* sim_idx = nullptr;
  const double* sim_val = nullptr;
  const int32_t* sim_cnt = nullptr;
  const int64_t* user_ptr = nullptr;
  const int32_t* pref_row = nullptr;
  const float* pref_val = nullptr;
  const int64_t* item_ids = nullptr;
};

void release(Replica& r) {
  if (!r.base) return;
  cudaSetDevice(r.device);
  cudaFree(r.base);
  r.base = nullptr;
}

}  // namespace

struct mb200_itembased_multi {
  mb200_multi* m = nullptr;
  int64_t num_items = 0, num_users = 0, nnz = 0;
  int32_t sim_ld = 1;
  std::vector<Replica> rep;  // rep[g] lives on m->ctx[g]'s device
  MultiStats st;             // last call: users per GPU (every user for create)
};

extern "C" {

int mb200_itembased_multi_create(mb200_multi* m, const int64_t* sim_idx, const double* sim_val, const int32_t* sim_cnt,
                                 int64_t num_items, int32_t sim_ld, const int64_t* user_ptr, const int32_t* pref_row,
                                 const float* pref_val, int64_t num_users, int64_t nnz, const int64_t* item_ids,
                                 mb200_itembased_multi** out) {
  if (!m) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_itembased_multi_create: handle is NULL");
  std::lock_guard<std::mutex> lock(m->mu);
  if (!out) return multi_bad_arg(m, "mb200_itembased_multi_create: out is NULL");
  *out = nullptr;
  if (sim_ld < 1 || num_items < 0 || num_items >= (1LL << 31) || num_users < 0 || nnz < 0)
    return multi_bad_arg(m, "mb200_itembased_multi_create: bad shape (sim_ld=%d num_items=%lld num_users=%lld nnz=%lld)",
                         sim_ld, (long long)num_items, (long long)num_users, (long long)nnz);
  if (!user_ptr || (num_items > 0 && (!sim_idx || !sim_val || !sim_cnt || !item_ids)) ||
      (nnz > 0 && (!pref_row || !pref_val)))
    return multi_bad_arg(m, "mb200_itembased_multi_create: NULL array argument");
  mb200_itembased_multi* h = new mb200_itembased_multi();
  h->m = m;
  h->num_items = num_items;
  h->num_users = num_users;
  h->nnz = nnz;
  h->sim_ld = sim_ld;
  h->rep.assign(m->n, Replica());
  // byte offsets of the arrays in a replica, each 256-byte aligned
  const size_t lists = (size_t)num_items * sim_ld;
  const size_t bytes[7] = {lists * 8, lists * 8, (size_t)num_items * 4, ((size_t)num_users + 1) * 8,
                           (size_t)nnz * 4, (size_t)nnz * 4, (size_t)num_items * 8};
  const void* src[7] = {sim_idx, sim_val, sim_cnt, user_ptr, pref_row, pref_val, item_ids};
  size_t off[7], total = 0;
  for (int i = 0; i < 7; i++) {
    off[i] = total;
    total += (bytes[i] + 255) / 256 * 256;
  }
  const int rc = run_parts(m, h->st, [&](int g, Part& p) {
    h->st.work[g] = num_users;
    Replica& r = h->rep[g];
    r.device = p.ctx->device;
    p.cuda(cudaMalloc(&r.base, total ? total : 1), "cudaMalloc");
    if (!p.ok()) return;
    char* b = (char*)r.base;
    for (int i = 0; i < 7; i++)
      if (p.ok() && bytes[i])
        p.cuda(cudaMemcpyAsync(b + off[i], src[i], bytes[i], cudaMemcpyHostToDevice, p.ctx->stream), "cudaMemcpyAsync H2D");
    p.finish();
    r.sim_idx = (const int64_t*)(b + off[0]);
    r.sim_val = (const double*)(b + off[1]);
    r.sim_cnt = (const int32_t*)(b + off[2]);
    r.user_ptr = (const int64_t*)(b + off[3]);
    r.pref_row = (const int32_t*)(b + off[4]);
    r.pref_val = (const float*)(b + off[5]);
    r.item_ids = (const int64_t*)(b + off[6]);
  });
  if (rc != MB200_OK) {
    for (auto& r : h->rep) release(r);
    delete h;
    return rc;
  }
  *out = h;
  return MB200_OK;
}

int mb200_itembased_multi_destroy(mb200_itembased_multi* h) {
  if (!h) return MB200_OK;
  {
    std::lock_guard<std::mutex> lock(h->m->mu);
    int caller_device = 0;
    cudaGetDevice(&caller_device);
    for (auto& r : h->rep) release(r);
    cudaSetDevice(caller_device);
  }
  delete h;
  return MB200_OK;
}

int mb200_itembased_multi_recommend(mb200_itembased_multi* h, const int64_t* users, int64_t m_users, int32_t how_many,
                                    int32_t max_prefs_per_user, int32_t boolean_data, const uint32_t* allowed,
                                    int64_t* out_item, float* out_value, int32_t* out_cnt) {
  if (!h) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_itembased_multi_recommend: handle is NULL");
  mb200_multi* m = h->m;
  std::lock_guard<std::mutex> lock(m->mu);
  if (how_many < 1 || how_many > IB_MAX_HOW)
    return multi_bad_arg(m, "mb200_itembased_multi_recommend: how_many must be in [1, %d] (got %d)", IB_MAX_HOW, how_many);
  if (max_prefs_per_user < 1)
    return multi_bad_arg(m, "mb200_itembased_multi_recommend: max_prefs_per_user must be >= 1 (got %d)",
                         max_prefs_per_user);
  if (m_users < 0) return multi_bad_arg(m, "mb200_itembased_multi_recommend: bad shape (m=%lld)", (long long)m_users);
  if (m_users > 0 && (!users || !out_item || !out_value || !out_cnt))
    return multi_bad_arg(m, "mb200_itembased_multi_recommend: NULL array argument");
  const int G = m->n;
  return run_parts(m, h->st, [&](int g, Part& p) {
    const std::vector<int64_t> rows = multi_gather(users, m_users, g, G);
    const int64_t mine = (int64_t)rows.size();
    h->st.work[g] = mine;
    if (!mine) return;
    std::vector<int64_t> hi((size_t)mine * how_many);
    std::vector<float> hv((size_t)mine * how_many);
    std::vector<int32_t> hc((size_t)mine);
    const Replica& r = h->rep[g];
    mb200_itembased_args a;
    memset(&a, 0, sizeof(a));
    a.sim_idx = r.sim_idx;
    a.sim_val = r.sim_val;
    a.sim_cnt = r.sim_cnt;
    a.num_items = h->num_items;
    a.sim_ld = h->sim_ld;
    a.user_ptr = r.user_ptr;
    a.pref_row = r.pref_row;
    a.pref_val = r.pref_val;
    a.num_users = h->num_users;
    a.nnz = h->nnz;
    a.item_ids = r.item_ids;
    a.allowed = allowed;
    a.users = rows.data();
    a.m = mine;
    a.how_many = how_many;
    a.max_prefs_per_user = max_prefs_per_user;
    a.boolean_data = boolean_data;
    a.out_item = hi.data();
    a.out_value = hv.data();
    a.out_cnt = hc.data();
    a.mem = MB200_MEM_HOST;  // the share and the results: staged by the context
    p.take(mb200_itembased_call(p.ctx, &a, true));
    if (!p.ok()) return;
    for (int64_t l = 0; l < mine; l++) {
      const int64_t t = l * G + g;
      memcpy(out_item + t * how_many, hi.data() + l * how_many, (size_t)how_many * 8);
      memcpy(out_value + t * how_many, hv.data() + l * how_many, (size_t)how_many * 4);
      out_cnt[t] = hc[(size_t)l];
    }
  });
}

int mb200_itembased_multi_last_stats(mb200_itembased_multi* h, int64_t* work, double* seconds, double* wall_s) {
  if (!h) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_itembased_multi_last_stats: handle is NULL");
  std::lock_guard<std::mutex> lock(h->m->mu);
  multi_last_stats(h->st, work, seconds, wall_s);
  return MB200_OK;
}

}  // extern "C"
