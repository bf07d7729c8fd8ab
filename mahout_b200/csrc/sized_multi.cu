// sized_multi.cu -- CosineCM with a CountMinSketchConfig on all GPUs of the process: one replica of the sized bank
// per GPU of an mb200_multi, the query users split between them.  Host code only: the kernels are cmsized.cu's.
//
// A neighbourhood, an estimate or a recommendation of the sized calls depends only on its user, the bank and the
// call's parameters, so the calls split by user with no traffic between GPUs:
//
//   create     one worker thread per GPU builds that GPU's mb200_sized_bank from the caller's host arrays
//   split      query position t goes to GPU t mod G; estimates go by user: the j-th distinct user row (ascending)
//              to GPU j mod G, with every pair of that user, so each distinct user's neighbourhood is computed once
//   run        each worker copies its share in (H2D), runs the single-context calls on device memory -- the
//              neighbourhood lists of recommend and estimates never leave the GPU -- and copies its results out
//              (D2H); the host scatters them to the caller's positions
//
// The results are the single-context calls' bit for bit for any G: the same kernels on the same bank, each query
// row computed on its own.  The workers share nothing, so there are no barriers: every worker runs its part to the
// end (or to its first failure) and the call joins them.  Host-side argument errors fail with MB200_ERR_BAD_ARG
// before any GPU work; a GPU's failure fails the call with the first failing GPU's code and "GPU d: <message>".
#include <string.h>

#include <algorithm>

#include "multi.cuh"

struct mb200_sized_multi {
  mb200_multi* m = nullptr;
  int64_t U = 0;
  std::vector<mb200_sized_bank*> bank;  // bank[g] lives on m->ctx[g]
  MultiStats st;                        // last call: queries (pairs for estimates, users for create) per GPU
};

namespace {

constexpr int NB_MAX_N = 1024;   // mb200_sized_neighborhood's n
constexpr int REC_MAX_HOW = 1024;  // mb200_sized_recommend's how_many

// GPU g's share of the query rows, its neighbourhood lists on the device ([mine][n], as mb200_sized_neighborhood
// returns them)
struct Lists {
  int64_t* rows = nullptr;
  int64_t* idx = nullptr;
  double* sim = nullptr;
  int32_t* cnt = nullptr;
};

Lists device_lists(Part& p, mb200_sized_bank* bank, const std::vector<int64_t>& rows, int32_t n, double min_similarity) {
  Lists L;
  const size_t q = rows.size();
  L.rows = p.upload(rows.data(), q);
  L.idx = p.alloc<int64_t>(q * n);
  L.sim = p.alloc<double>(q * n);
  L.cnt = p.alloc<int32_t>(q);
  if (p.ok())
    p.take(mb200_sized_neighborhood(bank, L.rows, (int64_t)q, n, min_similarity, L.idx, L.sim, L.cnt, MB200_MEM_DEVICE));
  return L;
}

}  // namespace

extern "C" {

int mb200_sized_multi_create(mb200_multi* m, int64_t users, const int32_t* width, const int32_t* depth,
                             const int64_t* a, const int64_t* b, int32_t frac_bits, const int64_t* user_ptr,
                             const int64_t* item, const float* pref, mb200_sized_multi** out) {
  if (!m) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_multi_create: handle is NULL");
  std::lock_guard<std::mutex> lock(m->mu);
  if (!out) return multi_bad_arg(m, "mb200_sized_multi_create: out is NULL");
  *out = nullptr;
  if (users < 0 || !a || !b || !user_ptr || (users > 0 && (!width || !depth)))
    return multi_bad_arg(m, "mb200_sized_multi_create: bad shape (users=%lld) or NULL array argument", (long long)users);
  mb200_sized_multi* sm = new mb200_sized_multi();
  sm->m = m;
  sm->U = users;
  sm->bank.assign(m->n, nullptr);
  const int rc = run_parts(sm->m, sm->st, [&](int g, Part& p) {
    sm->st.work[g] = users;
    p.take(mb200_sized_bank_create(p.ctx, users, width, depth, a, b, frac_bits, user_ptr, item, pref, MB200_MEM_HOST,
                                   &sm->bank[g]));
  });
  if (rc != MB200_OK) {
    for (auto* bk : sm->bank) mb200_sized_bank_destroy(bk);
    delete sm;
    return rc;
  }
  *out = sm;
  return MB200_OK;
}

int mb200_sized_multi_destroy(mb200_sized_multi* sm) {
  if (!sm) return MB200_OK;
  {
    std::lock_guard<std::mutex> lock(sm->m->mu);
    for (auto* bk : sm->bank) mb200_sized_bank_destroy(bk);
  }
  delete sm;
  return MB200_OK;
}

int mb200_sized_multi_neighborhood(mb200_sized_multi* sm, const int64_t* query_rows, int64_t q, int32_t n,
                                   double min_similarity, int64_t* out_idx, double* out_sim, int32_t* out_cnt) {
  if (!sm) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_multi_neighborhood: handle is NULL");
  mb200_multi* m = sm->m;
  std::lock_guard<std::mutex> lock(m->mu);
  if (n < 1 || n > NB_MAX_N)
    return multi_bad_arg(m, "mb200_sized_multi_neighborhood: n must be in [1, %d] (got %d)", NB_MAX_N, n);
  if (q < 0 || min_similarity != min_similarity)
    return multi_bad_arg(m, "mb200_sized_multi_neighborhood: bad shape (q=%lld) or NaN min_similarity", (long long)q);
  if (q > 0 && (!query_rows || !out_idx || !out_sim || !out_cnt))
    return multi_bad_arg(m, "mb200_sized_multi_neighborhood: NULL array argument");
  const int G = m->n;
  return run_parts(sm->m, sm->st, [&](int g, Part& p) {
    const std::vector<int64_t> rows = multi_gather(query_rows, q, g, G);
    const int64_t mine = (int64_t)rows.size();
    sm->st.work[g] = mine;
    if (!mine) return;
    Lists L = device_lists(p, sm->bank[g], rows, n, min_similarity);
    std::vector<int64_t> hi;
    std::vector<double> hs;
    std::vector<int32_t> hc;
    p.download(hi, L.idx, (size_t)mine * n);
    p.download(hs, L.sim, (size_t)mine * n);
    p.download(hc, L.cnt, (size_t)mine);
    p.finish();
    if (!p.ok()) return;
    for (int64_t l = 0; l < mine; l++) {
      const int64_t t = l * G + g;
      memcpy(out_idx + t * n, hi.data() + l * n, (size_t)n * 8);
      memcpy(out_sim + t * n, hs.data() + l * n, (size_t)n * 8);
      out_cnt[t] = hc[(size_t)l];
    }
  });
}

int mb200_sized_multi_recommend(mb200_sized_multi* sm, const int64_t* users, int64_t m_users, int32_t n,
                                double min_similarity, const int64_t* item_ptr, const int32_t* item_col, int64_t nnz,
                                const int64_t* item_ids, int64_t num_items, int32_t how_many, int include_known,
                                int64_t* out_item, float* out_value, int32_t* out_cnt) {
  if (!sm) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_multi_recommend: handle is NULL");
  mb200_multi* m = sm->m;
  std::lock_guard<std::mutex> lock(m->mu);
  if (n < 1 || n > NB_MAX_N) return multi_bad_arg(m, "mb200_sized_multi_recommend: n must be in [1, %d] (got %d)", NB_MAX_N, n);
  if (how_many < 1 || how_many > REC_MAX_HOW)
    return multi_bad_arg(m, "mb200_sized_multi_recommend: how_many must be in [1, %d] (got %d)", REC_MAX_HOW, how_many);
  if (m_users < 0 || nnz < 0 || num_items < 0 || num_items >= (1LL << 31) || min_similarity != min_similarity)
    return multi_bad_arg(m, "mb200_sized_multi_recommend: bad shape (m=%lld nnz=%lld num_items=%lld) or NaN min_similarity",
                   (long long)m_users, (long long)nnz, (long long)num_items);
  if (m_users > 0 && (!users || !item_ptr || (nnz > 0 && !item_col) || (num_items > 0 && !item_ids) || !out_item ||
                      !out_value || !out_cnt))
    return multi_bad_arg(m, "mb200_sized_multi_recommend: NULL array argument");
  if (m_users == 0) return run_parts(sm->m, sm->st, [](int, Part&) {});  // the stats of an empty call
  const int64_t U = sm->U;
  // the data model is host memory: its shape is checked here, as mb200_sized_recommend checks host arguments
  if (item_ptr[0] != 0 || item_ptr[U] != nnz)
    return multi_bad_arg(m, "mb200_sized_multi_recommend: item_ptr[0] must be 0 and item_ptr[users] = nnz (%lld)", (long long)nnz);
  for (int64_t t = 1; t < num_items; t++)
    if (item_ids[t] <= item_ids[t - 1]) return multi_bad_arg(m, "mb200_sized_multi_recommend: item_ids must be strictly ascending");
  const int G = m->n;
  return run_parts(sm->m, sm->st, [&](int g, Part& p) {
    const std::vector<int64_t> rows = multi_gather(users, m_users, g, G);
    const int64_t mine = (int64_t)rows.size();
    sm->st.work[g] = mine;
    if (!mine) return;
    Lists L = device_lists(p, sm->bank[g], rows, n, min_similarity);
    const int64_t* d_ptr = p.upload(item_ptr, (size_t)U + 1);
    const int32_t* d_col = p.upload(item_col, (size_t)nnz);
    const int64_t* d_ids = p.upload(item_ids, (size_t)num_items);
    int64_t* d_item = p.alloc<int64_t>((size_t)mine * how_many);
    float* d_value = p.alloc<float>((size_t)mine * how_many);
    int32_t* d_cnt = p.alloc<int32_t>((size_t)mine);
    if (p.ok())
      p.take(mb200_sized_recommend(sm->bank[g], L.idx, L.sim, L.cnt, n, d_ptr, d_col, nnz, d_ids, num_items, L.rows, mine,
                                   how_many, include_known, d_item, d_value, d_cnt, MB200_MEM_DEVICE));
    std::vector<int64_t> hi;
    std::vector<float> hv;
    std::vector<int32_t> hc;
    p.download(hi, d_item, (size_t)mine * how_many);
    p.download(hv, d_value, (size_t)mine * how_many);
    p.download(hc, d_cnt, (size_t)mine);
    p.finish();
    if (!p.ok()) return;
    for (int64_t l = 0; l < mine; l++) {
      const int64_t t = l * G + g;
      memcpy(out_item + t * how_many, hi.data() + l * how_many, (size_t)how_many * 8);
      memcpy(out_value + t * how_many, hv.data() + l * how_many, (size_t)how_many * 4);
      out_cnt[t] = hc[(size_t)l];
    }
  });
}

int mb200_sized_multi_estimate_prefs(mb200_sized_multi* sm, const int64_t* user, const int64_t* item_id, int64_t q,
                                     int32_t n, double min_similarity, float* out) {
  if (!sm) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_multi_estimate_prefs: handle is NULL");
  mb200_multi* m = sm->m;
  std::lock_guard<std::mutex> lock(m->mu);
  if (n < 1 || n > NB_MAX_N)
    return multi_bad_arg(m, "mb200_sized_multi_estimate_prefs: n must be in [1, %d] (got %d)", NB_MAX_N, n);
  if (q < 0 || min_similarity != min_similarity)
    return multi_bad_arg(m, "mb200_sized_multi_estimate_prefs: bad shape (q=%lld) or NaN min_similarity", (long long)q);
  if (q > 0 && (!user || !item_id || !out)) return multi_bad_arg(m, "mb200_sized_multi_estimate_prefs: NULL array argument");
  const int G = m->n;
  // distinct user rows, ascending: the j-th goes to GPU j mod G as row j / G of that GPU's lists
  std::vector<int64_t> uniq(user, user + q);
  std::sort(uniq.begin(), uniq.end());
  uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
  std::vector<std::vector<int64_t>> pos(G), nb_row(G);  // per GPU: the caller's pair positions, their list rows
  for (int64_t t = 0; t < q; t++) {
    const int64_t j = std::lower_bound(uniq.begin(), uniq.end(), user[t]) - uniq.begin();
    pos[j % G].push_back(t);
    nb_row[j % G].push_back(j / G);
  }
  return run_parts(sm->m, sm->st, [&](int g, Part& p) {
    const int64_t pairs = (int64_t)pos[g].size();
    sm->st.work[g] = pairs;
    if (!pairs) return;
    const std::vector<int64_t> rows = multi_gather(uniq.data(), (int64_t)uniq.size(), g, G);
    Lists L = device_lists(p, sm->bank[g], rows, n, min_similarity);
    std::vector<int64_t> pu((size_t)pairs), pi((size_t)pairs);
    for (int64_t l = 0; l < pairs; l++) {
      pu[(size_t)l] = user[pos[g][(size_t)l]];
      pi[(size_t)l] = item_id[pos[g][(size_t)l]];
    }
    const int64_t* d_user = p.upload(pu.data(), (size_t)pairs);
    const int64_t* d_row = p.upload(nb_row[g].data(), (size_t)pairs);
    const int64_t* d_item = p.upload(pi.data(), (size_t)pairs);
    float* d_out = p.alloc<float>((size_t)pairs);
    if (p.ok())
      p.take(mb200_sized_estimate_prefs(sm->bank[g], L.idx, L.sim, L.cnt, (int64_t)rows.size(), n, d_user, d_row,
                                        d_item, pairs, d_out, MB200_MEM_DEVICE));
    std::vector<float> h;
    p.download(h, d_out, (size_t)pairs);
    p.finish();
    if (!p.ok()) return;
    for (int64_t l = 0; l < pairs; l++) out[pos[g][(size_t)l]] = h[(size_t)l];
  });
}

int mb200_sized_multi_last_stats(mb200_sized_multi* sm, int64_t* work, double* seconds, double* wall_s) {
  if (!sm) return mb200_fail(nullptr, MB200_ERR_BAD_ARG, "mb200_sized_multi_last_stats: handle is NULL");
  std::lock_guard<std::mutex> lock(sm->m->mu);
  multi_last_stats(sm->st, work, seconds, wall_s);
  return MB200_OK;
}

}  // extern "C"
