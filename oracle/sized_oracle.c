/*
 * sized_oracle.c -- CPU ORACLE (test infrastructure, NOT the product) of CosineCM with a CountMinSketchConfig.
 *
 * User u's sketch has its own (width[u], depth[u]); the prefs of user row u are [user_ptr[u], user_ptr[u+1]), given
 * as the doubles CosineCM.exportProfile adds (CosineCM.java:41-58).  Everything is built per pair from the per-sketch
 * primitives of mahout_oracle.c (orc_cm_update, orc_cm_cosine, orc_clamp_similarity, orc_cm_get), which this library
 * links against (oracle/sized.py builds it next to libmahout_oracle.so).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* mahout_oracle.c */
void orc_cm_update(double *count, int32_t w, int32_t d, const int64_t *a, const int64_t *b, const int64_t *keys,
                   const double *incs, int64_t n);
double orc_cm_get(const double *count, int32_t w, int32_t d, const int64_t *a, const int64_t *b, int64_t key);
double orc_cm_cosine(const double *ca, const double *cb, int32_t w, int32_t d);
double orc_clamp_similarity(double r);

/* the sketch CosineCM.exportProfile builds for user u at (w, d) */
static double *sized_profile(int64_t u, int32_t w, int32_t d, const int64_t *a, const int64_t *b,
                             const int64_t *user_ptr, const int64_t *item, const double *pref) {
  double *c = (double *)calloc((size_t)w * (size_t)d, sizeof(double));
  orc_cm_update(c, w, d, a, b, item + user_ptr[u], pref + user_ptr[u], user_ptr[u + 1] - user_ptr[u]);
  return c;
}

/* every user's own sketch: getExportedCMProfile(u) */
static double **sized_own(int64_t U, const int32_t *width, const int32_t *depth, const int64_t *a, const int64_t *b,
                          const int64_t *user_ptr, const int64_t *item, const double *pref, int nthreads) {
  double **own = (double **)malloc(sizeof(double *) * (size_t)(U > 0 ? U : 1));
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 64)
  for (int64_t u = 0; u < U; u++) own[u] = sized_profile(u, width[u], depth[u], a, b, user_ptr, item, pref);
  return own;
}

static void sized_free(double **own, int64_t U) {
  for (int64_t u = 0; u < U; u++) free(own[u]);
  free(own);
}

typedef struct {
  double sim;
  int64_t idx;
} sized_elem;

/* (similarity desc, index asc) */
static int sized_cmp(const void *p, const void *q) {
  const sized_elem *x = (const sized_elem *)p, *y = (const sized_elem *)q;
  if (x->sim != y->sim) return x->sim > y->sim ? -1 : 1;
  return x->idx < y->idx ? -1 : (x->idx > y->idx);
}

/* NearestNUserNeighborhood(n, min_similarity) over CosineCM.userSimilarity exactly as written (CosineCM.java:84-96):
 * for query u1 and every user u2 != u1, u1's prefs are sketched at u2's (width, depth) and compared with u2's own
 * sketch; NaN never admitted, sim >= min_similarity is; the best n under (sim desc, row asc).  u1's re-sketch depends
 * on u2 only through the shape, so it is built once per (query, shape).  out_idx / out_sim [q][n] (unused -1 / 0),
 * out_cnt [q]. */
void orc_sized_neighborhood(int64_t U, const int32_t *width, const int32_t *depth, const int64_t *a,
                            const int64_t *b, const int64_t *user_ptr, const int64_t *item, const double *pref,
                            const int64_t *queries, int64_t q, int n, double min_similarity, int nthreads,
                            int64_t *out_idx, double *out_sim, int32_t *out_cnt) {
  if (nthreads < 1) nthreads = 1;
  double **own = sized_own(U, width, depth, a, b, user_ptr, item, pref, nthreads);
  int32_t *cls = (int32_t *)malloc(sizeof(int32_t) * (size_t)(U > 0 ? U : 1));
  int32_t *sw = (int32_t *)malloc(sizeof(int32_t) * (size_t)(U > 0 ? U : 1));
  int32_t *sd = (int32_t *)malloc(sizeof(int32_t) * (size_t)(U > 0 ? U : 1));
  int32_t nshapes = 0;
  for (int64_t u = 0; u < U; u++) {
    int32_t s = 0;
    while (s < nshapes && (sw[s] != width[u] || sd[s] != depth[u])) s++;
    if (s == nshapes) {
      sw[s] = width[u];
      sd[s] = depth[u];
      nshapes++;
    }
    cls[u] = s;
  }
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 1)
  for (int64_t t = 0; t < q; t++) {
    const int64_t u1 = queries[t];
    double **at = (double **)calloc((size_t)(nshapes > 0 ? nshapes : 1), sizeof(double *));
    sized_elem *cand = (sized_elem *)malloc(sizeof(sized_elem) * (size_t)(U > 0 ? U : 1));
    int64_t m = 0;
    for (int64_t u2 = 0; u2 < U; u2++) {
      if (u2 == u1) continue;
      const int32_t s = cls[u2];
      if (!at[s]) at[s] = sized_profile(u1, width[u2], depth[u2], a, b, user_ptr, item, pref);
      const double r = orc_clamp_similarity(orc_cm_cosine(at[s], own[u2], width[u2], depth[u2]));
      if (!isnan(r) && r >= min_similarity) {
        cand[m].sim = r;
        cand[m].idx = u2;
        m++;
      }
    }
    qsort(cand, (size_t)m, sizeof(sized_elem), sized_cmp);
    const int64_t keep = m < n ? m : n;
    for (int64_t j = 0; j < n; j++) {
      out_idx[t * n + j] = j < keep ? cand[j].idx : -1;
      out_sim[t * n + j] = j < keep ? cand[j].sim : 0.0;
    }
    out_cnt[t] = (int32_t)keep;
    for (int32_t s = 0; s < nshapes; s++) free(at[s]);
    free(at);
    free(cand);
  }
  free(cls);
  free(sw);
  free(sd);
  sized_free(own, U);
}

/* GenericUserBasedRecommender.doEstimatePreference (GenericUserBasedRecommender.java:134-184) with each neighbour's own
 * sketch: for query t (user row user[t], neighbourhood row nb_row[t], or user[t] when nb_row is NULL) the listed
 * v != user[t] in list order:
 *   p = (float) cm_get(own[v]), s = clamp(sim);  p != 0 and s not NaN: pref += s * p, tot += s, count++
 *   out[t] = count <= 1 ? NaN : (float) (pref / tot) */
void orc_sized_estimate(int64_t U, const int32_t *width, const int32_t *depth, const int64_t *a, const int64_t *b,
                        const int64_t *user_ptr, const int64_t *item, const double *pref, const int64_t *nb_idx,
                        const double *nb_sim, const int32_t *nb_cnt, int32_t nb_ld, const int64_t *user,
                        const int64_t *nb_row, const int64_t *item_id, int64_t q, int nthreads, float *out) {
  if (nthreads < 1) nthreads = 1;
  double **own = sized_own(U, width, depth, a, b, user_ptr, item, pref, nthreads);
#pragma omp parallel for num_threads(nthreads) schedule(static)
  for (int64_t t = 0; t < q; t++) {
    const int64_t u = user[t], row = nb_row ? nb_row[t] : u;
    double preference = 0.0, total = 0.0;
    int count = 0;
    for (int32_t j = 0; j < nb_cnt[row]; j++) {
      const int64_t v = nb_idx[row * nb_ld + j];
      if (v == u) continue;
      const float p = (float)orc_cm_get(own[v], width[v], depth[v], a, b, item_id[t]);
      const double s = orc_clamp_similarity(nb_sim[row * nb_ld + j]);
      if (p != 0.0f && !isnan(s)) {
        preference += s * (double)p;
        total += s;
        count++;
      }
    }
    out[t] = count <= 1 ? NAN : (float)(preference / total);
  }
  sized_free(own, U);
}
