/*
 * JNI glue: Java_org_apache_mahout_cf_taste_impl_common_NativeSketch_* -> include/mahout_b200.h.
 * 1:1, no logic.  Status codes map to exceptions the reference throws at the same places:
 *   MB200_ERR_BAD_ARG            -> IllegalArgumentException (Guava Preconditions, DoubleCountMinSketch.java:117)
 *   MB200_ERR_CM_DELTA/_EPSILON  -> IllegalArgumentException carrying the CMException text
 *   everything else              -> org.apache.mahout.cf.taste.common.TasteException
 *
 * NOT BUILT IN THIS REPOSITORY: the image has no jni.h.  Build where a JDK exists with
 *   gcc -shared -fPIC -I$JAVA_HOME/include -I$JAVA_HOME/include/linux -Iinclude \
 *       jni/mahout_b200_jni.c -Lmahout_b200 -lmahout_b200 -o libmahout_b200_jni.so
 */
#include <jni.h>
#include <stddef.h>
#include <stdint.h>

#include "mahout_b200.h"

#define JNI_FN(name) Java_org_apache_mahout_cf_taste_impl_common_NativeSketch_##name

static void throw_status(JNIEnv* env, int rc, mb200_ctx* ctx) {
  const char* cls = (rc == MB200_ERR_BAD_ARG || rc == MB200_ERR_CM_DELTA || rc == MB200_ERR_CM_EPSILON)
                        ? "java/lang/IllegalArgumentException"
                        : "org/apache/mahout/cf/taste/common/TasteException";
  (*env)->ThrowNew(env, (*env)->FindClass(env, cls), mb200_last_error(ctx));
}
#define CHECK(rc, ctx) do { int rc_ = (rc); if (rc_ != MB200_OK) { throw_status(env, rc_, (ctx)); } } while (0)

JNIEXPORT jlong JNICALL JNI_FN(createContext)(JNIEnv* env, jclass c, jint device) {
  mb200_ctx* ctx = NULL;
  CHECK(mb200_create(device, &ctx), NULL);
  return (jlong)(intptr_t)ctx;
}

JNIEXPORT void JNICALL JNI_FN(destroyContext)(JNIEnv* env, jclass c, jlong ctx) {
  mb200_destroy((mb200_ctx*)(intptr_t)ctx);
}

JNIEXPORT void JNICALL JNI_FN(hashParams)(JNIEnv* env, jclass c, jlong seed, jint depth, jlongArray a, jlongArray b) {
  jlong* pa = (*env)->GetLongArrayElements(env, a, NULL);
  jlong* pb = (*env)->GetLongArrayElements(env, b, NULL);
  int rc = mb200_hash_params(seed, depth, (int64_t*)pa, (int64_t*)pb);
  (*env)->ReleaseLongArrayElements(env, a, pa, 0);
  (*env)->ReleaseLongArrayElements(env, b, pb, 0);
  CHECK(rc, NULL);
}

JNIEXPORT jlong JNICALL JNI_FN(createBank)(JNIEnv* env, jclass c, jlong ctx, jlong entities, jint depth, jint width,
                                           jlongArray a, jlongArray b, jint fracBits) {
  mb200_bank* bank = NULL;
  jlong* pa = (*env)->GetLongArrayElements(env, a, NULL);
  jlong* pb = (*env)->GetLongArrayElements(env, b, NULL);
  int rc = mb200_bank_create_params((mb200_ctx*)(intptr_t)ctx, entities, depth, width, (int64_t*)pa, (int64_t*)pb,
                                    fracBits, &bank);
  (*env)->ReleaseLongArrayElements(env, a, pa, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, b, pb, JNI_ABORT);
  CHECK(rc, (mb200_ctx*)(intptr_t)ctx);
  return (jlong)(intptr_t)bank;
}

JNIEXPORT void JNICALL JNI_FN(destroyBank)(JNIEnv* env, jclass c, jlong bank) {
  mb200_bank_destroy((mb200_bank*)(intptr_t)bank);
}

JNIEXPORT void JNICALL JNI_FN(update)(JNIEnv* env, jclass c, jlong bank, jobject entity, jobject key, jobject inc, jlong n) {
  const int64_t* e = entity ? (const int64_t*)(*env)->GetDirectBufferAddress(env, entity) : NULL;
  const int64_t* k = (const int64_t*)(*env)->GetDirectBufferAddress(env, key);
  const float* v = (const float*)(*env)->GetDirectBufferAddress(env, inc);
  CHECK(mb200_bank_update((mb200_bank*)(intptr_t)bank, e, k, v, n, MB200_MEM_HOST), NULL);
}

JNIEXPORT void JNICALL JNI_FN(updateOne)(JNIEnv* env, jclass c, jlong bank, jlong entity, jlong key, jdouble inc) {
  int64_t e = entity, k = key;
  double v = inc;
  CHECK(mb200_bank_update_f64((mb200_bank*)(intptr_t)bank, &e, &k, &v, 1, MB200_MEM_HOST), NULL);
}

JNIEXPORT jdouble JNICALL JNI_FN(query)(JNIEnv* env, jclass c, jlong bank, jlong entity, jlong key) {
  int64_t e = entity, k = key;
  double out = 0.0;
  CHECK(mb200_bank_query((mb200_bank*)(intptr_t)bank, &e, &k, 1, &out, MB200_MEM_HOST), NULL);
  return out;
}

JNIEXPORT jdouble JNICALL JNI_FN(cosine)(JNIEnv* env, jclass c, jlong bankA, jlong ea, jlong bankB, jlong eb) {
  int64_t a = ea, b = eb;
  double out = 0.0;
  CHECK(mb200_bank_cross_cosine((mb200_bank*)(intptr_t)bankA, &a, (mb200_bank*)(intptr_t)bankB, &b, 1, &out,
                                MB200_MEM_HOST), NULL);
  return out;
}

JNIEXPORT void JNICALL JNI_FN(cosineTopK)(JNIEnv* env, jclass c, jlong bank, jint k, jdouble threshold,
                                          jboolean excludeSelf, jint dtype, jint precision, jlongArray outIdx,
                                          jdoubleArray outSim, jintArray outCnt) {
  jlong* pi = (*env)->GetLongArrayElements(env, outIdx, NULL);
  jdouble* ps = (*env)->GetDoubleArrayElements(env, outSim, NULL);
  jint* pc = (*env)->GetIntArrayElements(env, outCnt, NULL);
  int rc = mb200_bank_cosine_topk((mb200_bank*)(intptr_t)bank, k, threshold, excludeSelf, dtype, precision,
                                  (int64_t*)pi, ps, (int32_t*)pc, MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, outIdx, pi, 0);
  (*env)->ReleaseDoubleArrayElements(env, outSim, ps, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, pc, 0);
  CHECK(rc, NULL);
}

JNIEXPORT jobject JNICALL JNI_FN(allocPinned)(JNIEnv* env, jclass c, jlong bytes) {
  void* p = NULL;
  CHECK(mb200_host_alloc(bytes, &p), NULL);
  return p ? (*env)->NewDirectByteBuffer(env, p, bytes) : NULL;
}

JNIEXPORT void JNICALL JNI_FN(freePinned)(JNIEnv* env, jclass c, jobject buffer) {
  mb200_host_free((*env)->GetDirectBufferAddress(env, buffer));
}
/* ---- ingest (PreparePreferenceMatrixJob on the GPU) ------------------------------------------------ */
JNIEXPORT jlong JNICALL JNI_FN(parsePrefs)(JNIEnv* env, jclass c, jlong ctx, jobject text, jlong bytes,
                                           jboolean booleanData, jfloat ratingShift, jboolean transpose) {
  mb200_events* ev = NULL;
  CHECK(mb200_events_parse((mb200_ctx*)(intptr_t)ctx, (const char*)(*env)->GetDirectBufferAddress(env, text), bytes,
                           MB200_MEM_HOST, booleanData, ratingShift, transpose, &ev), (mb200_ctx*)(intptr_t)ctx);
  return (jlong)(intptr_t)ev;
}

JNIEXPORT jlong JNICALL JNI_FN(eventCount)(JNIEnv* env, jclass c, jlong events) {
  int64_t n = 0;
  CHECK(mb200_events_count((mb200_events*)(intptr_t)events, &n), NULL);
  return n;
}

JNIEXPORT void JNICALL JNI_FN(destroyEvents)(JNIEnv* env, jclass c, jlong events) {
  mb200_events_destroy((mb200_events*)(intptr_t)events);
}

JNIEXPORT jlong JNICALL JNI_FN(prepare)(JNIEnv* env, jclass c, jlong events, jint minPrefsPerUser) {
  mb200_prefs* p = NULL;
  CHECK(mb200_events_prepare((mb200_events*)(intptr_t)events, minPrefsPerUser, &p), NULL);
  return (jlong)(intptr_t)p;
}

/* info[0..2] = surviving events, items (matrix rows), users */
JNIEXPORT void JNICALL JNI_FN(prefsInfo)(JNIEnv* env, jclass c, jlong prefs, jlongArray info) {
  int64_t v[3] = {0, 0, 0};
  CHECK(mb200_prefs_info((mb200_prefs*)(intptr_t)prefs, &v[0], &v[1], &v[2]), NULL);
  (*env)->SetLongArrayRegion(env, info, 0, 3, (const jlong*)v);
}

JNIEXPORT void JNICALL JNI_FN(prefsTables)(JNIEnv* env, jclass c, jlong prefs, jlongArray itemId, jintArray indexValues) {
  jlong* pi = (*env)->GetLongArrayElements(env, itemId, NULL);
  jint* px = (*env)->GetIntArrayElements(env, indexValues, NULL);
  int rc = mb200_prefs_tables((mb200_prefs*)(intptr_t)prefs, (int64_t*)pi, (int32_t*)px);
  (*env)->ReleaseLongArrayElements(env, itemId, pi, 0);
  (*env)->ReleaseIntArrayElements(env, indexValues, px, 0);
  CHECK(rc, NULL);
}

/* K1 straight from the prepared (device-resident) events: entity = row, key = user, inc = pref */
JNIEXPORT void JNICALL JNI_FN(updateFromPrefs)(JNIEnv* env, jclass c, jlong bank, jlong prefs) {
  int64_t *row = NULL, *user = NULL, n = 0;
  float* pref = NULL;
  CHECK(mb200_prefs_info((mb200_prefs*)(intptr_t)prefs, &n, NULL, NULL), NULL);
  CHECK(mb200_prefs_columns((mb200_prefs*)(intptr_t)prefs, &row, &user, &pref), NULL);
  CHECK(mb200_bank_update((mb200_bank*)(intptr_t)bank, row, user, pref, n, MB200_MEM_DEVICE), NULL);
}

JNIEXPORT void JNICALL JNI_FN(destroyPrefs)(JNIEnv* env, jclass c, jlong prefs) {
  mb200_prefs_destroy((mb200_prefs*)(intptr_t)prefs);
}
/* clearBank, check, queryMany, read, cmDims follow the same pattern (one C call each). */

/* ---- the whole similarity phase over all GPUs of the process (csrc/job.cu) ------------------------------------ */
static void throw_multi(JNIEnv* env, int rc, mb200_multi* m) {
  const char* cls = rc == MB200_ERR_BAD_ARG ? "java/lang/IllegalArgumentException"
                                            : "org/apache/mahout/cf/taste/common/TasteException";
  (*env)->ThrowNew(env, (*env)->FindClass(env, cls), mb200_multi_last_error(m));
}

JNIEXPORT jlong JNICALL JNI_FN(createMulti)(JNIEnv* env, jclass c, jint numGpus) {
  mb200_multi* m = NULL;
  int rc = mb200_create_multi(numGpus, NULL, &m);
  if (rc != MB200_OK) throw_multi(env, rc, NULL);
  return (jlong)(intptr_t)m;
}

JNIEXPORT void JNICALL JNI_FN(destroyMulti)(JNIEnv* env, jclass c, jlong multi) {
  mb200_multi_destroy((mb200_multi*)(intptr_t)multi);
}

JNIEXPORT void JNICALL JNI_FN(jobItemSimilarity)(JNIEnv* env, jclass c, jlong multi, jlongArray row, jlongArray key,
                                                 jfloatArray value, jlong numRows, jint k, jdouble threshold, jint width,
                                                 jint depth, jlong seed, jboolean exactMeasure, jint fracBits, jint dtype,
                                                 jint precision, jlongArray outIdx, jdoubleArray outSim, jintArray outCnt,
                                                 jlongArray stats) {
  mb200_multi* m = (mb200_multi*)(intptr_t)multi;
  const jsize n = (*env)->GetArrayLength(env, row);
  jlong* prow = (*env)->GetLongArrayElements(env, row, NULL);
  jlong* pkey = (*env)->GetLongArrayElements(env, key, NULL);
  jfloat* pval = (*env)->GetFloatArrayElements(env, value, NULL);
  jlong* pidx = (*env)->GetLongArrayElements(env, outIdx, NULL);
  jdouble* psim = (*env)->GetDoubleArrayElements(env, outSim, NULL);
  jint* pcnt = (*env)->GetIntArrayElements(env, outCnt, NULL);
  const int64_t one = 1, zero = 0;
  mb200_job_params p;
  mb200_job_stats st;
  p.k = k;
  p.threshold = threshold;
  p.width = width;
  p.depth = depth;
  p.seed = seed;
  p.hash_a = exactMeasure ? &one : NULL;
  p.hash_b = exactMeasure ? &zero : NULL;
  p.frac_bits = fracBits;
  p.dtype = dtype;
  p.precision = precision;
  int rc = mb200_job_item_similarity(m, (const int64_t*)prow, (const int64_t*)pkey, (const float*)pval, n, numRows, &p,
                                     (int64_t*)pidx, (double*)psim, (int32_t*)pcnt, &st);
  (*env)->ReleaseLongArrayElements(env, row, prow, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, key, pkey, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, value, pval, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outIdx, pidx, 0);
  (*env)->ReleaseDoubleArrayElements(env, outSim, psim, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, pcnt, 0);
  if (rc != MB200_OK) {
    throw_multi(env, rc, m);
    return;
  }
  if (stats != NULL && (*env)->GetArrayLength(env, stats) >= 9) {
    jlong w[9];
    w[0] = st.n_gpus;
    w[1] = st.events;
    w[2] = st.rows;
    w[3] = st.similarities_kept;
    w[4] = st.fallback_rows;
    w[5] = st.events_busiest_gpu;
    w[6] = (jlong)(st.route_s * 1e3);
    w[7] = (jlong)(st.build_s * 1e3);
    w[8] = (jlong)(st.cosine_s * 1e3);
    (*env)->SetLongArrayRegion(env, stats, 0, 9, w);
  }
}

JNIEXPORT void JNICALL JNI_FN(updateU8)(JNIEnv* env, jclass c, jlong bank, jobject entity, jobject key, jobject quanta,
                                        jlong n) {
  const uint32_t* e = entity ? (const uint32_t*)(*env)->GetDirectBufferAddress(env, entity) : NULL;
  const uint32_t* k = (const uint32_t*)(*env)->GetDirectBufferAddress(env, key);
  const uint8_t* q = (const uint8_t*)(*env)->GetDirectBufferAddress(env, quanta);
  CHECK(mb200_bank_update_u8((mb200_bank*)(intptr_t)bank, e, k, q, n, MB200_MEM_HOST), NULL);
}


/* ---- GenericUserBasedRecommender over the user bank (csrc/recommend.cu) --------------------------------------- */
JNIEXPORT void JNICALL JNI_FN(estimatePrefs)(JNIEnv* env, jclass c, jlong bank, jlongArray nbIdx, jdoubleArray nbSim,
                                             jintArray nbCnt, jint nbLd, jlongArray user, jlongArray itemId,
                                             jfloatArray out) {
  const jsize rows = (*env)->GetArrayLength(env, nbCnt), q = (*env)->GetArrayLength(env, user);
  jlong* pi = (*env)->GetLongArrayElements(env, nbIdx, NULL);
  jdouble* ps = (*env)->GetDoubleArrayElements(env, nbSim, NULL);
  jint* pc = (*env)->GetIntArrayElements(env, nbCnt, NULL);
  jlong* pu = (*env)->GetLongArrayElements(env, user, NULL);
  jlong* pt = (*env)->GetLongArrayElements(env, itemId, NULL);
  jfloat* po = (*env)->GetFloatArrayElements(env, out, NULL);
  int rc = (*env)->GetArrayLength(env, itemId) != q || (*env)->GetArrayLength(env, out) != q
               ? MB200_ERR_BAD_ARG
               : mb200_bank_estimate_prefs((mb200_bank*)(intptr_t)bank, (const int64_t*)pi, ps, (const int32_t*)pc, rows,
                                           nbLd, (const int64_t*)pu, NULL, (const int64_t*)pt, q, (float*)po,
                                           MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, nbIdx, pi, JNI_ABORT);
  (*env)->ReleaseDoubleArrayElements(env, nbSim, ps, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, nbCnt, pc, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, user, pu, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemId, pt, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, out, po, 0);
  CHECK(rc, NULL);
}

JNIEXPORT void JNICALL JNI_FN(recommend)(JNIEnv* env, jclass c, jlong bank, jlongArray nbIdx, jdoubleArray nbSim,
                                         jintArray nbCnt, jint nbLd, jlongArray itemPtr, jintArray itemCol,
                                         jlongArray itemIds, jlongArray users, jint howMany, jboolean includeKnown,
                                         jlongArray outItem, jfloatArray outValue, jintArray outCnt) {
  jlong* pi = (*env)->GetLongArrayElements(env, nbIdx, NULL);
  jdouble* ps = (*env)->GetDoubleArrayElements(env, nbSim, NULL);
  jint* pc = (*env)->GetIntArrayElements(env, nbCnt, NULL);
  jlong* pp = (*env)->GetLongArrayElements(env, itemPtr, NULL);
  jint* pl = (*env)->GetIntArrayElements(env, itemCol, NULL);
  jlong* pd = (*env)->GetLongArrayElements(env, itemIds, NULL);
  jlong* pu = (*env)->GetLongArrayElements(env, users, NULL);
  jlong* oi = (*env)->GetLongArrayElements(env, outItem, NULL);
  jfloat* ov = (*env)->GetFloatArrayElements(env, outValue, NULL);
  jint* oc = (*env)->GetIntArrayElements(env, outCnt, NULL);
  const jsize m = (*env)->GetArrayLength(env, users);
  int rc = (*env)->GetArrayLength(env, outCnt) != m ||
                   (int64_t)(*env)->GetArrayLength(env, outItem) != (int64_t)m * howMany ||
                   (*env)->GetArrayLength(env, outValue) != (*env)->GetArrayLength(env, outItem)
               ? MB200_ERR_BAD_ARG
               : mb200_bank_recommend((mb200_bank*)(intptr_t)bank, (const int64_t*)pi, ps, (const int32_t*)pc, nbLd,
                                      (const int64_t*)pp, (const int32_t*)pl, (*env)->GetArrayLength(env, itemCol),
                                      (const int64_t*)pd, (*env)->GetArrayLength(env, itemIds), (const int64_t*)pu, m,
                                      howMany, includeKnown, (int64_t*)oi, (float*)ov, (int32_t*)oc, MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, nbIdx, pi, JNI_ABORT);
  (*env)->ReleaseDoubleArrayElements(env, nbSim, ps, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, nbCnt, pc, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemPtr, pp, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, itemCol, pl, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemIds, pd, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, users, pu, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outItem, oi, 0);
  (*env)->ReleaseFloatArrayElements(env, outValue, ov, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, oc, 0);
  CHECK(rc, NULL);
}

/* ---- RecommenderJob's aggregate-and-recommend phase over the item top-k lists (csrc/recommend.cu) ------------- */
JNIEXPORT void JNICALL JNI_FN(recommendItemBased)(JNIEnv* env, jclass c, jlong ctx, jlongArray simIdx,
                                                  jdoubleArray simVal, jintArray simCnt, jint simLd, jlongArray userPtr,
                                                  jintArray prefRow, jfloatArray prefVal, jlongArray itemIds,
                                                  jintArray allowed, jlongArray users, jint howMany,
                                                  jint maxPrefsPerUser, jboolean booleanData, jlongArray outItem,
                                                  jfloatArray outValue, jintArray outCnt) {
  mb200_itembased_args a;
  a.sim_idx = (const int64_t*)(*env)->GetLongArrayElements(env, simIdx, NULL);
  a.sim_val = (*env)->GetDoubleArrayElements(env, simVal, NULL);
  a.sim_cnt = (const int32_t*)(*env)->GetIntArrayElements(env, simCnt, NULL);
  a.num_items = (*env)->GetArrayLength(env, simCnt);
  a.sim_ld = simLd;
  a.user_ptr = (const int64_t*)(*env)->GetLongArrayElements(env, userPtr, NULL);
  a.pref_row = (const int32_t*)(*env)->GetIntArrayElements(env, prefRow, NULL);
  a.pref_val = (*env)->GetFloatArrayElements(env, prefVal, NULL);
  a.num_users = (int64_t)(*env)->GetArrayLength(env, userPtr) - 1;
  a.nnz = (*env)->GetArrayLength(env, prefRow);
  a.item_ids = (const int64_t*)(*env)->GetLongArrayElements(env, itemIds, NULL);
  a.allowed = allowed ? (const uint32_t*)(*env)->GetIntArrayElements(env, allowed, NULL) : NULL;
  a.users = (const int64_t*)(*env)->GetLongArrayElements(env, users, NULL);
  a.m = (*env)->GetArrayLength(env, users);
  a.how_many = howMany;
  a.max_prefs_per_user = maxPrefsPerUser;
  a.boolean_data = booleanData;
  a.out_item = (int64_t*)(*env)->GetLongArrayElements(env, outItem, NULL);
  a.out_value = (*env)->GetFloatArrayElements(env, outValue, NULL);
  a.out_cnt = (int32_t*)(*env)->GetIntArrayElements(env, outCnt, NULL);
  a.mem = MB200_MEM_HOST;
  int rc = (int64_t)(*env)->GetArrayLength(env, simIdx) != a.num_items * simLd ||
                   (*env)->GetArrayLength(env, simVal) != (*env)->GetArrayLength(env, simIdx) ||
                   (*env)->GetArrayLength(env, prefVal) != a.nnz || (*env)->GetArrayLength(env, itemIds) != a.num_items ||
                   (allowed && (*env)->GetArrayLength(env, allowed) != (a.num_items + 31) / 32) ||
                   (*env)->GetArrayLength(env, outCnt) != a.m ||
                   (int64_t)(*env)->GetArrayLength(env, outItem) != a.m * howMany ||
                   (*env)->GetArrayLength(env, outValue) != (*env)->GetArrayLength(env, outItem)
               ? MB200_ERR_BAD_ARG
               : mb200_recommend_item_based((mb200_ctx*)(intptr_t)ctx, &a);
  (*env)->ReleaseLongArrayElements(env, simIdx, (jlong*)a.sim_idx, JNI_ABORT);
  (*env)->ReleaseDoubleArrayElements(env, simVal, (jdouble*)a.sim_val, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, simCnt, (jint*)a.sim_cnt, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, userPtr, (jlong*)a.user_ptr, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, prefRow, (jint*)a.pref_row, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, prefVal, (jfloat*)a.pref_val, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemIds, (jlong*)a.item_ids, JNI_ABORT);
  if (allowed) (*env)->ReleaseIntArrayElements(env, allowed, (jint*)a.allowed, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, users, (jlong*)a.users, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outItem, (jlong*)a.out_item, 0);
  (*env)->ReleaseFloatArrayElements(env, outValue, a.out_value, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, (jint*)a.out_cnt, 0);
  CHECK(rc, (mb200_ctx*)(intptr_t)ctx);
}

/* ---- CosineCM with a CountMinSketchConfig: per-user sketch sizes (csrc/cmsized.cu) ------------------------------ */
JNIEXPORT jlong JNICALL JNI_FN(createSizedBank)(JNIEnv* env, jclass c, jlong ctx, jintArray width, jintArray depth,
                                                jlongArray a, jlongArray b, jint fracBits, jlongArray userPtr,
                                                jlongArray item, jfloatArray pref) {
  mb200_sized_bank* bank = NULL;
  const jsize users = (*env)->GetArrayLength(env, width);
  jint* pw = (*env)->GetIntArrayElements(env, width, NULL);
  jint* pd = (*env)->GetIntArrayElements(env, depth, NULL);
  jlong* pa = (*env)->GetLongArrayElements(env, a, NULL);
  jlong* pb = (*env)->GetLongArrayElements(env, b, NULL);
  jlong* pp = (*env)->GetLongArrayElements(env, userPtr, NULL);
  jlong* pi = (*env)->GetLongArrayElements(env, item, NULL);
  jfloat* pv = (*env)->GetFloatArrayElements(env, pref, NULL);
  int rc = (*env)->GetArrayLength(env, depth) != users || (*env)->GetArrayLength(env, userPtr) != users + 1 ||
                   (*env)->GetArrayLength(env, pref) != (*env)->GetArrayLength(env, item) ||
                   (users > 0 && pp[users] != (*env)->GetArrayLength(env, item))
               ? MB200_ERR_BAD_ARG
               : mb200_sized_bank_create((mb200_ctx*)(intptr_t)ctx, users, (const int32_t*)pw, (const int32_t*)pd,
                                         (const int64_t*)pa, (const int64_t*)pb, fracBits, (const int64_t*)pp,
                                         (const int64_t*)pi, (const float*)pv, MB200_MEM_HOST, &bank);
  (*env)->ReleaseIntArrayElements(env, width, pw, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, depth, pd, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, a, pa, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, b, pb, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, userPtr, pp, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, item, pi, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, pref, pv, JNI_ABORT);
  CHECK(rc, (mb200_ctx*)(intptr_t)ctx);
  return (jlong)(intptr_t)bank;
}

JNIEXPORT void JNICALL JNI_FN(destroySizedBank)(JNIEnv* env, jclass c, jlong bank) {
  mb200_sized_bank_destroy((mb200_sized_bank*)(intptr_t)bank);
}

JNIEXPORT void JNICALL JNI_FN(sizedPairCosine)(JNIEnv* env, jclass c, jlong bank, jlongArray u1, jlongArray u2,
                                               jdoubleArray out) {
  const jsize n = (*env)->GetArrayLength(env, u1);
  jlong* p1 = (*env)->GetLongArrayElements(env, u1, NULL);
  jlong* p2 = (*env)->GetLongArrayElements(env, u2, NULL);
  jdouble* po = (*env)->GetDoubleArrayElements(env, out, NULL);
  int rc = (*env)->GetArrayLength(env, u2) != n || (*env)->GetArrayLength(env, out) != n
               ? MB200_ERR_BAD_ARG
               : mb200_sized_pair_cosine((mb200_sized_bank*)(intptr_t)bank, (const int64_t*)p1, (const int64_t*)p2, n,
                                         po, MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, u1, p1, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, u2, p2, JNI_ABORT);
  (*env)->ReleaseDoubleArrayElements(env, out, po, 0);
  CHECK(rc, NULL);
}

JNIEXPORT void JNICALL JNI_FN(sizedNeighborhood)(JNIEnv* env, jclass c, jlong bank, jlongArray queryRows, jint n,
                                                 jdouble minSimilarity, jlongArray outIdx, jdoubleArray outSim,
                                                 jintArray outCnt) {
  const jsize q = (*env)->GetArrayLength(env, queryRows);
  jlong* pq = (*env)->GetLongArrayElements(env, queryRows, NULL);
  jlong* oi = (*env)->GetLongArrayElements(env, outIdx, NULL);
  jdouble* os = (*env)->GetDoubleArrayElements(env, outSim, NULL);
  jint* oc = (*env)->GetIntArrayElements(env, outCnt, NULL);
  int rc = (*env)->GetArrayLength(env, outCnt) != q || (int64_t)(*env)->GetArrayLength(env, outIdx) != (int64_t)q * n ||
                   (*env)->GetArrayLength(env, outSim) != (*env)->GetArrayLength(env, outIdx)
               ? MB200_ERR_BAD_ARG
               : mb200_sized_neighborhood((mb200_sized_bank*)(intptr_t)bank, (const int64_t*)pq, q, n, minSimilarity,
                                          (int64_t*)oi, os, (int32_t*)oc, MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, queryRows, pq, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outIdx, oi, 0);
  (*env)->ReleaseDoubleArrayElements(env, outSim, os, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, oc, 0);
  CHECK(rc, NULL);
}

JNIEXPORT void JNICALL JNI_FN(sizedEstimatePrefs)(JNIEnv* env, jclass c, jlong bank, jlongArray nbIdx,
                                                  jdoubleArray nbSim, jintArray nbCnt, jint nbLd, jlongArray user,
                                                  jlongArray nbRow, jlongArray itemId, jfloatArray out) {
  const jsize rows = (*env)->GetArrayLength(env, nbCnt), q = (*env)->GetArrayLength(env, user);
  jlong* pi = (*env)->GetLongArrayElements(env, nbIdx, NULL);
  jdouble* ps = (*env)->GetDoubleArrayElements(env, nbSim, NULL);
  jint* pc = (*env)->GetIntArrayElements(env, nbCnt, NULL);
  jlong* pu = (*env)->GetLongArrayElements(env, user, NULL);
  jlong* pr = nbRow ? (*env)->GetLongArrayElements(env, nbRow, NULL) : NULL;
  jlong* pt = (*env)->GetLongArrayElements(env, itemId, NULL);
  jfloat* po = (*env)->GetFloatArrayElements(env, out, NULL);
  int rc = (*env)->GetArrayLength(env, itemId) != q || (*env)->GetArrayLength(env, out) != q ||
                   (nbRow && (*env)->GetArrayLength(env, nbRow) != q)
               ? MB200_ERR_BAD_ARG
               : mb200_sized_estimate_prefs((mb200_sized_bank*)(intptr_t)bank, (const int64_t*)pi, ps,
                                            (const int32_t*)pc, rows, nbLd, (const int64_t*)pu, (const int64_t*)pr,
                                            (const int64_t*)pt, q, (float*)po, MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, nbIdx, pi, JNI_ABORT);
  (*env)->ReleaseDoubleArrayElements(env, nbSim, ps, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, nbCnt, pc, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, user, pu, JNI_ABORT);
  if (pr) (*env)->ReleaseLongArrayElements(env, nbRow, pr, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemId, pt, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, out, po, 0);
  CHECK(rc, NULL);
}

JNIEXPORT void JNICALL JNI_FN(sizedRecommend)(JNIEnv* env, jclass c, jlong bank, jlongArray nbIdx, jdoubleArray nbSim,
                                              jintArray nbCnt, jint nbLd, jlongArray itemPtr, jintArray itemCol,
                                              jlongArray itemIds, jlongArray users, jint howMany,
                                              jboolean includeKnown, jlongArray outItem, jfloatArray outValue,
                                              jintArray outCnt) {
  jlong* pi = (*env)->GetLongArrayElements(env, nbIdx, NULL);
  jdouble* ps = (*env)->GetDoubleArrayElements(env, nbSim, NULL);
  jint* pc = (*env)->GetIntArrayElements(env, nbCnt, NULL);
  jlong* pp = (*env)->GetLongArrayElements(env, itemPtr, NULL);
  jint* pl = (*env)->GetIntArrayElements(env, itemCol, NULL);
  jlong* pd = (*env)->GetLongArrayElements(env, itemIds, NULL);
  jlong* pu = (*env)->GetLongArrayElements(env, users, NULL);
  jlong* oi = (*env)->GetLongArrayElements(env, outItem, NULL);
  jfloat* ov = (*env)->GetFloatArrayElements(env, outValue, NULL);
  jint* oc = (*env)->GetIntArrayElements(env, outCnt, NULL);
  const jsize m = (*env)->GetArrayLength(env, users);
  /* row t of the lists is users[t]'s neighbourhood */
  int rc = (*env)->GetArrayLength(env, nbCnt) != m || (*env)->GetArrayLength(env, outCnt) != m ||
                   nbLd < 1 || (int64_t)(*env)->GetArrayLength(env, nbIdx) != (int64_t)m * nbLd ||
                   (*env)->GetArrayLength(env, nbSim) != (*env)->GetArrayLength(env, nbIdx) ||
                   (int64_t)(*env)->GetArrayLength(env, outItem) != (int64_t)m * howMany ||
                   (*env)->GetArrayLength(env, outValue) != (*env)->GetArrayLength(env, outItem)
               ? MB200_ERR_BAD_ARG
               : mb200_sized_recommend((mb200_sized_bank*)(intptr_t)bank, (const int64_t*)pi, ps, (const int32_t*)pc,
                                       nbLd, (const int64_t*)pp, (const int32_t*)pl,
                                       (*env)->GetArrayLength(env, itemCol), (const int64_t*)pd,
                                       (*env)->GetArrayLength(env, itemIds), (const int64_t*)pu, m, howMany,
                                       includeKnown, (int64_t*)oi, (float*)ov, (int32_t*)oc, MB200_MEM_HOST);
  (*env)->ReleaseLongArrayElements(env, nbIdx, pi, JNI_ABORT);
  (*env)->ReleaseDoubleArrayElements(env, nbSim, ps, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, nbCnt, pc, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemPtr, pp, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, itemCol, pl, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemIds, pd, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, users, pu, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outItem, oi, 0);
  (*env)->ReleaseFloatArrayElements(env, outValue, ov, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, oc, 0);
  CHECK(rc, NULL);
}

/* ---- the sized bank on all GPUs of the process (csrc/sized_multi.cu) ------------------------------------------- */
JNIEXPORT jlong JNICALL JNI_FN(createSizedMulti)(JNIEnv* env, jclass c, jlong multi, jintArray width, jintArray depth,
                                                 jlongArray a, jlongArray b, jint fracBits, jlongArray userPtr,
                                                 jlongArray item, jfloatArray pref) {
  mb200_multi* m = (mb200_multi*)(intptr_t)multi;
  mb200_sized_multi* sm = NULL;
  const jsize users = (*env)->GetArrayLength(env, width);
  jint* pw = (*env)->GetIntArrayElements(env, width, NULL);
  jint* pd = (*env)->GetIntArrayElements(env, depth, NULL);
  jlong* pa = (*env)->GetLongArrayElements(env, a, NULL);
  jlong* pb = (*env)->GetLongArrayElements(env, b, NULL);
  jlong* pp = (*env)->GetLongArrayElements(env, userPtr, NULL);
  jlong* pi = (*env)->GetLongArrayElements(env, item, NULL);
  jfloat* pv = (*env)->GetFloatArrayElements(env, pref, NULL);
  int rc = (*env)->GetArrayLength(env, depth) != users || (*env)->GetArrayLength(env, userPtr) != users + 1 ||
                   (*env)->GetArrayLength(env, pref) != (*env)->GetArrayLength(env, item) ||
                   (users > 0 && pp[users] != (*env)->GetArrayLength(env, item))
               ? MB200_ERR_BAD_ARG
               : mb200_sized_multi_create(m, users, (const int32_t*)pw, (const int32_t*)pd, (const int64_t*)pa,
                                          (const int64_t*)pb, fracBits, (const int64_t*)pp, (const int64_t*)pi,
                                          (const float*)pv, &sm);
  (*env)->ReleaseIntArrayElements(env, width, pw, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, depth, pd, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, a, pa, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, b, pb, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, userPtr, pp, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, item, pi, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, pref, pv, JNI_ABORT);
  if (rc != MB200_OK) throw_multi(env, rc, m);
  return (jlong)(intptr_t)sm;
}

JNIEXPORT void JNICALL JNI_FN(destroySizedMulti)(JNIEnv* env, jclass c, jlong sizedMulti) {
  mb200_sized_multi_destroy((mb200_sized_multi*)(intptr_t)sizedMulti);
}

JNIEXPORT void JNICALL JNI_FN(sizedMultiNeighborhood)(JNIEnv* env, jclass c, jlong sizedMulti, jlongArray queryRows,
                                                      jint n, jdouble minSimilarity, jlongArray outIdx,
                                                      jdoubleArray outSim, jintArray outCnt) {
  const jsize q = (*env)->GetArrayLength(env, queryRows);
  jlong* pq = (*env)->GetLongArrayElements(env, queryRows, NULL);
  jlong* oi = (*env)->GetLongArrayElements(env, outIdx, NULL);
  jdouble* os = (*env)->GetDoubleArrayElements(env, outSim, NULL);
  jint* oc = (*env)->GetIntArrayElements(env, outCnt, NULL);
  int rc = (*env)->GetArrayLength(env, outCnt) != q || (int64_t)(*env)->GetArrayLength(env, outIdx) != (int64_t)q * n ||
                   (*env)->GetArrayLength(env, outSim) != (*env)->GetArrayLength(env, outIdx)
               ? MB200_ERR_BAD_ARG
               : mb200_sized_multi_neighborhood((mb200_sized_multi*)(intptr_t)sizedMulti, (const int64_t*)pq, q, n,
                                                minSimilarity, (int64_t*)oi, os, (int32_t*)oc);
  (*env)->ReleaseLongArrayElements(env, queryRows, pq, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outIdx, oi, 0);
  (*env)->ReleaseDoubleArrayElements(env, outSim, os, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, oc, 0);
  if (rc != MB200_OK) throw_multi(env, rc, NULL);  /* the calling thread's message: "GPU d: ..." */
}

JNIEXPORT void JNICALL JNI_FN(sizedMultiRecommend)(JNIEnv* env, jclass c, jlong sizedMulti, jlongArray users, jint n,
                                                   jdouble minSimilarity, jlongArray itemPtr, jintArray itemCol,
                                                   jlongArray itemIds, jint howMany, jboolean includeKnown,
                                                   jlongArray outItem, jfloatArray outValue, jintArray outCnt) {
  jlong* pu = (*env)->GetLongArrayElements(env, users, NULL);
  jlong* pp = (*env)->GetLongArrayElements(env, itemPtr, NULL);
  jint* pl = (*env)->GetIntArrayElements(env, itemCol, NULL);
  jlong* pd = (*env)->GetLongArrayElements(env, itemIds, NULL);
  jlong* oi = (*env)->GetLongArrayElements(env, outItem, NULL);
  jfloat* ov = (*env)->GetFloatArrayElements(env, outValue, NULL);
  jint* oc = (*env)->GetIntArrayElements(env, outCnt, NULL);
  const jsize m = (*env)->GetArrayLength(env, users);
  int rc = (*env)->GetArrayLength(env, outCnt) != m ||
                   (int64_t)(*env)->GetArrayLength(env, outItem) != (int64_t)m * howMany ||
                   (*env)->GetArrayLength(env, outValue) != (*env)->GetArrayLength(env, outItem)
               ? MB200_ERR_BAD_ARG
               : mb200_sized_multi_recommend((mb200_sized_multi*)(intptr_t)sizedMulti, (const int64_t*)pu, m, n,
                                             minSimilarity, (const int64_t*)pp, (const int32_t*)pl,
                                             (*env)->GetArrayLength(env, itemCol), (const int64_t*)pd,
                                             (*env)->GetArrayLength(env, itemIds), howMany, includeKnown, (int64_t*)oi,
                                             (float*)ov, (int32_t*)oc);
  (*env)->ReleaseLongArrayElements(env, users, pu, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemPtr, pp, JNI_ABORT);
  (*env)->ReleaseIntArrayElements(env, itemCol, pl, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemIds, pd, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, outItem, oi, 0);
  (*env)->ReleaseFloatArrayElements(env, outValue, ov, 0);
  (*env)->ReleaseIntArrayElements(env, outCnt, oc, 0);
  if (rc != MB200_OK) throw_multi(env, rc, NULL);
}

JNIEXPORT void JNICALL JNI_FN(sizedMultiEstimatePrefs)(JNIEnv* env, jclass c, jlong sizedMulti, jlongArray user,
                                                       jlongArray itemId, jint n, jdouble minSimilarity,
                                                       jfloatArray out) {
  const jsize q = (*env)->GetArrayLength(env, user);
  jlong* pu = (*env)->GetLongArrayElements(env, user, NULL);
  jlong* pt = (*env)->GetLongArrayElements(env, itemId, NULL);
  jfloat* po = (*env)->GetFloatArrayElements(env, out, NULL);
  int rc = (*env)->GetArrayLength(env, itemId) != q || (*env)->GetArrayLength(env, out) != q
               ? MB200_ERR_BAD_ARG
               : mb200_sized_multi_estimate_prefs((mb200_sized_multi*)(intptr_t)sizedMulti, (const int64_t*)pu,
                                                  (const int64_t*)pt, q, n, minSimilarity, (float*)po);
  (*env)->ReleaseLongArrayElements(env, user, pu, JNI_ABORT);
  (*env)->ReleaseLongArrayElements(env, itemId, pt, JNI_ABORT);
  (*env)->ReleaseFloatArrayElements(env, out, po, 0);
  if (rc != MB200_OK) throw_multi(env, rc, NULL);
}
