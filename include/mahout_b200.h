/*
 * mahout_b200.h -- C ABI of libmahout_b200.so: the B200-native (sm_100a) replacement for the
 * sketch-similarity hot path of jalhajj/mahout.  Plain `extern "C"`, opaque handles, plain
 * pointers and sizes; no torch / C++ types.  This is exactly what a JNI (or cgo/ctypes) binding
 * of the reference would bind -- see INTEGRATION.md for the Java/JNI stub.
 *
 * Every function returns an int status (MB200_OK == 0, negative == error class); the message
 * of the last error on a context is available from mb200_last_error().  There is NO CPU
 * fallback: without a CUDA device mb200_create() fails with MB200_ERR_NO_DEVICE.
 *
 * `file:line` cites are into the reference tree (mr/src/main/java/org/apache/mahout/...).
 */
#ifndef MAHOUT_B200_H
#define MAHOUT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MB200_VERSION 1

/* status codes; the JNI glue maps BAD_ARG -> IllegalArgumentException (Guava Preconditions in
 * DoubleCountMinSketch.java:117-118), CM_* -> AbstractCountMinSketch.CMException
 * (AbstractCountMinSketch.java:21-27,71-76), everything else -> TasteException / IOException. */
#define MB200_OK 0
#define MB200_BAND_PENDING 1     /* mb200_cosine_finish: not an error -- see mb200_cosine_args.defer_uncertified */
#define MB200_ERR_BAD_ARG (-1)
#define MB200_ERR_CUDA (-2)
#define MB200_ERR_OOM (-3)
#define MB200_ERR_INEXACT (-4)   /* an increment is not a multiple of the bank's quantum 2^-frac_bits */
#define MB200_ERR_RANGE (-5)     /* a counter left the range in which FP64 sums are exact         */
#define MB200_ERR_NO_DEVICE (-6)
#define MB200_ERR_CM_DELTA (-7)  /* "delta must be between 0 and 1, exclusive"                     */
#define MB200_ERR_CM_EPSILON (-8)
#define MB200_ERR_UNSUPPORTED (-9)
#define MB200_ERR_PULL_TIMEOUT (-10) /* pull-gather: a peer block had not arrived when K3 gave up (~4 s); the staged
                                        operand completes once the copy stream drains: mb200_gather_wait, then push
                                        again without ready_flags (what similarity.fused_gather_cosine and job.cu do) */

#define MB200_MEM_HOST 0
#define MB200_MEM_DEVICE 1

#define MB200_MAX_BLOCKS 64 /* shards / gathered blocks per job */
#define MB200_MAX_DEPTH 32 /* CountMinSketchConfig searches depths 1..24 (CountMinSketchConfig.java:28-29) */

/* element type of the normalised sketch rows fed to the tensor cores */
#define MB200_DTYPE_F16 0  /* rows scaled by 2^12; 11-bit significand (TF32-grade) at BF16 MMA rate */
#define MB200_DTYPE_BF16 1

/* cosine precision modes */
#define MB200_PRECISION_TENSOR 0   /* similarities straight from the FP32 tensor accumulators      */
#define MB200_PRECISION_RESCORED 1 /* tensor cores select k+margin candidates, which are re-scored
                                      exactly from the integer counters: similarities bit-equal to
                                      DoubleCountMinSketch.cosine, top-k sets exact (default)      */
#define MB200_PRECISION_CERTIFIED 2 /* top-k SETS exact, similarities from the tensor cores (<= 1e-3
                                      relative): only the candidates whose membership the tensor
                                      values cannot decide are re-scored exactly                  */

typedef struct mb200_ctx mb200_ctx;
typedef struct mb200_bank mb200_bank;

/* ---- context ------------------------------------------------------------------------- */
int mb200_create(int device, mb200_ctx** out);
int mb200_destroy(mb200_ctx* ctx);
const char* mb200_last_error(mb200_ctx* ctx); /* ctx may be NULL: error of the failed create */
/* run all subsequent work of this context on `cuda_stream` (a cudaStream_t; NULL = the
 * context's own stream).  Lets the caller bracket calls with its own CUDA events. */
int mb200_set_stream(mb200_ctx* ctx, void* cuda_stream);
int mb200_sync(mb200_ctx* ctx);
/* tunables (defaults are what bench.py measures) */
#define MB200_OPT_GROUP_MIN_EVENTS 1 /* bank-mode updates of at least this many events are grouped by entity on
                                        the device first (default 65536; 0 = always; INT64_MAX = never) */
#define MB200_OPT_GROUP_PREFETCH 2   /* the partition passes of that grouping pull their next tile into L2 with
                                        cp.async.bulk.prefetch (default 0: measured neutral on B200, profiles/r2_k1_bank.md) */
#define MB200_OPT_MAX_FALLBACK_ROWS 4 /* RESCORED / CERTIFIED: fail with MB200_ERR_UNSUPPORTED instead of sending more
                                        than this many rows through the exact full-row path (default -1: no limit) */
int mb200_set_option(mb200_ctx* ctx, int option, int64_t value);
/* the cosine stage keeps its device workspaces (candidate lists, gathered rows of the single-GPU
 * convenience call) on the context between calls; this frees them */
int mb200_release_workspace(mb200_ctx* ctx);

/* kernel ids for mb200_kernel_time */
#define MB200_K_UPDATE 0     /* K1 sketch update                 */
#define MB200_K_NORMALIZE 1  /* K2 row norms + 16-bit conversion */
#define MB200_K_COSINE 2     /* K3 tcgen05 S.S^T + top-k epilogue */
#define MB200_K_RESCORE 3    /* K5 merge + exact re-score / certification */
#define MB200_K_PARSE 4     /* ingest: line count + scan + parse    */
#define MB200_K_PREPARE 5   /* ingest: hash-table preparation + compaction */
#define MB200_K_GROUP 6     /* K1 bank mode: histogram + scans + the two partition passes in front of K1 */
#define MB200_K_ROUTE 7     /* sharded ingest: partition by owner GPU + peer scatter */
#define MB200_K_RECOMMEND 8 /* recommenders: user-based estimates + candidates + top-N; item-based rank sort + aggregation */
#define MB200_K_COUNT 9
/* when profiling is on every launch of the kernels above is bracketed with CUDA events on the
 * launching stream; mb200_kernel_time syncs and returns the accumulated ms and launch count
 * since the last reset. */
int mb200_set_profiling(mb200_ctx* ctx, int on);
int mb200_kernel_time(mb200_ctx* ctx, int kernel_id, double* total_ms, int64_t* launches);
int mb200_reset_profile(mb200_ctx* ctx);
/* number of kernels this library has launched on the context since creation */
int mb200_launch_count(mb200_ctx* ctx, int64_t* launches);
/* what the context holds and has done (SURVEY.md 8b: mb200_stats) */
typedef struct mb200_stats {
  int32_t device, num_sms;
  int64_t launches;            /* kernels launched since creation */
  int64_t workspace_bytes;     /* grow-only device workspaces: the cosine stage's and every other call's scratch */
  int64_t staging_bytes;       /* grow-only device staging of host-memory arguments, results and K1 events */
  int64_t last_fallback_rows;  /* rows of the last cosine call that took the exact full-row path */
  int32_t cosine_job_active;
  char device_name[64];
  /* cumulative job counters of this context (RowSimilarityJob.Counters, RowSimilarityJob.java:84, as far as they
   * exist on this path): events applied by mb200_bank_update* (USED_OBSERVATIONS), entity rows whose top-k was
   * computed (ROWS), rows that took the exact full-row path */
  int64_t events_updated;
  int64_t rows_scored;
  int64_t fallback_rows_total;
  int64_t band_rows_total;       /* rows settled by the band pass (second targeted K3 sweep) */
  int64_t h2d_bytes, d2h_bytes;  /* bytes the library itself copied for MB200_MEM_HOST arguments / results */
} mb200_stats;
int mb200_get_stats(mb200_ctx* ctx, mb200_stats* out);

/* ---- pinned host memory ---------------------------------------------------------------- */
/* Page-locked host buffers for the MB200_MEM_HOST paths (a JNI binding wraps them with
 * NewDirectByteBuffer, the way the reference's JavaCPP pointers own native memory,
 * viennacl/.../javacpp/MatrixBase.scala:33-36).  Pageable buffers are accepted everywhere too;
 * they just copy slower. */
int mb200_host_alloc(int64_t bytes, void** out);
int mb200_host_free(void* ptr);
int mb200_host_register(void* ptr, int64_t bytes);
int mb200_host_unregister(void* ptr);

/* ---- hash family --------------------------------------------------------------------- */
/* HashFunctionBuilder(seed): a[i], b[i] = abs(nextLong()), abs(nextLong()) from one
 * java.util.Random(seed) (HashFunctionBuilder.java:23-28,40-60).  Host-side set-up. */
int mb200_hash_params(int64_t seed, int depth, int64_t* a, int64_t* b);
/* AbstractCountMinSketch(delta, epsilon): w = ceil(e/eps), d = ceil(ln(1/delta))
 * (AbstractCountMinSketch.java:69-83); MB200_ERR_CM_DELTA / _EPSILON on the rejected ranges. */
int mb200_cm_dims(double delta, double epsilon, int32_t* width, int32_t* depth);
/* HashFunction.hash(key) = ((a*key + b) mod (2^63-25)) mod w for n keys, on the device
 * (HashFunction.java:31-34). */
int mb200_hash_keys(mb200_ctx* ctx, int64_t a, int64_t b, int32_t w, const int64_t* keys,
                    int64_t n, int32_t* out, int mem);

/* ---- sketch bank: E sketches of d x W counters, C[e][i][j], one hash family --------------- */
/* Replaces `new DoubleCountMinSketch(w, d, hfBuilder)` per entity (DoubleCountMinSketch.java:32-36,
 * CosineCM.java:41-58).  Counters are HBM-resident 64-bit fixed point with quantum 2^-frac_bits
 * (0 <= frac_bits <= 40); they convert to the reference's FP64 counters bit-exactly as long as
 * every increment is a multiple of the quantum (checked on the device, MB200_ERR_INEXACT) and
 * |counter| < 2^53 quanta (MB200_ERR_RANGE). */
int mb200_bank_create(mb200_ctx* ctx, int64_t entities, int32_t depth, int32_t width, int64_t seed,
                      int32_t frac_bits, mb200_bank** out);
/* same, with explicit hash parameters (sketches that must share one HashFunctionBuilder) */
int mb200_bank_create_params(mb200_ctx* ctx, int64_t entities, int32_t depth, int32_t width,
                             const int64_t* a, const int64_t* b, int32_t frac_bits,
                             mb200_bank** out);
int mb200_bank_destroy(mb200_bank* bank);
int mb200_bank_clear(mb200_bank* bank);
/* Checkpoint of a bank (the reference persists its per-user sketch configuration the same way, as a file next to
 * the data: CountMinSketchConfig's .ser cache, CountMinSketchConfig.java:170-219): header (shape, quantum, hash
 * parameters, event count) + the raw fixed-point counters.  mb200_bank_load creates a new bank with exactly the
 * dumped state; MB200_ERR_BAD_ARG on a file that is not a dump or is truncated. */
int mb200_bank_dump(mb200_bank* bank, const char* path);
int mb200_bank_load(mb200_ctx* ctx, const char* path, mb200_bank** out);
/* device pointer of the raw int64 counters (for an NCCL all-reduce of replica sketches) */
int mb200_bank_counters(mb200_bank* bank, void** device_ptr, int64_t* cells);
/* 64-byte CUDA IPC handle of the counters: another rank maps them with mb200_peer_open */
int mb200_bank_ipc_handle(mb200_bank* bank, void* ipc_handle_64_bytes);
/* int32 copy of the counters into DEVICE memory out[E][d][W] (INT_MIN where a counter does not fit) */
int mb200_bank_narrow32(mb200_bank* bank, int32_t* out);

/* DoubleCountMinSketch.update(key, increment) for n events (DoubleCountMinSketch.java:72-80):
 * C[entity[t]][i][h_i(key[t])] += inc[t] for i < d.  `entity` may be NULL when entities == 1.
 * Pointers are host (chunked, double-buffered H2D inside the call) or device memory.
 * Asynchronous for device memory; errors found on the device surface at the next
 * mb200_bank_check / read / query / cosine call. */
int mb200_bank_update(mb200_bank* bank, const int64_t* entity, const int64_t* key,
                      const float* inc, int64_t n, int mem);
int mb200_bank_update_f64(mb200_bank* bank, const int64_t* entity, const int64_t* key,
                          const double* inc, int64_t n, int mem);
/* The same update in the narrow wire format, for callers whose IDs fit 32 bits and whose increments are small
 * multiples of the bank's quantum (MovieLens-style data: int IDs, half-star ratings): u32 entity / key and ONE
 * BYTE per increment holding the number of quanta, increment = quanta[t] * 2^-frac_bits.  5 bytes per event over
 * PCIe for a single sketch (9 with entities) instead of 12 (20).  Same counters, bit for bit. */
int mb200_bank_update_u8(mb200_bank* bank, const uint32_t* entity, const uint32_t* key, const uint8_t* quanta,
                         int64_t n, int mem);
/* The same update for events that are already grouped by entity -- the shape the reference itself works
 * on: CosineCM.exportProfile walks ONE entity's PreferenceArray into ONE sketch (CosineCM.java:41-58).
 * row_ptr [entities + 1] (CSR: the events of entity e are [row_ptr[e], row_ptr[e+1]), row_ptr[0] = 0,
 * row_ptr[entities] = n); key / inc [n].  Skips the device-side grouping passes of mb200_bank_update. */
int mb200_bank_update_grouped(mb200_bank* bank, const int64_t* row_ptr, const int64_t* key, const float* inc,
                              int64_t n, int mem);
/* synchronise and report MB200_ERR_INEXACT / _RANGE / _BAD_ARG (entity out of range) */
int mb200_bank_check(mb200_bank* bank);

/* counters of entities [e0, e1) as the reference's doubles, out[(e-e0)][i][j] */
int mb200_bank_read(mb200_bank* bank, int64_t e0, int64_t e1, double* out, int mem);
/* the same counters as int32 quanta (counter = out * 2^-frac_bits): half the bytes of mb200_bank_read on the way
 * back to the host; MB200_ERR_RANGE if a counter does not fit 31 bits */
int mb200_bank_read_i32(mb200_bank* bank, int64_t e0, int64_t e1, int32_t* out, int mem);
/* DoubleCountMinSketch.get(key): min_i C[e][i][h_i(key)] (DoubleCountMinSketch.java:94-103) */
int mb200_bank_query(mb200_bank* bank, const int64_t* entity, const int64_t* key, int64_t n,
                     double* out, int mem);
/* DoubleCountMinSketch.cosine(a, b) for n entity pairs, FP64 (DoubleCountMinSketch.java:114-149):
 * min over rows of AB/(sqrt(AA)*sqrt(BB)), rows with zero denominator skipped, NaN if none. */
int mb200_bank_pair_cosine(mb200_bank* bank, const int64_t* ea, const int64_t* eb, int64_t n,
                           double* out, int mem);
/* same between the sketches of two banks (e.g. two single-sketch banks = two
 * DoubleCountMinSketch objects); MB200_ERR_BAD_ARG with the reference's message when widths or
 * depths differ (Preconditions.checkArgument, DoubleCountMinSketch.java:117-118). */
int mb200_bank_cross_cosine(mb200_bank* bank_a, const int64_t* ea, mb200_bank* bank_b,
                            const int64_t* eb, int64_t n, double* out, int mem);

/* ---- user-based recommendation over a bank of user sketches ------------------------------------------------ */
/* GenericUserBasedRecommender (GenericUserBasedRecommender.java:134-184) with CosineCM's point query, over the
 * neighbourhood lists of mb200_bank_cosine_topk: nb_idx / nb_sim [rows][nb_ld], nb_cnt [rows] exactly as that call
 * returns them (host or device memory, so a device-resident top-k feeds straight in).  For user row u and item i the
 * listed neighbours v != u are visited in list order:
 *   p = (float) DoubleCountMinSketch.get,  s = clamp(sim, -1, 1) (NaN stays NaN)
 *   p != 0 and s not NaN:  pref += s * (double) p  (product and sum rounded separately),  tot += s,  count++
 *   estimate = count <= 1 ? NaN : (float) (pref / tot)
 * Out-of-range user rows, neighbour indexes, counts and item_col entries are found on the device and fail the call
 * with MB200_ERR_BAD_ARG. */
/* doEstimatePreference for q (user row, itemID) pairs -> out[q] (NaN = no estimate).  The neighbourhood of query t
 * is row nb_row[t] of the nb_rows-row lists (nb_row NULL: row user[t], with nb_rows = the bank's entities). */
int mb200_bank_estimate_prefs(mb200_bank* bank, const int64_t* nb_idx, const double* nb_sim, const int32_t* nb_cnt,
                              int64_t nb_rows, int32_t nb_ld, const int64_t* user, const int64_t* nb_row,
                              const int64_t* item_id, int64_t q, float* out, int mem);
/* recommend(user, how_many) for m user rows.  Neighbourhood lists [entities][nb_ld] indexed by user row.  Data model
 * = the items each user row rated, CSR: item_ptr [entities + 1] (item_ptr[0] = 0, item_ptr[entities] = nnz),
 * item_col [nnz] dense item numbers into item_ids [num_items] (strictly ascending itemIDs).  Candidates = items of
 * the listed neighbours, minus the user's own unless include_known; NaN estimates dropped; ranked by (value desc,
 * itemID asc).  out_item / out_value [m][how_many] (unused slots -1 / 0), out_cnt [m].  how_many in [1, 1024]. */
int mb200_bank_recommend(mb200_bank* bank, const int64_t* nb_idx, const double* nb_sim, const int32_t* nb_cnt,
                         int32_t nb_ld, const int64_t* item_ptr, const int32_t* item_col, int64_t nnz,
                         const int64_t* item_ids, int64_t num_items, const int64_t* users, int64_t m, int32_t how_many,
                         int include_known, int64_t* out_item, float* out_value, int32_t* out_cnt, int mem);
/* what the last mb200_bank_recommend on the context did: users whose candidates were estimated by streaming the
 * neighbours' sketch rows through shared memory or by gathering single counters (chosen per user by bytes: rows
 * c*d*W*8 per candidate chunk against C*c*d*32), candidate chunks, candidates (sum, max), sketch rows streamed,
 * counters gathered, pipeline stages (0: rows too wide to stage) and candidates per chunk */
typedef struct mb200_recommend_plan {
  int64_t stream_users, gather_users, chunks, candidates, candidates_max, stream_rows, gather_loads;
  int32_t stages, chunk_candidates;
} mb200_recommend_plan;
int mb200_recommend_last_plan(mb200_ctx* ctx, mb200_recommend_plan* out);

/* ---- CosineCM with a CountMinSketchConfig: every user's sketch at its own (width, depth) ---------------------- */
/* The sized bank holds user u's sketch at (width[u], depth[u]) -- mb200_cm_dims(getDelta(u), getEpsilon(u)), as
 * `new DoubleCountMinSketch(delta, epsilon, hfb)` sizes it -- all users sharing one hash family a[], b[] (HOST arrays of
 * at least max(depth) entries).  The data model is CSR by user row: the prefs of row u are [user_ptr[u], user_ptr[u+1]),
 * user_ptr[0] = 0; every (item, pref) given is added (CosineCM.exportProfile).  Counters are int64 fixed point with
 * quantum 2^-frac_bits; MB200_ERR_INEXACT / _RANGE as for banks (a sketch row whose sum of squared quanta reaches
 * 2^53 is out of range too).  depth in [1, 32], width >= 1; malformed widths, depths or user_ptr fail with
 * MB200_ERR_BAD_ARG.  The bank keeps the prefs on the device: queries re-sketch users from them.  width, depth, user_ptr,
 * item and pref are in `mem`. */
typedef struct mb200_sized_bank mb200_sized_bank;
int mb200_sized_bank_create(mb200_ctx* ctx, int64_t users, const int32_t* width, const int32_t* depth, const int64_t* a,
                            const int64_t* b, int32_t frac_bits, const int64_t* user_ptr, const int64_t* item,
                            const float* pref, int mem, mb200_sized_bank** out);
int mb200_sized_bank_destroy(mb200_sized_bank* bank);
/* user row u's own sketch as the reference's doubles, HOST out[depth[u]][width[u]] */
int mb200_sized_bank_read(mb200_sized_bank* bank, int64_t user, double* out);
/* CosineCM.userSimilarity(u1[t], u2[t]) exactly as written (CosineCM.java:84-96): u1's prefs sketched at u2's
 * shape, DoubleCountMinSketch.cosine against u2's own sketch (min over rows of AB/(sqrt(AA)*sqrt(BB)), rows with a
 * zero denominator skipped, NaN if none), clamped to [-1, 1] with NaN kept.  Bit-equal to
 * mb200_bank_cross_cosine on two banks of u2's shape.  MB200_ERR_RANGE if a re-sketched row's sum of squared quanta
 * reaches 2^53 (the FP64 sums would no longer be exact). */
int mb200_sized_pair_cosine(mb200_sized_bank* bank, const int64_t* u1, const int64_t* u2, int64_t n, double* out,
                            int mem);
/* NearestNUserNeighborhood(n, min_similarity) over that similarity for the q query rows: every other user v is
 * scored as userSimilarity(query, v); NaN is never admitted, sim >= min_similarity is (negatives too: pass -INFINITY
 * for no threshold); the best n under (sim desc, user row asc) are kept.  n in [1, 1024].  out_idx / out_sim
 * [q][n] (unused slots -1 / 0), out_cnt [q] -- mb200_bank_cosine_topk's list format. */
int mb200_sized_neighborhood(mb200_sized_bank* bank, const int64_t* query_rows, int64_t q, int32_t n,
                             double min_similarity, int64_t* out_idx, double* out_sim, int32_t* out_cnt, int mem);
/* mb200_bank_estimate_prefs's contract, except that neighbour v's point query is min over v's own depth[v] rows of
 * C_v[i][h_i(item) mod width[v]] (the sketch CosineCM.getExportedCMProfile(v) caches). */
int mb200_sized_estimate_prefs(mb200_sized_bank* bank, const int64_t* nb_idx, const double* nb_sim,
                               const int32_t* nb_cnt, int64_t nb_rows, int32_t nb_ld, const int64_t* user,
                               const int64_t* nb_row, const int64_t* item_id, int64_t q, float* out, int mem);
/* what the last mb200_sized_neighborhood on the context did: queries, distinct candidate shapes (classes), classes
 * whose query sketches were built in shared memory or in a per-CTA global slice, pair FMAs of the shape model
 * (sum over classes of queries * members * depth * width), query batches, work items, the largest query tile and
 * the shared-memory budget for query sketches */
typedef struct mb200_sized_plan {
  int64_t queries, classes, smem_classes, global_classes, pair_fmas, batches, items;
  int32_t query_tile_max, smem_bytes;
} mb200_sized_plan;
int mb200_sized_last_plan(mb200_ctx* ctx, mb200_sized_plan* out);
/* recommend(user, how_many) for m user rows over per-user sketch shapes: mb200_bank_recommend's contract (the data
 * model as CSR over the bank's user rows, item_ptr [users + 1]; candidates, NaN dropped, (value desc, itemID asc)),
 * except that the neighbourhood of users[t] is row t of the lists (nb_idx / nb_sim [m][nb_ld], nb_cnt [m], as
 * mb200_sized_neighborhood returns them for users) and every estimate is mb200_sized_estimate_prefs's, bit for bit.
 * Negative similarities can make an estimate negative or infinite; it ranks by value like any other.  Out-of-range
 * user rows, counts, neighbour indexes, item_ptr ranges and item_col entries fail with MB200_ERR_BAD_ARG. */
int mb200_sized_recommend(mb200_sized_bank* bank, const int64_t* nb_idx, const double* nb_sim, const int32_t* nb_cnt,
                          int32_t nb_ld, const int64_t* item_ptr, const int32_t* item_col, int64_t nnz,
                          const int64_t* item_ids, int64_t num_items, const int64_t* users, int64_t m,
                          int32_t how_many, int include_known, int64_t* out_item, float* out_value, int32_t* out_cnt,
                          int mem);
/* what the last mb200_sized_recommend on the context did.  Per candidate chunk each listed neighbour is either
 * streamed (its whole sketch, or row by row when the sketch does not fit a stage, through a shared-memory ring) or
 * gathered (one counter per candidate and row), whichever moves fewer bytes (8*d*w against chunk*d*32); rows wider
 * than a stage are always gathered.  users, chunks, candidates (sum, max), neighbour visits streamed (row_visits:
 * those streamed row by row) / gathered (gathered includes too_wide: visits that would have streamed but did not fit
 * a stage), bytes streamed, counters gathered, neighbour terms (sum over users of candidates * listed neighbours other than the user), pipeline
 * stages, bytes per stage and candidates per chunk. */
typedef struct mb200_sized_recommend_plan {
  int64_t users, chunks, candidates, candidates_max, stream_visits, row_visits, gather_visits, too_wide_visits,
      stream_bytes, gather_loads, terms;
  int32_t stages, stage_bytes, chunk_candidates;
} mb200_sized_recommend_plan;
int mb200_sized_recommend_last_plan(mb200_ctx* ctx, mb200_sized_recommend_plan* out);

/* ---- item-based recommendation over the item top-k lists (RecommenderJob's aggregate-and-recommend phase) ---- */
/* UserVectorSplitterMapper + PartialMultiplyMapper + AggregateAndRecommendReducer of upstream RecommenderJob
 * (cf/taste/hadoop/item/), restated in DESIGN.md section 3.  For user row u:
 *   prefs equal to +-0 are not part of the user vector; with more than max_prefs_per_user (P) prefs, T = the P-th
 *   largest |pref| and only the prefs with |pref| >= T are considered (ties at T all kept);
 *   the considered prefs are visited in ascending item row j, and for every entry (i, s) of row j's list
 *     num[i] += s * (double) p_j  (product and sum rounded separately),  den[i] += |s|,  cnt[i]++
 *   (boolean_data: num[i] += s); the considered items themselves get no prediction (upstream's NaN diagonal);
 *   prediction = cnt >= 2 ? (float) (num / den) : none   (boolean_data: (float) num)
 *   predictions that are NaN or <= Float.MIN_VALUE are dropped, then the allowed-items mask; ranked by
 *   (value desc, itemID asc), the first how_many kept.
 * Every array is in the memory space `mem`.  Out-of-range list entries or counts, a malformed user_ptr, pref_row
 * entries out of range or not strictly ascending within a user, and user rows out of range are found on the device
 * and fail the call with MB200_ERR_BAD_ARG.  mb200_itembased_multi_recommend (below) returns the same bytes from all
 * GPUs of an mb200_multi, each user row computed on one of them. */
typedef struct mb200_itembased_args {
  /* the similarity matrix: row j = item j's top-k list exactly as mb200_bank_cosine_topk writes it */
  const int64_t* sim_idx;  /* [num_items][sim_ld] item rows */
  const double* sim_val;   /* [num_items][sim_ld] */
  const int32_t* sim_cnt;  /* [num_items] */
  int64_t num_items;
  int32_t sim_ld;
  /* the user vectors, CSR over user rows: prefs of row u are [user_ptr[u], user_ptr[u+1]), item rows ascending */
  const int64_t* user_ptr; /* [num_users + 1] */
  const int32_t* pref_row; /* [nnz] */
  const float* pref_val;   /* [nnz] */
  int64_t num_users, nnz;
  const int64_t* item_ids; /* [num_items] row -> itemID (output and tie rule; any order) */
  const uint32_t* allowed; /* optional [ceil(num_items / 32)] bit mask over item rows (--itemsFile); NULL = all */
  const int64_t* users;    /* [m] user rows to serve */
  int64_t m;
  int32_t how_many;            /* [1, 1024] */
  int32_t max_prefs_per_user;  /* >= 1 */
  int32_t boolean_data;
  int64_t* out_item;  /* [m][how_many] itemIDs, -1 unused */
  float* out_value;   /* [m][how_many], 0 unused */
  int32_t* out_cnt;   /* [m] */
  int32_t mem;        /* MB200_MEM_HOST or MB200_MEM_DEVICE, for every array above */
} mb200_itembased_args;
int mb200_recommend_item_based(mb200_ctx* ctx, const mb200_itembased_args* args);
/* what the last mb200_recommend_item_based on the context did: users served, users whose accumulators were an
 * open-addressing table in shared memory (smem) or dense per-CTA slices over num_items (dense) -- chosen per user
 * from B = the sum of the considered lists' counts --, list entries visited (partial products; sum and max over
 * users), users with more than max_prefs_per_user prefs (a threshold T was computed), the largest candidate count,
 * table slots per CTA and dense slices */
typedef struct mb200_itembased_plan {
  int64_t users, smem_users, dense_users, entries, entries_max, pruned_users, candidates_max;
  int32_t table_slots, dense_slices;
} mb200_itembased_plan;
int mb200_itembased_last_plan(mb200_ctx* ctx, mb200_itembased_plan* out);

/* ---- sharded ingest: events travel to the GPU that owns their row ------------------------------ */
/* Item-hash sharding (SURVEY.md 8e): owner(row) = row mod shards, local row = row div shards.  Every GPU
 * holds an arbitrary slice of the event stream in DEVICE memory.
 *   mb200_route_count    how many of these events belong to each shard (HOST counts[shards]; synchronises).
 *                        The callers exchange the shards x shards count matrix (a few hundred bytes, their
 *                        collective) so that every source knows where its region starts in every destination.
 *   mb200_route_scatter  one kernel partitions the events by owner in shared memory and writes every owner's
 *                        run straight into that GPU's receive columns: dst_row / dst_key / dst_inc are HOST
 *                        arrays of `shards` DEVICE pointers (the local columns, or a peer's mapped with
 *                        mb200_peer_alloc / mb200_peer_open), dst_offset[s] the first slot of THIS source in
 *                        destination s.  The row written is the local row.  Asynchronous on the context's
 *                        stream; the destinations may be read after a cross-GPU barrier behind it.
 * The order of the events inside a destination is unspecified (sketch updates commute). */
int mb200_route_count(mb200_ctx* ctx, const int64_t* row, int64_t n, int32_t shards, int64_t* counts);
int mb200_route_scatter(mb200_ctx* ctx, const int64_t* row, const int64_t* key, const float* inc, int64_t n,
                        int32_t shards, void* const* dst_row, void* const* dst_key, void* const* dst_inc,
                        const int64_t* dst_offset);

/* ---- ingest: text preference data -> device-resident events -> preference matrix ------------ */
/* The step in front of the sketch path (PreparePreferenceMatrixJob.java:54-114), so that the events
 * never leave the GPU between the input file and K1.
 *
 * mb200_events_parse = ToEntityPrefsMapper.map (ToEntityPrefsMapper.java:56-76) over a whole text
 * buffer: lines `userID,itemID[,pref[,...]]` split on tab or comma; Long.parseLong / Float.parseFloat
 * (+ rating_shift); pref = 1.0 when absent or boolean_data; transpose swaps the first two columns.
 * Blank lines are skipped (a deliberate leniency for trailing newlines: the reference's mapper would
 * throw NumberFormatException from Long.parseLong("")); a malformed line fails the call with MB200_ERR_BAD_ARG and a message
 * naming the Java exception and the byte offset.  Events keep the order of the lines. */
typedef struct mb200_events mb200_events;
typedef struct mb200_prefs mb200_prefs;
int mb200_events_parse(mb200_ctx* ctx, const char* text, int64_t bytes, int mem, int boolean_data,
                       float rating_shift, int transpose, mb200_events** out);
/* the same object from binary columns */
int mb200_events_create(mb200_ctx* ctx, const int64_t* user, const int64_t* item, const float* pref,
                        int64_t n, int mem, mb200_events** out);
int mb200_events_count(mb200_events* ev, int64_t* n);
/* DEVICE pointers of the columns, valid until mb200_events_destroy */
int mb200_events_columns(mb200_events* ev, int64_t** user, int64_t** item, float** pref);
/* copies to HOST arrays of mb200_events_count elements (NULL = skip the column) */
int mb200_events_read(mb200_events* ev, int64_t* user, int64_t* item, float* pref);
int mb200_events_destroy(mb200_events* ev);
/* TasteHadoopUtils.idToIndex (TasteHadoopUtils.java:56-58) for n ids */
int mb200_id_to_index(mb200_ctx* ctx, const int64_t* ids, int64_t n, int32_t* out, int mem);
/* The bookkeeping of the preparation phase: item index = idToIndex(itemID); per index the minimum
 * itemID over ALL lines (ItemIDIndexReducer.java:31-46); the last preference of a (user, index) pair
 * wins (userVector.set, ToUserVectorsReducer.java:66-82); users with fewer than min_prefs_per_user
 * distinct indexes are dropped.  The result holds the surviving events in input order with their
 * dense row number (rank of the index among the distinct indexes, ascending) -- ready for
 * mb200_bank_update(entity = row, key = user, inc = pref, MB200_MEM_DEVICE). */
int mb200_events_prepare(mb200_events* ev, int32_t min_prefs_per_user, mb200_prefs** out);
int mb200_prefs_info(mb200_prefs* p, int64_t* n, int64_t* num_items, int64_t* num_users);
int mb200_prefs_columns(mb200_prefs* p, int64_t** row, int64_t** user, float** pref); /* DEVICE */
/* DEVICE column: a dense number 0..num_users-1 per surviving event's user -- the counter column of the
 * exact measure (bank of depth 1, width num_users, hash parameters a = 1, b = 0) */
int mb200_prefs_user_columns(mb200_prefs* p, int64_t** ucol);
/* copies of the surviving events to HOST arrays of n elements each (NULL = skip the column): what a host-side
 * driver hands to mb200_job_item_similarity when the preparation ran on one GPU and the job runs on several */
int mb200_prefs_read(mb200_prefs* p, int64_t* row, int64_t* user, int64_t* ucol, float* pref);
/* HOST tables of num_items entries: row -> itemID written to the output, row -> index */
int mb200_prefs_tables(mb200_prefs* p, int64_t* item_id, int32_t* index_values);
int mb200_prefs_destroy(mb200_prefs* p);

/* ---- all-pairs cosine + per-row top-k ----------------------------------------------------- */
/* Single-GPU convenience: normalise the bank's rows (K2), compute every pair's sketch cosine
 * -- min over depth of the per-row cosines, DoubleCountMinSketch.cosine -- on the tensor cores
 * with the top-k fused into the epilogue (K3), merge / re-score (K5).  Keeps, per entity, the k
 * best under the total order (similarity desc, index asc).  Semantics of RowSimilarityJob with
 * CosineSimilarity (RowSimilarityJob.java:478-501,515-559; TopElementsQueue.java:26-59): a
 * similarity is kept iff sim >= threshold and sim > Double.MIN_VALUE; NaN (no comparable row)
 * never; the diagonal is dropped when exclude_self.  Pass threshold <= 0 for "no threshold"
 * (RowSimilarityJob.NO_THRESHOLD).
 * out_idx / out_sim are [entities][k] (unused slots: -1 / 0), out_cnt [entities]. */
int mb200_bank_cosine_topk(mb200_bank* bank, int32_t k, double threshold, int exclude_self,
                           int dtype, int precision, int64_t* out_idx, double* out_sim,
                           int32_t* out_cnt, int mem);

/* Building blocks of the item-sharded multi-GPU path (one process per GPU; the all-gather of
 * the normalised rows between the two calls is the caller's NCCL collective).  All pointers
 * are DEVICE pointers.
 *
 * Normalised rows: rows16 is [d][rows][ld] 16-bit elements, ld = mb200_row_ld(width), holding
 * x / ||x||_2 * 2^12 (F16) or x / ||x||_2 (BF16), zero padded to ld.  valid is
 * [d][mb200_valid_words(rows)] uint32 bit masks: bit e set <=> sketch row (e, depth) has a
 * non-zero norm (rows with zero denominator are skipped by the reference,
 * DoubleCountMinSketch.java:138). */
int64_t mb200_row_ld(int32_t width);
int64_t mb200_valid_words(int64_t rows);
int mb200_bank_normalize(mb200_bank* bank, int dtype, void* rows16, uint32_t* valid);
/* after mb200_bank_normalize: did K2 see a negative counter (or a row norm >= 2^36 quanta)?  Synchronises.
 * Sticky until mb200_bank_clear.  Feed the OR over all banks of a job into mb200_cosine_args.mixed_sign. */
int mb200_bank_sign_info(mb200_bank* bank, int32_t* mixed_sign);

typedef struct mb200_cosine_args {
  /* A side: the entities this GPU answers for */
  const void* a_rows;      /* [d][a_count][ld] */
  const uint32_t* a_valid; /* [d][valid_words(a_count)] */
  int64_t a_count;
  int64_t a_id_mul, a_id_off; /* global index of local row r = r * a_id_mul + a_id_off */
  /* B side: b_blocks gathered blocks of b_count rows each, block g laid out [d][b_count][ld] at
   * b_rows + g * d * b_count * ld (what all_gather_into_tensor of the shards produces) */
  const void* b_rows;
  const uint32_t* b_valid; /* [b_blocks][d][valid_words(b_count)] */
  int64_t b_count;
  int32_t b_blocks;
  int64_t b_id_mul, b_id_add; /* global index of row l of block g = l * b_id_mul + g * b_id_add */
  int32_t depth, width;
  int32_t dtype, precision;
  int32_t k;
  double threshold;
  int32_t exclude_self;
  int32_t block_n; /* 0 = auto; N tile of the tensor-core kernel (128 or 256) */
  /* MB200_PRECISION_RESCORED only: the raw fixed-point counters the candidates are re-scored
   * from, a_counters [a_count][d][width], b_counters [b_blocks][b_count][d][width] */
  const int64_t* a_counters;
  const int64_t* b_counters;
  /* outputs (device): [a_count][k], [a_count][k], [a_count] */
  int64_t* out_idx;
  double* out_sim;
  int32_t* out_cnt;
  /* debug / parity: if non-NULL the tensor-core similarities (after min over depth, NaN where no
   * row was comparable) are also written densely, [a_count][dense_ld] floats, column = position
   * of the B row (block g, row l) -> g * tiles_per_block * block_n + l */
  float* dense_out;
  int64_t dense_ld;
  /* MB200_PRECISION_CERTIFIED across GPUs: instead of one gathered b_counters array, a HOST array of
   * b_blocks DEVICE pointers, block g -> that shard's counters [b_count][d][width] (the local bank, or
   * a peer's bank mapped with mb200_bank_ipc_handle + mb200_peer_open).  Only the handful of
   * candidates the tensor values cannot decide are read through them.  NULL otherwise. */
  const int64_t* const* b_counter_blocks;
  /* optional, with b_counter_blocks: int32 copies of the same blocks (mb200_bank_narrow32 into
   * mb200_peer_alloc memory) -- the undecided candidates are then read at half the NVLink bytes; a
   * counter that does not fit is stored as INT_MIN and sends the row to the exact full-row path,
   * which reads b_counter_blocks */
  const int32_t* const* b_counter_blocks32;
  /* non-zero when any counter of the A or B side may be negative (negative increments, rating_shift) or a
   * row norm reaches 2^36 quanta -- mb200_bank_sign_info of every bank involved, OR-ed.  The tensor-core
   * values then carry an absolute instead of a relative error bound, and RESCORED / CERTIFIED widen their
   * admission threshold, certification bound and undecided band accordingly.  mb200_bank_cosine_topk
   * sets it by itself. */
  int32_t mixed_sign;
  /* mb200_cosine_finish of a job whose B side was STREAMED (several pushes; the pieces are gone): instead of sending
   * the uncertified rows through the exact full-row path, return MB200_BAND_PENDING and keep the job alive.  The
   * caller then pushes the same pieces once more -- K3 sweeps them for those rows only, with the fixed per-row cuts
   * -- and calls mb200_cosine_finish again (its arguments are ignored the second time), which completes the band
   * pass.  mb200_cosine_last_band_rows tells how many rows are waiting. */
  int32_t defer_uncertified;
} mb200_cosine_args;

int mb200_cosine_topk(mb200_ctx* ctx, const mb200_cosine_args* args);

/* Incremental form of mb200_cosine_topk: the B side arrives in pieces -- row chunks of an
 * all-gather that is still in flight (C1 overlapped with K3, SURVEY.md 8e) or peer blocks streamed
 * through a ring when the gathered rows do not fit in HBM (config 5).
 *   begin  fixes the A side and the parameters (a_*, depth, width, dtype, precision, k, threshold,
 *          exclude_self, block_n, dense_* of `args`; its b_*, *_counters and out_* are ignored).
 *   push   queues K3 for one piece on the context's stream and returns; the piece's memory may be
 *          reused once the work queued so far has completed (mb200_sync, or an event recorded by
 *          the caller on the stream it set with mb200_set_stream).  Per-row candidates and
 *          thresholds persist across pushes, so later pieces start with the bound of the earlier.
 *   finish merges, (RESCORED) re-scores and writes out_idx / out_sim / out_cnt of `fin`, then
 *          frees the job.  RESCORED needs fin->a_counters and fin->b_counters for the WHOLE B side
 *          resident, with fin->b_count / b_blocks / b_id_mul / b_id_add describing its layout.
 *   abort  frees a job without results.
 * One job per context at a time. */
typedef struct mb200_cosine_job mb200_cosine_job;
typedef struct mb200_cosine_piece {
  const void* b_rows;      /* [b_blocks][d][b_count][ld] */
  const uint32_t* b_valid; /* [b_blocks][d][valid_words(b_count)] */
  int64_t b_count;
  int32_t b_blocks;
  /* global index of row l of block g of this piece = l * b_id_mul + g * b_id_add + b_id_base */
  int64_t b_id_mul, b_id_add, b_id_base;
  /* pull-gather (see mb200_gather_pull): K3 reads block g only once ready_flags[g] == ready_epoch,
   * and sweeps the blocks starting with first_block.  NULL / 0 / 0 otherwise. */
  const uint32_t* ready_flags;
  uint32_t ready_epoch;
  int32_t first_block;
} mb200_cosine_piece;
/* The all-gather fused into K3 (C1 + K3 of SURVEY.md 8e as one kernel's worth of time): every GPU keeps
 * its normalised rows in a peer-accessible buffer; mb200_gather_pull queues, on the context's copy
 * stream, one DMA per shard from the owner's memory over NVLink into the local staging operand
 * [blocks][d][b_count][ld] (ring order; the own block is copied on the compute stream itself, ahead of
 * K3, because a copy inside one GPU may need SMs and the persistent K3 leaves none), each followed by a
 * stream memory operation that publishes the block's arrival flag.  K3 is launched at once on the compute stream
 * with the flags in its piece: its TMA producer waits for a block's flag before the first tile of
 * that block, so the transfer of block g+1 hides behind the tensor-core sweep of block g and no SM
 * is spent on communication.  The caller provides the cross-rank ordering: all ranks must have
 * finished K2 before any pull starts, and must not overwrite their rows before every peer's K3 is
 * done (two stream-ordered barriers per step, see similarity.fused_gather_cosine).
 *   mb200_peer_alloc   cudaMalloc + a 64-byte IPC handle to send to the other ranks
 *   mb200_peer_open    map a peer's buffer from its handle (once; mappings persist)
 *   mb200_gather_wait  block until the queued pulls are complete */
int mb200_peer_alloc(mb200_ctx* ctx, int64_t bytes, void** ptr, void* ipc_handle_64_bytes);
int mb200_peer_open(mb200_ctx* ctx, const void* ipc_handle_64_bytes, void** ptr);
int mb200_peer_close(mb200_ctx* ctx, void* ptr);
int mb200_peer_free(mb200_ctx* ctx, void* ptr);
int mb200_gather_pull(mb200_ctx* ctx, void* staging_rows, uint32_t* staging_valid,
                      const void* const* peer_rows, const uint32_t* const* peer_valid, int32_t blocks,
                      int32_t my_block, int64_t rows_bytes_per_block, int64_t valid_bytes_per_block,
                      const uint32_t** ready_flags, uint32_t* epoch);
int mb200_gather_wait(mb200_ctx* ctx);
/* Copies of the peers' int32 counter banks (mb200_bank_narrow32) for MB200_PRECISION_CERTIFIED, when they fit the
 * local memory: queued on the copy stream BEHIND the row pulls (call after mb200_gather_pull), one DMA per peer
 * block dst_blocks[g] <- src_blocks[g] (g != my_block), in ring order.  The undecided candidates of k_certify and
 * of the band pass are then read from local HBM instead of one NVLink round trip per row of counters -- the same
 * peer rows are wanted by thousands of local rows (measured at 2 GPUs, 125000 x 250000, depth 4: k_certify
 * 222-272 ms through the peer mappings, 46 ms on one GPU with half the columns).
 *   mb200_gather_fence  the compute stream waits (on the device) for everything queued on the copy stream so far */
int mb200_gather_pull_counters(mb200_ctx* ctx, void* const* dst_blocks, const void* const* src_blocks,
                               int32_t blocks, int32_t my_block, int64_t bytes_per_block);
int mb200_gather_fence(mb200_ctx* ctx);
int mb200_cosine_begin(mb200_ctx* ctx, const mb200_cosine_args* args, mb200_cosine_job** job);
int mb200_cosine_push(mb200_cosine_job* job, const mb200_cosine_piece* piece);
int mb200_cosine_finish(mb200_cosine_job* job, const mb200_cosine_args* fin);
int mb200_cosine_abort(mb200_cosine_job* job);
/* rows whose top-k could not be certified from the tensor-core candidates during the last mb200_cosine_topk /
 * mb200_cosine_finish / mb200_bank_cosine_topk on ctx.  They first get a BAND PASS: a second K3 sweep over those rows
 * only, with a fixed per-row cut below which no column can be in the top-k, every column above it re-scored exactly
 * (needs the B side of a one-push job still resident: pass b_rows / b_valid again in the finish arguments; the
 * one-shot calls do).  What the band pass cannot settle -- counters outside the exact-integer range, tie groups
 * beyond 2048 columns, or no band pass possible -- takes the exact full-row path (every column, integer dot
 * products at memory speed): mb200_cosine_last_fallback_rows. */
int mb200_cosine_last_band_rows(mb200_ctx* ctx, int64_t* rows);
int mb200_cosine_last_fallback_rows(mb200_ctx* ctx, int64_t* rows);

/* ---- the whole item-similarity phase, on one GPU or on all GPUs of the box ------------------------------- */
/* One process drives n_gpus GPUs: one mb200_ctx and one host worker thread per GPU, peer access between all of
 * them (SURVEY.md 8b: `mb200_create(int n_gpus, ...)`).  devices may be NULL (GPUs 0 .. n_gpus-1); n_gpus == 0
 * takes every visible GPU.  An explicit list may name a device more than once: that device gets one context per
 * entry (no peer access is needed between them), and n_gpus is bounded by MB200_MAX_BLOCKS, not by the visible
 * GPUs.  This is what a JVM binds for `--numGpus`. */
typedef struct mb200_multi mb200_multi;
int mb200_create_multi(int32_t n_gpus, const int32_t* devices, mb200_multi** out);
int mb200_multi_destroy(mb200_multi* m);
int mb200_multi_gpus(mb200_multi* m, int32_t* n_gpus);
int mb200_multi_ctx(mb200_multi* m, int32_t g, mb200_ctx** out); /* GPU g's context (owned by m) */
const char* mb200_multi_last_error(mb200_multi* m);

typedef struct mb200_job_params {
  int32_t k;          /* --maxSimilaritiesPerItem (ItemSimilarityJob.java:88,105) */
  double threshold;   /* --threshold; <= 0 = RowSimilarityJob.NO_THRESHOLD */
  int32_t width, depth;
  int64_t seed;       /* HashFunctionBuilder seed ... */
  const int64_t* hash_a; /* ... or explicit parameters [depth] (both NULL = from seed); a = 1, b = 0 with width = */
  const int64_t* hash_b; /*     number of users and dense user numbers as keys is the exact measure          */
  int32_t frac_bits;
  int32_t dtype;      /* MB200_DTYPE_* */
  int32_t precision;  /* MB200_PRECISION_* */
} mb200_job_params;

typedef struct mb200_job_stats {
  int32_t n_gpus;
  int64_t events;              /* USED_OBSERVATIONS of RowSimilarityJob.Counters (RowSimilarityJob.java:84) */
  int64_t rows;                /* ROWS */
  int64_t similarities_kept;   /* entries written over all rows (<= rows * k) */
  int64_t fallback_rows;       /* rows that took the exact full-row path */
  int64_t events_busiest_gpu;  /* events received by the fullest shard */
  double route_s, build_s, cosine_s; /* host wall clock of the three stages (GPU 0's worker) */
} mb200_job_stats;

/* Phase 1 of ItemSimilarityJob.run (ItemSimilarityJob.java:146-162) for prepared events in HOST memory: dense item
 * rows [0, num_items), keys (user IDs, or dense user numbers for the exact measure), preferences.  Items are
 * sharded by row mod n_gpus; events are routed to their owners over NVLink, every GPU builds its shard's
 * sketches (K1), normalises (K2) and computes its block row of the similarity matrix against the rows pulled
 * from its peers (K3, top-k fused) -- see csrc/job.cu.  out_idx / out_sim are [num_items][k] in global row
 * order (unused slots -1 / 0), out_cnt [num_items]; stats may be NULL.  RESCORED pulls the peers' counters
 * whole (n_gpus x the shard bank per GPU); CERTIFIED reads only the undecided candidates remotely. */
int mb200_job_item_similarity(mb200_multi* m, const int64_t* row, const int64_t* key, const float* inc, int64_t n,
                              int64_t num_items, const mb200_job_params* p, int64_t* out_idx, double* out_sim,
                              int32_t* out_cnt, mb200_job_stats* stats);

/* ---- CosineCM with a CountMinSketchConfig on all GPUs of m: one sized-bank replica per GPU --------------------- */
/* mb200_sized_multi_create builds one full mb200_sized_bank on every GPU of m, all GPUs in parallel, from the same
 * HOST arrays (mb200_sized_bank_create's meaning).  Each replica costs what one sized bank costs: counters
 * (cells + 2) * 8 B, sums of squares rows * 8 B, quanta nnz * 8 B, hash residues nnz * max(depth) * 8 B, and 36 B per
 * user of shapes and offsets.  The calls below take and return HOST arrays in the caller's order and split the work
 * by user: query position t goes to GPU t mod G; estimates go by user, the j-th distinct user row (ascending) to GPU
 * j mod G with every pair of that user.  Results are bit-identical to the single-context calls for any G (floats,
 * NaN slots, counts, unused slots -1 / 0).  NULL arrays, q or m < 0, n outside [1, 1024], how_many outside [1, 1024],
 * a NaN min_similarity or a malformed item CSR fail with MB200_ERR_BAD_ARG before any GPU work; a device-found error
 * fails the call with the first failing GPU's code and "GPU d: <message>" (mb200_multi_last_error).  The handle stays
 * usable after a failed call.  One call at a time per mb200_multi: every call holds m's lock. */
typedef struct mb200_sized_multi mb200_sized_multi;
int mb200_sized_multi_create(mb200_multi* m, int64_t users, const int32_t* width, const int32_t* depth,
                             const int64_t* a, const int64_t* b, int32_t frac_bits, const int64_t* user_ptr,
                             const int64_t* item, const float* pref, mb200_sized_multi** out);
int mb200_sized_multi_destroy(mb200_sized_multi* sm);
/* mb200_sized_neighborhood's contract: out_idx / out_sim [q][n], out_cnt [q] */
int mb200_sized_multi_neighborhood(mb200_sized_multi* sm, const int64_t* query_rows, int64_t q, int32_t n,
                                   double min_similarity, int64_t* out_idx, double* out_sim, int32_t* out_cnt);
/* recommend(user, how_many) for the m user rows: each GPU computes its users' neighbourhoods (n, min_similarity)
 * and runs mb200_sized_recommend over them; the lists never leave that GPU.  The data model as there: item_ptr
 * [users + 1], item_col [nnz], item_ids [num_items] strictly ascending.  out_item / out_value [m][how_many],
 * out_cnt [m]. */
int mb200_sized_multi_recommend(mb200_sized_multi* sm, const int64_t* users, int64_t m, int32_t n,
                                double min_similarity, const int64_t* item_ptr, const int32_t* item_col, int64_t nnz,
                                const int64_t* item_ids, int64_t num_items, int32_t how_many, int include_known,
                                int64_t* out_item, float* out_value, int32_t* out_cnt);
/* doEstimatePreference for the q pairs (user[t], item_id[t]) over each user's neighbourhood (n, min_similarity),
 * each distinct user's neighbourhood computed once: mb200_sized_estimate_prefs's values, float32 out [q] */
int mb200_sized_multi_estimate_prefs(mb200_sized_multi* sm, const int64_t* user, const int64_t* item_id, int64_t q,
                                     int32_t n, double min_similarity, float* out);
/* the last call on sm (create included): work[g] = queries (pairs for estimates, users for create) given to GPU g,
 * seconds[g] = host wall clock of GPU g's worker, wall_s = the call's wall clock.  work and seconds have
 * mb200_multi_gpus entries; any pointer may be NULL. */
int mb200_sized_multi_last_stats(mb200_sized_multi* sm, int64_t* work, double* seconds, double* wall_s);

/* ---- item-based recommendation on all GPUs of m: one replica of the lists and user vectors per GPU ------------ */
/* mb200_itembased_multi_create copies the item top-k lists (sim_idx / sim_val [num_items][sim_ld], sim_cnt
 * [num_items]), the user CSR (user_ptr [num_users + 1], pref_row / pref_val [nnz]) and item_ids [num_items], all HOST
 * arrays with mb200_itembased_args' meaning, to every GPU of m once, all GPUs in parallel: num_items * (16 * sim_ld +
 * 12) + 8 * nnz + 8 * (num_users + 1) bytes per GPU.  The replicas live until destroy.
 * mb200_itembased_multi_recommend serves the m user rows `users` (HOST) with mb200_recommend_item_based's
 * semantics: query position t goes to GPU t mod G, each GPU uploads only its share of the users and the allowed mask
 * (optional HOST [ceil(num_items / 32)] words, NULL = all items), and out_item / out_value [m][how_many], out_cnt [m]
 * (HOST) are exactly what mb200_recommend_item_based on one context returns for the same arguments -- values,
 * itemIDs, counts and the -1 / 0 fill of unused slots, byte for byte, for any G, either accumulator path, with and
 * without boolean_data and allowed.  Repeated calls of the same or a smaller shape allocate no device memory.
 * NULL arrays, m < 0, how_many outside [1, 1024], max_prefs_per_user < 1 and bad shapes fail with
 * MB200_ERR_BAD_ARG before any GPU work; an error found on a device (a user row out of range, a malformed CSR or
 * list) fails the call with the first failing GPU's code and "GPU d: <message>" (mb200_multi_last_error).  The
 * handle stays usable after a failed call.  One call at a time per mb200_multi: every call holds m's lock.
 * mb200_itembased_multi_last_stats: the last call on h (create included): work[g] = users given to GPU g (every
 * user for create), seconds[g] = host wall clock of GPU g's worker, wall_s = the call's wall clock; GPU g's plan is
 * mb200_itembased_last_plan of mb200_multi_ctx(m, g).  Any pointer may be NULL. */
typedef struct mb200_itembased_multi mb200_itembased_multi;
int mb200_itembased_multi_create(mb200_multi* m, const int64_t* sim_idx, const double* sim_val, const int32_t* sim_cnt,
                                 int64_t num_items, int32_t sim_ld, const int64_t* user_ptr, const int32_t* pref_row,
                                 const float* pref_val, int64_t num_users, int64_t nnz, const int64_t* item_ids,
                                 mb200_itembased_multi** out);
int mb200_itembased_multi_recommend(mb200_itembased_multi* h, const int64_t* users, int64_t m, int32_t how_many,
                                    int32_t max_prefs_per_user, int32_t boolean_data, const uint32_t* allowed,
                                    int64_t* out_item, float* out_value, int32_t* out_cnt);
int mb200_itembased_multi_last_stats(mb200_itembased_multi* h, int64_t* work, double* seconds, double* wall_s);
int mb200_itembased_multi_destroy(mb200_itembased_multi* h);

#ifdef __cplusplus
}
#endif
#endif /* MAHOUT_B200_H */
