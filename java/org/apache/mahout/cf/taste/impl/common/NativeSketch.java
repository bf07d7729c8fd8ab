/*
 * JNI surface of libmahout_b200.so for the sketch-similarity hot path.  One Java `native` method per
 * C-ABI entry point of include/mahout_b200.h; jni/mahout_b200_jni.c is the 1:1 glue.
 *
 * NOT COMPILED IN THIS REPOSITORY: the build image has no JDK (no javac, no jni.h).  The file is
 * the binding a maintainer adds to the reference tree (mr/src/main/java/...); see INTEGRATION.md.
 */
package org.apache.mahout.cf.taste.impl.common;

import java.nio.ByteBuffer;

public final class NativeSketch {

  static {
    // resolved through -Djava.library.path, which bin/mahout already derives from $JAVA_LIBRARY_PATH
    // (bin/mahout:338-340); same loading convention as the ViennaCL backend (Context.scala:61-65)
    System.loadLibrary("mahout_b200_jni");
  }

  private NativeSketch() { }

  public static final int MEM_HOST = 0;
  public static final int DTYPE_F16 = 0;
  public static final int DTYPE_BF16 = 1;
  public static final int PRECISION_TENSOR = 0;
  public static final int PRECISION_RESCORED = 1;
  public static final int PRECISION_CERTIFIED = 2;
  /** words of the stats array of jobItemSimilarity: gpus, events, rows, similarities kept, fallback rows,
   *  events on the busiest GPU, route / build / cosine milliseconds */
  public static final int JOB_STATS_WORDS = 9;

  public static int precisionOf(String name) {
    if ("tensor".equals(name)) {
      return PRECISION_TENSOR;
    }
    if ("certified".equals(name)) {
      return PRECISION_CERTIFIED;
    }
    if ("rescored".equals(name)) {
      return PRECISION_RESCORED;
    }
    throw new IllegalArgumentException("--precision must be rescored, certified or tensor");
  }

  /** mb200_create / mb200_destroy: returns the opaque context handle. Throws if there is no B200. */
  public static native long createContext(int device);
  public static native void destroyContext(long ctx);

  /** mb200_hash_params: a[i], b[i] of HashFunctionBuilder(seed) (HashFunctionBuilder.java:40-60). */
  public static native void hashParams(long seed, int depth, long[] a, long[] b);

  /** mb200_cm_dims: throws AbstractCountMinSketch.CMException-compatible IllegalArgumentException. */
  public static native int[] cmDims(double delta, double epsilon);

  /** mb200_bank_create_params / mb200_bank_destroy / mb200_bank_clear */
  public static native long createBank(long ctx, long entities, int depth, int width, long[] a, long[] b,
                                       int fracBits);
  public static native void destroyBank(long bank);
  public static native void clearBank(long bank);

  /**
   * mb200_bank_update: direct buffers over pinned memory (allocPinned) hold little-endian
   * int64 entity / int64 key / float32 increment arrays; entity may be null for a single sketch.
   */
  public static native void update(long bank, ByteBuffer entity, ByteBuffer key, ByteBuffer inc, long n);
  public static native void updateOne(long bank, long entity, long key, double inc);
  public static native void check(long bank);

  /** mb200_bank_query: DoubleCountMinSketch.get (DoubleCountMinSketch.java:94-103). */
  public static native double query(long bank, long entity, long key);
  public static native void queryMany(long bank, long[] entity, long[] key, double[] out);

  /** mb200_bank_read: counters of entities [e0, e1) as doubles, out[(e - e0)][i][j]. */
  public static native void read(long bank, long e0, long e1, double[] out);

  /** mb200_bank_cross_cosine: DoubleCountMinSketch.cosine (DoubleCountMinSketch.java:114-149). */
  public static native double cosine(long bankA, long entityA, long bankB, long entityB);

  /**
   * mb200_bank_cosine_topk: RowSimilarityJob semantics with the sketch cosine; outIdx / outSim are
   * [entities][k], outCnt [entities].
   */
  public static native void cosineTopK(long bank, int k, double threshold, boolean excludeSelf, int dtype,
                                       int precision, long[] outIdx, double[] outSim, int[] outCnt);

  /**
   * Ingest on the GPU.  parsePrefs = ToEntityPrefsMapper.map over one text split held in a direct
   * buffer (ToEntityPrefsMapper.java:56-76); prepare = idToIndex + ItemIDIndexReducer +
   * ToUserVectorsReducer (last pref of a (user, index) pair wins, minPrefsPerUser); updateFromPrefs feeds
   * the prepared, still device-resident events to mb200_bank_update (entity = matrix row, key = userID).
   */
  public static native long parsePrefs(long ctx, ByteBuffer text, long bytes, boolean booleanData, float ratingShift,
                                       boolean transpose);
  public static native long eventCount(long events);
  public static native void destroyEvents(long events);
  public static native long prepare(long events, int minPrefsPerUser);
  public static native void prefsInfo(long prefs, long[] info);
  public static native void prefsTables(long prefs, long[] itemId, int[] indexValues);
  public static native void updateFromPrefs(long bank, long prefs);
  public static native void destroyPrefs(long prefs);

  /**
   * mb200_create_multi / mb200_multi_destroy / mb200_job_item_similarity: phase 1 of ItemSimilarityJob.run
   * (ItemSimilarityJob.java:146-162) as one call over numGpus GPUs of this process (0 = all).  row / key / value are
   * the prepared events (dense rows, user keys, preferences); exactMeasure selects the identity hash family (one
   * counter column per key, width = number of distinct keys).  outIdx / outSim are [numRows][k], outCnt [numRows].
   */
  public static native long createMulti(int numGpus);
  public static native void destroyMulti(long multi);
  public static native void jobItemSimilarity(long multi, long[] row, long[] key, float[] value, long numRows, int k,
                                              double threshold, int width, int depth, long seed, boolean exactMeasure,
                                              int fracBits, int dtype, int precision, long[] outIdx, double[] outSim,
                                              int[] outCnt, long[] stats);

  /** mb200_bank_update_u8: the narrow wire format (uint32 entity / key, one byte of quanta per event). */
  public static native void updateU8(long bank, ByteBuffer entity, ByteBuffer key, ByteBuffer quanta, long n);

  /**
   * mb200_bank_estimate_prefs: GenericUserBasedRecommender.doEstimatePreference (GenericUserBasedRecommender.java:
   * 134-184) with the sketch point query for the (user row, itemID) pairs user[t], itemId[t] over the neighbourhood
   * lists of cosineTopK (nbIdx / nbSim [rows][nbLd], nbCnt [rows]); out[t] is NaN where there is no estimate.
   */
  public static native void estimatePrefs(long bank, long[] nbIdx, double[] nbSim, int[] nbCnt, int nbLd, long[] user,
                                          long[] itemId, float[] out);

  /**
   * mb200_bank_recommend: GenericUserBasedRecommender.recommend(userID, howMany) for the user rows `users`.  The data
   * model is CSR over user rows: itemPtr [rows + 1], itemCol = dense item numbers into itemIds (ascending itemIDs).
   * outItem / outValue are [users][howMany] (unused -1 / 0), outCnt [users].
   */
  public static native void recommend(long bank, long[] nbIdx, double[] nbSim, int[] nbCnt, int nbLd, long[] itemPtr,
                                      int[] itemCol, long[] itemIds, long[] users, int howMany, boolean includeKnown,
                                      long[] outItem, float[] outValue, int[] outCnt);

  /**
   * mb200_recommend_item_based: RecommenderJob's aggregate-and-recommend phase (UserVectorSplitterMapper,
   * PartialMultiplyMapper, AggregateAndRecommendReducer) for the user rows `users`.  The similarity matrix is the
   * item top-k lists of cosineTopK (simIdx / simVal [items][simLd], simCnt [items]); the user vectors are CSR over
   * user rows: userPtr [users + 1], prefRow = item rows ascending within a user, prefVal.  itemIds maps rows to
   * itemIDs; allowed is an optional bit mask over item rows (null = every item).  outItem / outValue are
   * [users][howMany] (unused -1 / 0), outCnt [users].
   */
  public static native void recommendItemBased(long ctx, long[] simIdx, double[] simVal, int[] simCnt, int simLd,
                                               long[] userPtr, int[] prefRow, float[] prefVal, long[] itemIds,
                                               int[] allowed, long[] users, int howMany, int maxPrefsPerUser,
                                               boolean booleanData, long[] outItem, float[] outValue, int[] outCnt);

  /**
   * mb200_sized_bank_create: CosineCM with a CountMinSketchConfig -- user row u's sketch at (width[u], depth[u]) =
   * the (w, d) of new DoubleCountMinSketch(getDelta(u), getEpsilon(u), hfb), all users sharing the hash parameters
   * a / b (hashParams for the largest depth).  The data model is CSR by user row: userPtr [users + 1], item / pref.
   */
  public static native long createSizedBank(long ctx, int[] width, int[] depth, long[] a, long[] b, int fracBits,
                                            long[] userPtr, long[] item, float[] pref);
  public static native void destroySizedBank(long sizedBank);

  /** mb200_sized_pair_cosine: CosineCM.userSimilarity(u1[t], u2[t]) (u1 re-sketched at u2's size), clamped. */
  public static native void sizedPairCosine(long sizedBank, long[] u1, long[] u2, double[] out);

  /**
   * mb200_sized_neighborhood: NearestNUserNeighborhood(n, minSimilarity) over that similarity for the user rows
   * queryRows (Double.NEGATIVE_INFINITY = no threshold).  outIdx / outSim are [queries][n] (unused -1 / 0), outCnt
   * [queries].
   */
  public static native void sizedNeighborhood(long sizedBank, long[] queryRows, int n, double minSimilarity,
                                              long[] outIdx, double[] outSim, int[] outCnt);

  /**
   * mb200_sized_estimate_prefs: doEstimatePreference for the (user row, itemID) pairs user[t], itemId[t] over the
   * lists of sizedNeighborhood (row nbRow[t] of them; nbRow null = row user[t]), each neighbour point-queried in its
   * own sketch; out[t] is NaN where there is no estimate.
   */
  public static native void sizedEstimatePrefs(long sizedBank, long[] nbIdx, double[] nbSim, int[] nbCnt, int nbLd,
                                               long[] user, long[] nbRow, long[] itemId, float[] out);

  /**
   * mb200_sized_recommend: GenericUserBasedRecommender.recommend(userID, howMany) over the per-user sketch sizes for
   * the user rows `users`.  Row t of the lists (nbIdx / nbSim [users][nbLd], nbCnt [users], as sizedNeighborhood
   * returns them for `users`) is users[t]'s neighbourhood, and every estimate is sizedEstimatePrefs's.  The data
   * model is CSR over user rows: itemPtr [rows + 1], itemCol = dense item numbers into itemIds (ascending itemIDs).
   * outItem / outValue are [users][howMany] (unused -1 / 0), outCnt [users].
   */
  public static native void sizedRecommend(long sizedBank, long[] nbIdx, double[] nbSim, int[] nbCnt, int nbLd,
                                           long[] itemPtr, int[] itemCol, long[] itemIds, long[] users, int howMany,
                                           boolean includeKnown, long[] outItem, float[] outValue, int[] outCnt);

  /**
   * mb200_sized_multi_create / mb200_sized_multi_destroy: createSizedBank's inputs, one replica of the sized bank on
   * every GPU of a createMulti handle (--numGpus), built in parallel.  The calls below split their users between the
   * GPUs (query position t to GPU t mod G; estimates by distinct user) and return what the single-GPU calls return,
   * bit for bit, in the caller's order.  Destroy the sized handle before its multi handle.
   */
  public static native long createSizedMulti(long multi, int[] width, int[] depth, long[] a, long[] b, int fracBits,
                                             long[] userPtr, long[] item, float[] pref);
  public static native void destroySizedMulti(long sizedMulti);

  /** mb200_sized_multi_neighborhood: sizedNeighborhood over all GPUs; outIdx / outSim [queries][n], outCnt [queries]. */
  public static native void sizedMultiNeighborhood(long sizedMulti, long[] queryRows, int n, double minSimilarity,
                                                   long[] outIdx, double[] outSim, int[] outCnt);

  /**
   * mb200_sized_multi_recommend: each user's sizedNeighborhood(n, minSimilarity), then sizedRecommend over it on the
   * GPU that computed it (the lists never leave that GPU).  outItem / outValue [users][howMany], outCnt [users].
   */
  public static native void sizedMultiRecommend(long sizedMulti, long[] users, int n, double minSimilarity,
                                                long[] itemPtr, int[] itemCol, long[] itemIds, int howMany,
                                                boolean includeKnown, long[] outItem, float[] outValue, int[] outCnt);

  /**
   * mb200_sized_multi_estimate_prefs: doEstimatePreference for the (user row, itemID) pairs user[t], itemId[t] over
   * each user's sizedNeighborhood(n, minSimilarity), each distinct user's computed once; out[t] NaN = no estimate.
   */
  public static native void sizedMultiEstimatePrefs(long sizedMulti, long[] user, long[] itemId, int n,
                                                    double minSimilarity, float[] out);

  /** mb200_host_alloc / mb200_host_free wrapped as a direct ByteBuffer. */
  public static native ByteBuffer allocPinned(long bytes);
  public static native void freePinned(ByteBuffer buffer);
}
