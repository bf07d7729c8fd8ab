"""CosineCM -- the fork's sketch-based UserSimilarity, over the GPU sketch bank.

Mirrors cf/taste/impl/similarity/CosineCM.java: one count-min sketch per user built from the
user's preferences (key = itemID, increment = preference value, CosineCM.java:41-58), similarity
= DoubleCountMinSketch.cosine clamped to [-1, 1] (CosineCM.java:84-96 ->
AbstractSimilarity.normalizeWeightResult, AbstractSimilarity.java:313-330, unweighted), plus the
point-query consumer of GenericUserBasedRecommender.doEstimatePreference (:139-159).

The reference sizes u1's sketch by u2's (delta, epsilon) on every call and rebuilds it each time.
`userSimilarity` lets all users share one (width, depth) -- what BASELINE.json's configurations fix -- and
builds every profile once, in one K1 launch.  With a CountMinSketchConfig (SURVEY.md 8f-4),
`userSimilaritiesPerUserConfig` follows the reference's per-pair sizing on a SizedBank: every user's sketch
at its own cm_dims(getDelta(u), getEpsilon(u)), u1 re-sketched on the device at u2's shape.
"""
from __future__ import annotations

import math

import numpy as np

from . import sketch as sk


class CosineCM:
    def __init__(self, user, item, pref, width_or_delta=4096, depth_or_epsilon=4,
                 hfBuilder: sk.HashFunctionBuilder | int = 42, frac_bits: int = 1, ctx=None, config=None):
        """config: a configured CountMinSketchConfig -> `userSimilarityPerUserConfig` follows the reference's
        per-pair sizing (u1's sketch rebuilt with u2's (delta, epsilon), CosineCM.java:84-96)."""
        user = np.asarray(user, np.int64)
        self.config = config
        self._sized = None
        self._hfb = hfBuilder if isinstance(hfBuilder, sk.HashFunctionBuilder) else sk.HashFunctionBuilder(int(hfBuilder))
        self._frac_bits, self._ctx = frac_bits, ctx
        order = np.argsort(user, kind="stable")
        self._u_sorted = user[order]
        self._i_sorted = np.asarray(item, np.int64)[order]
        self._p_sorted = np.asarray(pref, np.float64)[order]
        if isinstance(width_or_delta, float) or isinstance(depth_or_epsilon, float):
            try:
                w, d = sk.cm_dims(float(width_or_delta), float(depth_or_epsilon))
            except sk.N.CMException as e:        # CosineCM.java:45-47 wraps it in a TasteException
                raise RuntimeError(f"CountMinSketch error:{e}") from e
        else:
            w, d = int(width_or_delta), int(depth_or_epsilon)
        self.user_ids = np.unique(user)
        self._row = np.searchsorted(self.user_ids, user)
        self.bank = sk.SketchBank(self.user_ids.shape[0], w, d, self._hfb, frac_bits, ctx)
        self.bank.update(self._row, np.asarray(item, np.int64), np.asarray(pref, np.float32))
        self.bank.check()

    def _rows(self, ids):
        ids = np.atleast_1d(np.asarray(ids, np.int64))
        r = np.searchsorted(self.user_ids, ids)
        ok = (r < self.user_ids.shape[0])
        ok[ok] = self.user_ids[r[ok]] == ids[ok]
        if not ok.all():
            raise KeyError(f"NoSuchUserException: {ids[~ok][:5].tolist()}")
        return r.astype(np.int64)

    def userSimilarity(self, userID1: int, userID2: int) -> float:
        return float(self.userSimilarities([userID1], [userID2])[0])

    def userSimilarities(self, ids1, ids2) -> np.ndarray:
        r = self.bank.pair_cosine(self._rows(ids1), self._rows(ids2))
        # normalizeWeightResult(result, 1, 0) for the non-NaN results: clamp to [-1, 1]
        return np.where(np.isnan(r), r, np.clip(r, -1.0, 1.0))

    def _prefs_of(self, userID: int):
        lo, hi = np.searchsorted(self._u_sorted, [userID, userID + 1])
        if lo == hi:
            raise KeyError(f"NoSuchUserException: {userID}")
        return self._i_sorted[lo:hi], self._p_sorted[lo:hi]

    def exportProfile(self, userID: int, delta: float, epsilon: float) -> sk.DoubleCountMinSketch:
        """CosineCM.exportProfile (:41-58): a fresh sketch of the user's preferences sized by (delta, epsilon)"""
        try:
            cm = sk.DoubleCountMinSketch(float(delta), float(epsilon), self._hfb, self._frac_bits, self._ctx)
        except sk.N.CMException as e:
            raise RuntimeError(f"CountMinSketch error:{e}") from e
        items, prefs = self._prefs_of(userID)
        cm.update(items, prefs)
        return cm

    def sized_model(self):
        """the inputs of a sized bank, host arrays: every user row's (width, depth) from `config`, shaped as `new
        DoubleCountMinSketch(delta, epsilon, hfb)` shapes it (cm_dims of the stored parameters, never best_dims),
        and the prefs as CSR by user row -- (width [U] int32, depth [U] int32, user_ptr [U+1], item, pref float32)"""
        if self.config is None:
            raise ValueError("no CountMinSketchConfig was given")
        dims = {}
        w = np.empty(self.user_ids.shape[0], np.int32)
        d = np.empty(self.user_ids.shape[0], np.int32)
        for r, u in enumerate(self.user_ids.tolist()):
            key = (self.config.getDelta(u), self.config.getEpsilon(u))
            if key not in dims:
                try:
                    dims[key] = sk.cm_dims(*key)
                except sk.N.CMException as e:    # CosineCM.java:45-47 wraps it in a TasteException
                    raise RuntimeError(f"CountMinSketch error:{e}") from e
            w[r], d[r] = dims[key]
        ptr = np.zeros(self.user_ids.shape[0] + 1, np.int64)
        np.cumsum(np.bincount(np.searchsorted(self.user_ids, self._u_sorted), minlength=self.user_ids.shape[0]),
                  out=ptr[1:])
        return w, d, ptr, self._i_sorted, self._p_sorted.astype(np.float32)

    def sized_bank(self) -> sk.SizedBank:
        """every user's sketch at its own (delta, epsilon) from `config` (sized_model); built on first use"""
        if self._sized is None:
            w, d, ptr, item, pref = self.sized_model()
            self._sized = sk.SizedBank(w, d, self._hfb, ptr, item, pref, self._frac_bits, self.bank.ctx)
        return self._sized

    def multi_sized_bank(self, multi):
        """sized_bank() replicated on every GPU of a MultiGpu (mahout_b200.multi.MultiSizedBank)"""
        w, d, ptr, item, pref = self.sized_model()
        return multi.sized_bank(w, d, self._hfb, ptr, item, pref, self._frac_bits)

    def userSimilaritiesPerUserConfig(self, ids1, ids2) -> np.ndarray:
        """CosineCM.userSimilarity exactly as written (:84-96) for the pairs (ids1[t], ids2[t]): user 1's prefs
        sketched at user 2's size, compared with user 2's own sketch, clamped to [-1, 1] (NaN kept)."""
        return self.sized_bank().pair_cosine(self._rows(ids1), self._rows(ids2))

    def userSimilarityPerUserConfig(self, userID1: int, userID2: int) -> float:
        """one pair of userSimilaritiesPerUserConfig"""
        return float(self.userSimilaritiesPerUserConfig([userID1], [userID2])[0])

    def doEstimatePreference(self, theUserID: int, theNeighborhood, itemID: int) -> float:
        """GenericUserBasedRecommender.doEstimatePreference with the sketch point query (:134-184): one batched pair
        cosine for the neighbours' similarities, then one query of mb200_bank_estimate_prefs over the neighbourhood
        (same accumulation order as the Java loop); NaN unless at least two neighbours contribute."""
        nb = np.asarray([u for u in np.atleast_1d(theNeighborhood) if u != theUserID], np.int64)
        if np.atleast_1d(theNeighborhood).shape[0] == 0 or nb.shape[0] == 0:
            return math.nan
        rows = self._rows(nb)
        u = self._rows(theUserID)
        sims = self.bank.pair_cosine(np.full(nb.shape[0], u[0], np.int64), rows)   # clamped on the device
        out = self.bank.estimate_prefs(rows[None, :], sims[None, :], np.array([nb.shape[0]], np.int32), u,
                                       np.array([itemID], np.int64), nb_row=np.zeros(1, np.int64))
        return float(out[0])

    def getExportedCMProfile(self, userID: int) -> np.ndarray:
        r = int(self._rows(userID)[0])
        return self.bank.read(r, r + 1)[0]

    def estimatePreference(self, userID: int, itemID: int) -> float:
        """GenericUserBasedRecommender.doEstimatePreference's sketch read: (float) cm.get(itemID),
        where 0.0 means "no preference" (NaN)."""
        v = float(np.float32(self.bank.query(self._rows(userID), np.array([itemID], np.int64))[0]))
        return math.nan if v == 0.0 else v

    def mostSimilarUserIDs(self, userID: int, howMany: int):
        """nearest users under the sketch cosine (ties: lower user index first)."""
        idx, sim, cnt = self.bank.cosine_topk(howMany)
        r = int(self._rows(userID)[0])
        return self.user_ids[idx[r, :cnt[r]]], sim[r, :cnt[r]]

    def close(self):
        if self._sized is not None:
            self._sized.close()
        self.bank.close()
