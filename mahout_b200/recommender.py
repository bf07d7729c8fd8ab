"""GenericUserBasedRecommender over CosineCM's user sketches, on the GPU.

Mirrors cf/taste/impl/recommender/GenericUserBasedRecommender.java with the fork's sketch point query
(GenericUserBasedRecommender.java:134-184): NearestNUserNeighborhood(n, minSimilarity) is the bank's re-scored
cosine top-n (similarities bit-equal to the pair cosine, ties by lower user row), computed once and kept on the
device; candidate items are the neighbours' items (getAllOtherItems), every candidate is estimated over the
neighbourhood and the best howMany are kept under (value desc, itemID asc) (TopItems, with this project's tie rule).
Both run in K_RECOMMEND (csrc/recommend.cu).

Documented deviation: cosine_topk never admits similarities <= 0 (the RowSimilarityJob rule), where
NearestNUserNeighborhood would when fewer than n users are positively similar.
"""
from __future__ import annotations

import numpy as np

from .cosinecm import CosineCM


def _item_csr(cm: CosineCM, device: int):
    """the data model as K_RECOMMEND takes it, on the device: the items each user row rated, CSR by user row
    (item_ptr [U+1], item_col int32), items as dense numbers of item_ids (ascending itemIDs)"""
    import torch
    rows = np.searchsorted(cm.user_ids, cm._u_sorted)
    item_ids = np.unique(cm._i_sorted)
    col = np.searchsorted(item_ids, cm._i_sorted)
    pairs = np.unique(rows.astype(np.int64) * item_ids.shape[0] + col)   # a user's item set
    prow, pcol = pairs // item_ids.shape[0], pairs % item_ids.shape[0]
    ptr = np.zeros(cm.user_ids.shape[0] + 1, np.int64)
    np.cumsum(np.bincount(prow, minlength=cm.user_ids.shape[0]), out=ptr[1:])
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).to(f"cuda:{device}")
                 for a in (ptr, pcol.astype(np.int32), item_ids))


class GenericUserBasedRecommender:
    def __init__(self, cm: CosineCM, neighborhood_size: int, min_similarity: float | None = None):
        self.cm = cm
        self.bank = cm.bank
        self.neighborhood_size = int(neighborhood_size)
        self._csr = _item_csr(cm, self.bank.ctx.device)
        self.item_ids = self._csr[2].cpu().numpy()
        self.nb_idx, self.nb_sim, self.nb_cnt = self.bank.cosine_topk(
            self.neighborhood_size, threshold=min_similarity, exclude_self=True, precision="rescored", device=True)

    def getUserNeighborhood(self, userID: int) -> np.ndarray:
        r = int(self.cm._rows(userID)[0])
        n = int(self.nb_cnt[r])
        return self.cm.user_ids[self.nb_idx[r, :n].cpu().numpy()]

    def recommend_all(self, howMany: int, userIDs=None, includeKnownItems: bool = False):
        """(user_ids [m], items [m, howMany] itemIDs (-1 unused), values [m, howMany] float32, counts [m])"""
        import torch
        user_ids = self.cm.user_ids if userIDs is None else np.atleast_1d(np.asarray(userIDs, np.int64))
        rows = np.arange(self.cm.user_ids.shape[0], dtype=np.int64) if userIDs is None else self.cm._rows(user_ids)
        dev = f"cuda:{self.bank.ctx.device}"
        items, vals, cnt = self.bank.recommend(self.nb_idx, self.nb_sim, self.nb_cnt, *self._csr,
                                               torch.from_numpy(rows).to(dev), howMany, includeKnownItems)
        return user_ids, items.cpu().numpy(), vals.cpu().numpy(), cnt.cpu().numpy()

    def recommend(self, userID: int, howMany: int, includeKnownItems: bool = False):
        """list of (itemID, value), best first"""
        _, items, vals, cnt = self.recommend_all(howMany, [userID], includeKnownItems)
        n = int(cnt[0])
        return [(int(i), float(v)) for i, v in zip(items[0, :n], vals[0, :n])]

    def estimate_preferences(self, userIDs, itemIDs) -> np.ndarray:
        """doEstimatePreference over the recommender's neighbourhoods for (userID, itemID) pairs -- the held-out
        pairs of one fold of a K-fold evaluation (RMSRecommenderEvaluatorKFold); float32, NaN = no estimate"""
        import torch
        dev = f"cuda:{self.bank.ctx.device}"
        rows = torch.from_numpy(self.cm._rows(userIDs)).to(dev)
        items = torch.from_numpy(np.ascontiguousarray(np.atleast_1d(itemIDs), np.int64)).to(dev)
        return self.bank.estimate_prefs(self.nb_idx, self.nb_sim, self.nb_cnt, rows, items).cpu().numpy()


class PerUserConfigUserBasedRecommender:
    """GenericUserBasedRecommender's neighbourhoods and estimates over CosineCM with a CountMinSketchConfig: every
    user's sketch at its own size (CosineCM.sized_bank), similarities as CosineCM.userSimilarity computes them (user 1
    re-sketched at user 2's size), NearestNUserNeighborhood(n, min_similarity) exactly -- NaN never admitted,
    negative similarities admitted when they pass min_similarity, ties by lower user row -- and doEstimatePreference
    point-querying each neighbour's own sketch; recommend() ranks the neighbours' items by those estimates.  All in
    K_RECOMMEND (csrc/cmsized.cu)."""

    def __init__(self, cm: CosineCM, n: int, min_similarity: float = float("-inf")):
        self.cm = cm
        self.bank = cm.sized_bank()
        self.n = int(n)
        self.min_similarity = float(min_similarity)
        self._csr = None   # the data model for recommend(), built on first use

    def _dev(self):
        return f"cuda:{self.bank.ctx.device}"

    def neighborhoods(self, userIDs=None):
        """(idx [m, n], sim [m, n], cnt [m]) as device tensors, rows = user rows (unused slots -1 / 0), for userIDs
        (every user when None)"""
        import torch
        rows = np.arange(self.cm.user_ids.shape[0], dtype=np.int64) if userIDs is None else self.cm._rows(userIDs)
        return self.bank.neighborhood(torch.from_numpy(rows).to(self._dev()), self.n, self.min_similarity)

    def getUserNeighborhood(self, userID: int) -> np.ndarray:
        idx, _, cnt = self.bank.neighborhood(self.cm._rows(userID), self.n, self.min_similarity)
        return self.cm.user_ids[idx[0, :int(cnt[0])]]

    def estimate_preferences(self, userIDs, itemIDs) -> np.ndarray:
        """doEstimatePreference for (userID, itemID) pairs over each user's neighbourhood; float32, NaN = none"""
        import torch
        rows = self.cm._rows(userIDs)
        uniq, inv = np.unique(rows, return_inverse=True)
        dev = self._dev()
        idx, sim, cnt = self.bank.neighborhood(torch.from_numpy(uniq).to(dev), self.n, self.min_similarity)
        items = torch.from_numpy(np.ascontiguousarray(np.atleast_1d(itemIDs), np.int64)).to(dev)
        return self.bank.estimate_prefs(idx, sim, cnt, torch.from_numpy(rows).to(dev), items,
                                        nb_row=torch.from_numpy(inv.astype(np.int64)).to(dev)).cpu().numpy()

    def recommend_all(self, howMany: int, userIDs=None, includeKnownItems: bool = False):
        """(user_ids [m], items [m, howMany] itemIDs (-1 unused), values [m, howMany] float32, counts [m]): each
        user's neighbourhood, then GenericUserBasedRecommender.recommend over it -- NaN estimates dropped, ranked by
        (value desc, itemID asc); negative and infinite estimates (negative similarities) rank by value"""
        import torch
        user_ids = self.cm.user_ids if userIDs is None else np.atleast_1d(np.asarray(userIDs, np.int64))
        rows = np.arange(self.cm.user_ids.shape[0], dtype=np.int64) if userIDs is None else self.cm._rows(user_ids)
        if self._csr is None:
            self._csr = _item_csr(self.cm, self.bank.ctx.device)
        rows_d = torch.from_numpy(rows).to(self._dev())
        idx, sim, cnt = self.bank.neighborhood(rows_d, self.n, self.min_similarity)
        items, vals, c = self.bank.recommend(idx, sim, cnt, *self._csr, rows_d, howMany, includeKnownItems)
        return user_ids, items.cpu().numpy(), vals.cpu().numpy(), c.cpu().numpy()

    def recommend(self, userID: int, howMany: int, includeKnownItems: bool = False):
        """list of (itemID, value), best first"""
        _, items, vals, cnt = self.recommend_all(howMany, [userID], includeKnownItems)
        n = int(cnt[0])
        return [(int(i), float(v)) for i, v in zip(items[0, :n], vals[0, :n])]
