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
    return tuple(torch.from_numpy(a).to(f"cuda:{device}") for a in _item_csr_host(cm))


def _item_csr_host(cm: CosineCM):
    """_item_csr's arrays in host memory"""
    rows = np.searchsorted(cm.user_ids, cm._u_sorted)
    item_ids = np.unique(cm._i_sorted)
    col = np.searchsorted(item_ids, cm._i_sorted)
    pairs = np.unique(rows.astype(np.int64) * item_ids.shape[0] + col)   # a user's item set
    prow, pcol = pairs // item_ids.shape[0], pairs % item_ids.shape[0]
    ptr = np.zeros(cm.user_ids.shape[0] + 1, np.int64)
    np.cumsum(np.bincount(prow, minlength=cm.user_ids.shape[0]), out=ptr[1:])
    return tuple(np.ascontiguousarray(a) for a in (ptr, pcol.astype(np.int32), item_ids))


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
    K_RECOMMEND (csrc/cmsized.cu).

    With `multi` (a mahout_b200.multi.MultiGpu) the sized bank is replicated on every GPU of that handle and every
    call splits its users between them (csrc/sized_multi.cu): the same results bit for bit, as host arrays."""

    def __init__(self, cm: CosineCM, n: int, min_similarity: float = float("-inf"), multi=None):
        self.cm = cm
        self.multi = multi
        self.bank = cm.sized_bank() if multi is None else None
        self.multi_bank = cm.multi_sized_bank(multi) if multi is not None else None
        self.n = int(n)
        self.min_similarity = float(min_similarity)
        self._csr = None   # the data model for recommend(), built on first use

    def _dev(self):
        return f"cuda:{self.bank.ctx.device}"

    def _all_rows(self, userIDs):
        return np.arange(self.cm.user_ids.shape[0], dtype=np.int64) if userIDs is None else self.cm._rows(userIDs)

    def neighborhoods(self, userIDs=None):
        """(idx [m, n], sim [m, n], cnt [m]), rows = user rows (unused slots -1 / 0), for userIDs (every user when
        None); device tensors on one GPU, numpy arrays with `multi`"""
        rows = self._all_rows(userIDs)
        if self.multi_bank is not None:
            return self.multi_bank.neighborhood(rows, self.n, self.min_similarity)
        import torch
        return self.bank.neighborhood(torch.from_numpy(rows).to(self._dev()), self.n, self.min_similarity)

    def getUserNeighborhood(self, userID: int) -> np.ndarray:
        b = self.multi_bank if self.multi_bank is not None else self.bank
        idx, _, cnt = b.neighborhood(self.cm._rows(userID), self.n, self.min_similarity)
        return self.cm.user_ids[idx[0, :int(cnt[0])]]

    def estimate_preferences(self, userIDs, itemIDs) -> np.ndarray:
        """doEstimatePreference for (userID, itemID) pairs over each user's neighbourhood; float32, NaN = none"""
        rows = self.cm._rows(userIDs)
        items = np.ascontiguousarray(np.atleast_1d(itemIDs), np.int64)
        if self.multi_bank is not None:
            return self.multi_bank.estimate_prefs(rows, items, self.n, self.min_similarity)
        import torch
        uniq, inv = np.unique(rows, return_inverse=True)
        dev = self._dev()
        idx, sim, cnt = self.bank.neighborhood(torch.from_numpy(uniq).to(dev), self.n, self.min_similarity)
        return self.bank.estimate_prefs(idx, sim, cnt, torch.from_numpy(rows).to(dev), torch.from_numpy(items).to(dev),
                                        nb_row=torch.from_numpy(inv.astype(np.int64)).to(dev)).cpu().numpy()

    def recommend_all(self, howMany: int, userIDs=None, includeKnownItems: bool = False):
        """(user_ids [m], items [m, howMany] itemIDs (-1 unused), values [m, howMany] float32, counts [m]): each
        user's neighbourhood, then GenericUserBasedRecommender.recommend over it -- NaN estimates dropped, ranked by
        (value desc, itemID asc); negative and infinite estimates (negative similarities) rank by value"""
        user_ids = self.cm.user_ids if userIDs is None else np.atleast_1d(np.asarray(userIDs, np.int64))
        rows = self._all_rows(None if userIDs is None else user_ids)
        if self.multi_bank is not None:
            if self._csr is None:
                self._csr = _item_csr_host(self.cm)
            items, vals, c = self.multi_bank.recommend_users(rows, self.n, self.min_similarity, *self._csr, howMany,
                                                             includeKnownItems)
            return user_ids, items, vals, c
        import torch
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
