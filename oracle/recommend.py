"""numpy restatement of GenericUserBasedRecommender over the sketch bank (mahout_b200.recommender, K_RECOMMEND).

TEST INFRASTRUCTURE ONLY.  Banks are the oracle's FP64 banks [E, d, w] (oracle.bank_update); the neighbourhood
lists are given (nb_idx / nb_sim / nb_cnt as cosine_topk returns them), so the product's estimates and top-N can be
compared bit for bit with identical inputs.  The neighbour slots are visited in list order, vectorised over the
candidates; numpy rounds s * p and the sum separately, as Java does.
"""
from __future__ import annotations

import numpy as np

from . import hash_many


def item_columns(a, b, w, items):
    """[d, n] columns of the items in every hash row"""
    items = np.ascontiguousarray(items, np.int64)
    return np.stack([hash_many(int(a[r]), int(b[r]), w, items) for r in range(len(a))]).astype(np.int64)


def estimate(bank, a, b, u, nb_idx_row, nb_sim_row, cnt, items, cols=None):
    """doEstimatePreference of user row u for every item of `items` over one neighbourhood row: float32 [n]"""
    E, d, w = bank.shape
    cols = item_columns(a, b, w, items) if cols is None else cols
    n = cols.shape[1]
    pref = np.zeros(n, np.float64)
    tot = np.zeros(n, np.float64)
    count = np.zeros(n, np.int64)
    for j in range(int(cnt)):
        v = int(nb_idx_row[j])
        if v == u:
            continue
        s = float(nb_sim_row[j])
        if np.isnan(s):
            continue
        s = min(max(s, -1.0), 1.0)
        p = bank[v][np.arange(d)[:, None], cols].min(axis=0).astype(np.float32).astype(np.float64)   # (float) cm.get
        m = p != 0.0
        pref[m] = pref[m] + s * p[m]
        tot[m] = tot[m] + s
        count[m] += 1
    with np.errstate(divide="ignore", invalid="ignore"):
        est = (pref / tot).astype(np.float32)
    est[count <= 1] = np.nan
    return est


def candidates(u, nb_idx_row, cnt, item_ptr, item_col, include_known):
    """dense item numbers rated by a listed neighbour, minus the user's own unless include_known, ascending"""
    parts = [item_col[item_ptr[v]:item_ptr[v + 1]] for v in (int(x) for x in nb_idx_row[:int(cnt)])]
    cand = np.unique(np.concatenate(parts)) if parts else np.zeros(0, np.int64)
    if not include_known:
        cand = np.setdiff1d(cand, item_col[item_ptr[u]:item_ptr[u + 1]])
    return cand.astype(np.int64)


def recommend(bank, a, b, nb_idx, nb_sim, nb_cnt, item_ptr, item_col, item_ids, users, how_many,
              include_known=False):
    """(items [m, how_many] itemIDs (-1 unused), values [m, how_many] float32 (0 unused), counts [m])"""
    m = len(users)
    out_i = np.full((m, how_many), -1, np.int64)
    out_v = np.zeros((m, how_many), np.float32)
    out_c = np.zeros(m, np.int32)
    for t, u in enumerate(int(x) for x in users):
        cand = candidates(u, nb_idx[u], nb_cnt[u], item_ptr, item_col, include_known)
        if cand.shape[0] == 0:
            continue
        est = estimate(bank, a, b, u, nb_idx[u], nb_sim[u], nb_cnt[u], item_ids[cand])
        ok = ~np.isnan(est)
        ids, val = item_ids[cand][ok], est[ok]
        order = np.lexsort((ids, -val.astype(np.float64)))[:how_many]   # (value desc, itemID asc)
        n = order.shape[0]
        out_i[t, :n], out_v[t, :n], out_c[t] = ids[order], val[order], n
    return out_i, out_v, out_c


def item_csr(user_rows, items, num_users):
    """the data model as the product takes it: (item_ptr [U+1], item_col, item_ids) from (user row, itemID) events"""
    item_ids = np.unique(items)
    col = np.searchsorted(item_ids, items)
    pairs = np.unique(np.asarray(user_rows, np.int64) * item_ids.shape[0] + col)
    prow, pcol = pairs // item_ids.shape[0], pairs % item_ids.shape[0]
    ptr = np.zeros(num_users + 1, np.int64)
    np.cumsum(np.bincount(prow, minlength=num_users), out=ptr[1:])
    return ptr, pcol.astype(np.int32), item_ids.astype(np.int64)
