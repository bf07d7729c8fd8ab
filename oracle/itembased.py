"""numpy restatement of RecommenderJob's aggregate-and-recommend phase (mahout_b200.itembased, K_RECOMMEND's
`k_itembased`).

TEST INFRASTRUCTURE ONLY.  The item top-k lists are taken as given (idx / sim / cnt as cosine_topk returns them), so
the product's output can be compared bit for bit on identical inputs.  Per user (rules 1-7 of DESIGN.md section 3):
prefs of +-0 are dropped; with more than P prefs only those with |pref| >= the P-th largest |pref| are considered;
the considered lists are visited in ascending item row, numpy rounding s * p and the sums separately as Java does;
the considered items get no prediction; non-boolean predictions need 2 datapoints; NaN and values <= Float.MIN_VALUE
are dropped; the allowed items are kept; order (value desc, itemID asc).
"""
from __future__ import annotations

import numpy as np

FLOAT_MIN_VALUE = np.float32(1.4e-45)


def considered(vals, max_prefs):
    """mask of the considered prefs of one user vector (vals float32, the user's prefs in row order)"""
    nz = vals != 0
    if int(nz.sum()) <= max_prefs:
        return nz
    a = np.abs(vals)
    T = np.sort(a[nz])[::-1][max_prefs - 1]
    return nz & (a >= T)


def predictions(idx, sim, cnt, rows, vals, num_items, max_prefs, boolean_data):
    """float32 predictions [num_items] of one user, NaN where there is none"""
    keep = considered(vals, max_prefs)
    num = np.zeros(num_items, np.float64)
    den = np.zeros(num_items, np.float64)
    used = np.zeros(num_items, np.int64)
    for j, p in zip(rows[keep], vals[keep]):
        c = int(cnt[j])
        ii, ss = idx[j, :c], sim[j, :c]
        if boolean_data:
            num[ii] = num[ii] + ss
        else:
            num[ii] = num[ii] + ss * np.float64(p)
            den[ii] = den[ii] + np.abs(ss)
        used[ii] += 1
    num[rows[keep]] = np.nan                            # upstream's NaN diagonal
    with np.errstate(divide="ignore", invalid="ignore"):
        pred = num.astype(np.float32) if boolean_data else (num / den).astype(np.float32)
    if not boolean_data:
        pred[used < 2] = np.nan
    pred[used == 0] = np.nan
    return pred


def recommend(idx, sim, cnt, user_ptr, pref_row, pref_val, item_ids, users, how_many, max_prefs=10,
              boolean_data=False, allowed=None):
    """(items [m, how_many] itemIDs (-1 unused), values [m, how_many] float32 (0 unused), counts [m]);
    allowed: bool [num_items] over item rows, or None"""
    idx, sim, cnt = np.asarray(idx), np.asarray(sim), np.asarray(cnt)
    item_ids = np.asarray(item_ids, np.int64)
    num_items = item_ids.shape[0]
    m = len(users)
    out_i = np.full((m, how_many), -1, np.int64)
    out_v = np.zeros((m, how_many), np.float32)
    out_c = np.zeros(m, np.int32)
    for t, u in enumerate(int(x) for x in users):
        lo, hi = int(user_ptr[u]), int(user_ptr[u + 1])
        pred = predictions(idx, sim, cnt, np.asarray(pref_row[lo:hi], np.int64), np.asarray(pref_val[lo:hi], np.float32),
                           num_items, max_prefs, boolean_data)
        ok = ~np.isnan(pred) & (pred > FLOAT_MIN_VALUE)
        if allowed is not None:
            ok &= allowed
        r = np.nonzero(ok)[0]
        order = np.lexsort((item_ids[r], -pred[r].astype(np.float64)))[:how_many]
        n = order.shape[0]
        out_i[t, :n], out_v[t, :n], out_c[t] = item_ids[r[order]], pred[r[order]], n
    return out_i, out_v, out_c


def user_csr(row, user, pref):
    """(user_ids, user_ptr, pref_row, pref_val) of de-duplicated (item row, userID, pref) events, as
    mahout_b200.itembased.user_vectors builds it"""
    row, user = np.asarray(row, np.int64), np.asarray(user, np.int64)
    order = np.lexsort((row, user))
    ids, counts = np.unique(user[order], return_counts=True)
    ptr = np.zeros(ids.shape[0] + 1, np.int64)
    np.cumsum(counts, out=ptr[1:])
    return ids, ptr, row[order].astype(np.int32), np.asarray(pref, np.float32)[order]
