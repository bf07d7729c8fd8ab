"""GenericUserBasedRecommender.recommend over CosineCM with a CountMinSketchConfig (mb200_sized_recommend).

TEST INFRASTRUCTURE ONLY (tests/ and tools/ parity legs) -- never imported from mahout_b200/.  Composed from
oracle.recommend.candidates, oracle.sized.sized_estimate and oracle.recommend.recommend's lexsort; row t of the lists
is users[t]'s neighbourhood.
"""
from __future__ import annotations

import numpy as np

from .recommend import candidates
from .sized import sized_estimate


def sized_recommend(width, depth, a, b, user_ptr, item, pref, nb_idx, nb_sim, nb_cnt, item_ptr, item_col, item_ids,
                    users, how_many, include_known=False, nthreads=None):
    """(items [m, how_many] itemIDs (-1 unused), values [m, how_many] float32 (0 unused), counts [m])"""
    users = np.asarray(users, np.int64)
    item_ids = np.asarray(item_ids, np.int64)
    m = users.shape[0]
    cands = [candidates(int(u), nb_idx[t], nb_cnt[t], item_ptr, item_col, include_known) for t, u in enumerate(users)]
    rows = np.repeat(np.arange(m, dtype=np.int64), [c.shape[0] for c in cands])
    cand = np.concatenate(cands) if m else np.zeros(0, np.int64)
    est = np.zeros(0, np.float32)
    if cand.shape[0]:      # every (user, candidate) of the call in one batch of point queries
        est = sized_estimate(width, depth, a, b, user_ptr, item, pref, nb_idx, nb_sim, nb_cnt, users[rows],
                             item_ids[cand], nb_row=rows, nthreads=nthreads)
    out_i = np.full((m, how_many), -1, np.int64)
    out_v = np.zeros((m, how_many), np.float32)
    out_c = np.zeros(m, np.int32)
    at = 0
    for t in range(m):
        k = cands[t].shape[0]
        e, ids = est[at:at + k], item_ids[cands[t]]
        at += k
        ok = ~np.isnan(e)
        ids, val = ids[ok], e[ok]
        order = np.lexsort((ids, -val.astype(np.float64)))[:how_many]   # (value desc, itemID asc)
        n = order.shape[0]
        out_i[t, :n], out_v[t, :n], out_c[t] = ids[order], val[order], n
    return out_i, out_v, out_c
