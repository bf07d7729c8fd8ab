"""The reference of recommend() over per-user sketch sizes (oracle.sized_recommend) against a plain loop over
orc_sized_estimate, and a case checked by hand where a negative similarity makes tot = 0, so that +inf, -inf and
dropped NaN estimates all occur.  CPU only."""
import math

import numpy as np

import oracle as orc
from oracle import recommend as orec
from oracle import sized as osz
from oracle.sized_recommend import sized_recommend

SEED = 7


def _loop(width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt, item_ptr, item_col, item_ids, users, how_many,
          include_known):
    out = []
    for t, u in enumerate(users):
        cand = set()
        for v in nb_idx[t, :nb_cnt[t]]:
            cand.update(item_col[item_ptr[v]:item_ptr[v + 1]].tolist())
        if not include_known:
            cand -= set(item_col[item_ptr[u]:item_ptr[u + 1]].tolist())
        scored = []
        for c in sorted(cand):
            e = osz.sized_estimate(width, depth, a, b, ptr, item, pref, nb_idx[t:t + 1], nb_sim[t:t + 1],
                                   nb_cnt[t:t + 1], [u], [item_ids[c]], nb_row=[0])[0]
            if not math.isnan(e):
                scored.append((-float(e), int(item_ids[c]), e))
        scored.sort()
        out.append([(i, e) for _, i, e in scored[:how_many]])
    return out


def test_sized_recommend_equals_a_loop_over_sized_estimate():
    rng = np.random.Generator(np.random.PCG64(5))
    U, I = 30, 50
    n = rng.integers(1, 15, U)
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum(n, out=ptr[1:])
    item = np.concatenate([rng.choice(I, k, replace=False) for k in n]).astype(np.int64) * 3 + 1
    pref = (rng.integers(-4, 11, ptr[-1]) * 0.5).astype(np.float32)
    width = rng.integers(1, 40, U).astype(np.int32)
    depth = rng.integers(1, 6, U).astype(np.int32)
    a, b = orc.hash_params(SEED, int(depth.max()))
    user_rows = np.repeat(np.arange(U), n)
    item_ptr, item_col, item_ids = orec.item_csr(user_rows, item, U)
    # lists for a subset with a repeated user (row t belongs to users[t]); negative similarities listed
    users = np.array([0, 3, 3, 7, 12, 29, 15], np.int64)
    nb_idx, nb_sim, nb_cnt = osz.sized_neighborhood(width, depth, a, b, ptr, item, pref, users, 8)
    nb_cnt[2] = 3                                         # the repeated user with a shorter list
    nb_idx[1, 1] = users[1]                               # the user itself listed: skipped by the estimates
    for how_many, known in ((5, False), (40, True), (1, False)):
        gi, gv, gc = sized_recommend(width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt, item_ptr, item_col,
                                     item_ids, users, how_many, known)
        want = _loop(width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt, item_ptr, item_col, item_ids, users,
                     how_many, known)
        assert sum(len(w) for w in want) > 0
        for t, w in enumerate(want):
            assert gc[t] == len(w)
            assert gi[t, :gc[t]].tolist() == [i for i, _ in w]
            assert gv[t, :gc[t]].tobytes() == np.array([e for _, e in w], np.float32).tobytes()
            assert (gi[t, gc[t]:] == -1).all() and (gv[t, gc[t]:] == 0).all()


def hand_model():
    """four users at collision-free widths.  User 0's list: user 1 (sim 0.5), user 2 (sim -0.5), user 3 (sim 0.25).
    item 10: 1 -> 2.0, 2 -> 4.0     pref = 1 - 2 = -1,   tot = 0     -> -inf
    item 20: 1 -> 2.0, 2 -> -4.0    pref = 1 + 2 = 3,    tot = 0     -> +inf
    item 30: 1 -> 3.0, 2 -> 3.0     pref = 0,            tot = 0     -> NaN, dropped
    item 40: 1 -> 2.0, 3 -> 4.0     pref = 2,            tot = 0.75  -> 2.6666667
    item 50: 3 -> 1.0               one neighbour                     -> NaN, dropped
    item 60: 1 -> -2.0, 3 -> 2.0    pref = -0.5,         tot = 0.75  -> -0.6666667
    item 70: 0 -> 1.0 (known), 1 -> 2.0, 3 -> 1.0   pref = 1.25, tot = 0.75 -> 1.6666666"""
    prefs = {0: {70: 1.0},
             1: {10: 2.0, 20: 2.0, 30: 3.0, 40: 2.0, 60: -2.0, 70: 2.0},
             2: {10: 4.0, 20: -4.0, 30: 3.0},
             3: {40: 4.0, 50: 1.0, 60: 2.0, 70: 1.0}}
    ptr = np.zeros(5, np.int64)
    np.cumsum([len(prefs[u]) for u in range(4)], out=ptr[1:])
    item = np.array([i for u in range(4) for i in prefs[u]], np.int64)
    pref = np.array([p for u in range(4) for p in prefs[u].values()], np.float32)
    width = np.array([1009, 2003, 4001, 8009], np.int32)
    depth = np.array([1, 2, 3, 2], np.int32)
    a, b = orc.hash_params(SEED, 3)
    for u in range(4):          # no two items share a counter in any row: every point query is the pref itself
        for r in range(int(depth[u])):
            cols = orc.hash_many(int(a[r]), int(b[r]), int(width[u]), np.array([10, 20, 30, 40, 50, 60, 70], np.int64))
            assert np.unique(cols).shape[0] == 7
    nb_idx = np.array([[1, 2, 3]], np.int64)
    nb_sim = np.array([[0.5, -0.5, 0.25]])
    nb_cnt = np.array([3], np.int32)
    return width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt


HAND_WANT = {False: [(20, np.inf), (40, np.float32(2 / 0.75)), (60, np.float32(-0.5 / 0.75)), (10, -np.inf)],
             True: [(20, np.inf), (40, np.float32(2 / 0.75)), (70, np.float32(1.25 / 0.75)),
                    (60, np.float32(-0.5 / 0.75)), (10, -np.inf)]}


def test_hand_checked_infinite_negative_and_dropped_estimates():
    width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt = hand_model()
    item_ptr, item_col, item_ids = orec.item_csr(np.repeat(np.arange(4), np.diff(ptr)), item, 4)
    for known, want in HAND_WANT.items():
        gi, gv, gc = sized_recommend(width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt, item_ptr, item_col,
                                     item_ids, [0], 8, known)
        assert gc[0] == len(want)
        assert gi[0, :gc[0]].tolist() == [i for i, _ in want]
        assert gv[0, :gc[0]].tobytes() == np.array([v for _, v in want], np.float32).tobytes()
        # the dropped ones are NaN estimates, not missing candidates
        e = osz.sized_estimate(width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt, [0, 0], [30, 50])
        assert np.isnan(e).all()
