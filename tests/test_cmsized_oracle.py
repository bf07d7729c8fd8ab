"""The oracle of CosineCM with a CountMinSketchConfig (orc_sized_neighborhood / orc_sized_estimate) against a Python
loop over the oracle's per-sketch primitives (cm_dims, cm_update, cm_cosine, clamp_similarity, cm_get), and a pair
checked by hand whose two directions differ.  CPU only."""
import math

import numpy as np

import oracle as orc
from oracle import sized as osz
from mahout_b200.cmconfig import CountMinSketchConfig

SEED = 7


def _model(rng, users, items, max_prefs):
    """CSR by user row with 1..max_prefs prefs per user, half-star prefs, some negative"""
    n = rng.integers(1, max_prefs + 1, users)
    ptr = np.zeros(users + 1, np.int64)
    np.cumsum(n, out=ptr[1:])
    item = np.concatenate([rng.choice(items, k, replace=False) for k in n]).astype(np.int64) + 1
    pref = (rng.integers(-4, 11, ptr[-1]) * 0.5).astype(np.float32)
    return ptr, item, pref


def _shapes(ptr, items, q):
    cfg = CountMinSketchConfig(q)
    uid = np.arange(ptr.shape[0] - 1)
    cfg.configure(uid, np.diff(ptr), items)
    wd = [orc.cm_dims(cfg.getDelta(u), cfg.getEpsilon(u)) for u in uid]
    return np.array([x[0] for x in wd], np.int32), np.array([x[1] for x in wd], np.int32)


def _sketch(u, w, d, a, b, ptr, item, pref):
    c = np.zeros((d, w))
    orc.cm_update(c, w, d, a, b, item[ptr[u]:ptr[u + 1]], pref[ptr[u]:ptr[u + 1]].astype(np.float64))
    return c


def _loop_neighborhood(width, depth, a, b, ptr, item, pref, queries, n, min_sim):
    U = width.shape[0]
    own = [_sketch(v, width[v], depth[v], a, b, ptr, item, pref) for v in range(U)]
    out = []
    for u in queries:
        cand = []
        for v in range(U):
            if v == u:
                continue
            s = orc.cm_cosine(_sketch(u, width[v], depth[v], a, b, ptr, item, pref), own[v], width[v], depth[v])
            s = s if math.isnan(s) else orc.clamp_similarity(s)
            if not math.isnan(s) and s >= min_sim:
                cand.append((-s, v))
        cand.sort()
        out.append([(v, -ms) for ms, v in cand[:n]])
    return out, own


def test_oracle_neighborhood_and_estimate_equal_the_primitive_loop():
    rng = np.random.Generator(np.random.PCG64(5))
    U, items = 40, 60
    ptr, item, pref = _model(rng, U, items, 25)
    width, depth = _shapes(ptr, items, 1.0)
    a, b = orc.hash_params(SEED, int(depth.max()))
    queries = np.arange(U)
    for n, min_sim in ((5, -np.inf), (50, 0.2), (3, -0.5)):
        want, own = _loop_neighborhood(width, depth, a, b, ptr, item, pref, queries, n, min_sim)
        idx, sim, cnt = osz.sized_neighborhood(width, depth, a, b, ptr, item, pref, queries, n, min_sim)
        for t, lst in enumerate(want):
            assert cnt[t] == len(lst)
            assert idx[t, :cnt[t]].tolist() == [v for v, _ in lst]
            assert sim[t, :cnt[t]].tobytes() == np.array([s for _, s in lst]).tobytes()
            assert (idx[t, cnt[t]:] == -1).all() and (sim[t, cnt[t]:] == 0).all()
    # doEstimatePreference with each neighbour's own sketch, in list order
    idx, sim, cnt = osz.sized_neighborhood(width, depth, a, b, ptr, item, pref, queries, 8)
    users = rng.integers(0, U, 300)
    its = rng.integers(1, items + 1, 300)
    got = osz.sized_estimate(width, depth, a, b, ptr, item, pref, idx, sim, cnt, users, its)
    for t in range(300):
        u = users[t]
        p_sum = tot = 0.0
        count = 0
        for j in range(cnt[u]):
            v = idx[u, j]
            if v == u:
                continue
            p = float(np.float32(orc.cm_get(own[v], width[v], depth[v], a, b, int(its[t]))))
            s = orc.clamp_similarity(sim[u, j])
            if p != 0.0 and not math.isnan(s):
                p_sum += s * p
                tot += s
                count += 1
        want = math.nan if count <= 1 else float(np.float32(p_sum / tot))
        assert (math.isnan(want) and math.isnan(got[t])) or got[t] == np.float32(want)


def test_hand_checked_pair_whose_directions_differ():
    """u1 has two prefs of 1.0, u2 one pref of 1.0.  Under the q = 1.0 config a one-pref user's sketch is (1, 1) and a
    two-pref user's (2, 2).  sim(u1 -> u2): u1 re-sketched at (1, 1) is the single counter 2 against u2's 1: exactly 1.
    sim(u2 -> u1): u2 at (2, 2) puts 1 in one column of each row; u1's own rows hold 1, 1 in different columns (the
    items are picked so): every row gives 1 / (1 * sqrt(2))."""
    items = 1000
    ptr_n = np.array([0, 2, 3], np.int64)
    width, depth = _shapes(ptr_n, items, 1.0)
    assert width.tolist() == [2, 1] and depth.tolist() == [2, 1]
    a, b = orc.hash_params(SEED, 2)
    x = next(k for k in range(1, items) if all(orc.hash_one(a[i], b[i], 2, k) != orc.hash_one(a[i], b[i], 2, 1)
                                               for i in range(2)))
    item = np.array([1, x, 5], np.int64)
    pref = np.ones(3, np.float32)
    idx, sim, cnt = osz.sized_neighborhood(width, depth, a, b, ptr_n, item, pref, [0, 1], 1)
    assert cnt.tolist() == [1, 1] and idx[:, 0].tolist() == [1, 0]
    assert sim[0, 0] == 1.0
    assert sim[1, 0] == 1.0 / (1.0 * math.sqrt(2.0))
