"""CPU checks of oracle/recommend.py, the numpy restatement the GPU recommender is compared with bit for bit:
pinned to a scalar per-item loop over oracle.cm_get / oracle.cm_cosine (GenericUserBasedRecommender's
doEstimatePreference as tests/test_sketch_gpu.py restates it), and a hand-made known answer."""
import math

import numpy as np

import oracle as orc
from oracle import recommend as orec


def _scalar_estimate(sk, w, d, a, b, u, nb, sims, item):
    preference = total = 0.0
    count = 0
    for v, s in zip(nb, sims):
        if v == u:
            continue
        p = float(np.float32(orc.cm_get(sk[v], w, d, a, b, item)))
        if p == 0.0 or math.isnan(s):
            continue
        s = min(max(s, -1.0), 1.0)
        preference += s * p
        total += s
        count += 1
    return math.nan if count <= 1 else float(np.float32(preference / total))


def test_oracle_matches_scalar_loop():
    rng = np.random.Generator(np.random.PCG64(5))
    U, w, d, k = 40, 64, 3, 6
    n = 900
    rows = rng.integers(0, U, n)
    items = rng.integers(1, 150, n) * 3
    pref = (rng.integers(-4, 9, n) * 0.5).astype(np.float32)          # negative increments too
    a, b = orc.hash_params(11, d)
    bank = np.zeros((U, d, w))
    orc.bank_update(bank, d, w, a, b, rows, items, pref)
    sk = [np.ascontiguousarray(bank[u]) for u in range(U)]
    # neighbourhoods: random lists (self, repeats and negative similarities allowed), sims from the scalar cosine
    nb_idx = rng.integers(0, U, (U, k))
    nb_cnt = rng.integers(0, k + 1, U).astype(np.int32)
    nb_sim = np.array([[orc.cm_cosine(sk[u], sk[v], w, d) for v in nb_idx[u]] for u in range(U)])
    ptr, col, ids = orec.item_csr(rows, items, U)
    for include_known in (False, True):
        got_i, got_v, got_c = orec.recommend(bank, a, b, nb_idx, nb_sim, nb_cnt, ptr, col, ids, np.arange(U), 7,
                                             include_known)
        for u in range(U):
            nb = [int(v) for v in nb_idx[u, :nb_cnt[u]]]
            cand = set()
            for v in nb:
                cand |= {int(x) for x in items[rows == v]}
            if not include_known:
                cand -= {int(x) for x in items[rows == u]}
            est = [(it, _scalar_estimate(sk, w, d, a, b, u, nb, nb_sim[u, :nb_cnt[u]], it)) for it in cand]
            est = sorted(((v, it) for it, v in est if not math.isnan(v)), key=lambda t: (-t[0], t[1]))[:7]
            assert got_c[u] == len(est)
            assert got_i[u, :len(est)].tolist() == [it for _, it in est]
            assert got_v[u, :len(est)].tolist() == [v for v, _ in est]
            assert (got_i[u, len(est):] == -1).all()


def test_hand_made_four_users():
    """Users 0..3 with exact one-column sketches (identity hash, w > itemIDs): every point query is the rating."""
    w, d = 16, 1
    a, b = np.ones(1, np.int64), np.zeros(1, np.int64)
    ratings = {0: {1: 5.0, 2: 3.0},
               1: {1: 4.0, 3: 2.0, 4: 1.0, 5: 2.0},
               2: {3: 4.0, 4: 2.0, 6: 5.0, 5: 1.0},
               3: {7: 5.0}}
    rows = [u for u, r in ratings.items() for _ in r]
    items = [i for r in ratings.values() for i in r]
    prefs = np.array([p for r in ratings.values() for p in r.values()], np.float32)
    bank = np.zeros((4, d, w))
    orc.bank_update(bank, d, w, a, b, rows, items, prefs)
    ptr, col, ids = orec.item_csr(rows, items, 4)
    nb_idx = np.array([[1, 2, 0], [0, 2, -1], [1, 0, -1], [0, 0, 0]])
    nb_sim = np.array([[0.5, 0.25, 1.0], [0.5, 0.5, 0.0], [0.75, 0.25, 0.0], [0.0, 0.0, 0.0]])
    nb_cnt = np.array([3, 2, 2, 0], np.int32)
    got_i, got_v, got_c = orec.recommend(bank, a, b, nb_idx, nb_sim, nb_cnt, ptr, col, ids, np.arange(4), 10)
    # user 0: neighbours 1, 2 (itself skipped); items 3, 4, 5 rated by both, 6 by one only (count <= 1: NaN);
    # 3: (0.5*2 + 0.25*4) / 0.75 = 2.666.., 4: (0.5*1 + 0.25*2) / 0.75 = 1.333.., 5: (0.5*2 + 0.25*1) / 0.75
    # = 1.666..; own items 1, 2 removed
    assert got_c[0] == 3
    assert got_i[0, :3].tolist() == [3, 5, 4]
    assert got_v[0, :3].tolist() == [np.float32(2.0 / 0.75), np.float32(1.25 / 0.75), np.float32(1.0 / 0.75)]
    # user 1: neighbours 0 and 2 share no item with each other: every candidate has one contribution -> none
    assert got_c[1] == 0 and (got_i[1] == -1).all() and (got_v[1] == 0).all()
    # user 3: empty neighbourhood
    assert got_c[3] == 0
    # with the known items: user 2's neighbours 1 and 0 both rated item 1 (4 and 5): one estimate, 4.25
    got_i, got_v, got_c = orec.recommend(bank, a, b, nb_idx, nb_sim, nb_cnt, ptr, col, ids, np.arange(4), 10, True)
    assert got_i[2, :got_c[2]].tolist() == [1]
    assert got_v[2, 0] == np.float32((0.75 * 4 + 0.25 * 5) / 1.0)
    # ties: two candidates with the same estimate come out lower itemID first
    ratings_t = {0: {9: 1.0}, 1: {4: 2.0, 2: 2.0}, 2: {4: 2.0, 2: 2.0}}
    rows = [u for u, r in ratings_t.items() for _ in r]
    items = [i for r in ratings_t.values() for i in r]
    prefs = np.array([p for r in ratings_t.values() for p in r.values()], np.float32)
    bank = np.zeros((3, d, w))
    orc.bank_update(bank, d, w, a, b, rows, items, prefs)
    ptr, col, ids = orec.item_csr(rows, items, 3)
    nb_idx = np.array([[1, 2], [0, 2], [0, 1]])
    nb_sim = np.full((3, 2), 0.5)
    got_i, got_v, got_c = orec.recommend(bank, a, b, nb_idx, nb_sim, np.array([2, 2, 2], np.int32), ptr, col, ids,
                                         np.arange(3), 1)
    assert got_c[0] == 1 and got_i[0, 0] == 2 and got_v[0, 0] == 2.0
