"""CosineCM with a CountMinSketchConfig on all GPUs of the process (mb200_sized_multi_*, csrc/sized_multi.cu): one
sized-bank replica per GPU, users split t mod G.  Every call is checked byte for byte -- floats, NaN slots, counts and
unused slots -- against the same SizedBank call on one context, at G = 1, 2 and all visible GPUs."""
import ctypes as C
import math

import numpy as np
import pytest

from test_cmsized_recommend_gpu import _data, _edge_model, _ml100k

pytestmark = pytest.mark.gpu

SEED = 11


def _gpus():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


@pytest.fixture(scope="module")
def ctx(mb):
    c = mb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", params=[1, 2, 0, "0,0"], ids=["G1", "G2", "Gall", "G2-one-device"])
def multi(request):
    """a MultiGpu over 1, 2 or all visible GPUs (the last only when that is more than 2), and two contexts on GPU 0:
    the split, the scatter and a failure on the second worker at G = 2 on a one-GPU machine"""
    from mahout_b200.multi import MultiGpu
    have = _gpus()
    g = request.param
    if g == 2 and have < 2:
        pytest.skip("needs 2 GPUs")
    if g == 0 and have <= 2:
        pytest.skip("all visible GPUs is already covered")
    m = MultiGpu(devices=[0, 0]) if g == "0,0" else MultiGpu(g)
    yield m
    m.close()


def _pair(mb, ctx, multi, width, depth, ptr, item, pref):
    single = mb.SizedBank(width, depth, mb.HashFunctionBuilder(SEED), ptr, item, pref, 1, ctx)
    many = multi.sized_bank(width, depth, mb.HashFunctionBuilder(SEED), ptr, item, pref, 1)
    return single, many


def _same(got, want):
    for g, w in zip(got, want):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape and g.dtype == w.dtype
        assert g.tobytes() == w.tobytes()


def _single_estimates(bank, rows, items, n, ms):
    """PerUserConfigUserBasedRecommender.estimate_preferences on one context"""
    uniq, inv = np.unique(rows, return_inverse=True)
    idx, sim, cnt = bank.neighborhood(uniq, n, ms)
    return bank.estimate_prefs(idx, sim, cnt, rows, items, nb_row=inv.astype(np.int64))


def _check_all(single, many, ptr, item, users, n, ms, how_many=(10,), known=(False, True), pairs=None):
    """neighbourhood, recommend and estimates of `users` against the single context, byte for byte"""
    want = single.neighborhood(users, n, ms)
    _same(many.neighborhood(users, n, ms), want)
    data = _data(ptr, item)
    for h in how_many:
        for k in known:
            w = single.recommend(*want, *data, users, h, k)
            _same(many.recommend_users(users, n, ms, *data, h, k), w)
    if pairs is not None:
        rows, items = pairs
        _same([many.estimate_prefs(rows, items, n, ms)], [_single_estimates(single, rows, items, n, ms)])
    return want


def _pairs(rng, U, items, k):
    """k (user row, itemID) pairs: repeated users, rated items and items nobody rated"""
    rows = rng.integers(0, U, k).astype(np.int64)
    rows[: k // 4] = rows[0]
    it = np.where(rng.random(k) < 0.7, rng.choice(items, k), items.max() + 1 + rng.integers(0, 50, k)).astype(np.int64)
    return rows, it


@pytest.mark.parametrize("q", [1.0, 0.5])
def test_ml100k_all_users(mb, ctx, multi, q):
    rng = np.random.Generator(np.random.PCG64(1))
    width, depth, ptr, item, pref = _ml100k(rng, q)
    single, many = _pair(mb, ctx, multi, width, depth, ptr, item, pref)
    U = width.shape[0]
    users = np.arange(U)
    pairs = _pairs(rng, U, np.unique(item), 5000)
    _, _, cnt = _check_all(single, many, ptr, item, users, 30, -np.inf, how_many=(10, 1024), pairs=pairs)
    assert cnt.sum() > 0
    many.close()
    single.close()


def test_shuffled_subset_with_repeats(mb, ctx, multi):
    rng = np.random.Generator(np.random.PCG64(5))
    width, depth, ptr, item, pref = _ml100k(rng, 1.0)
    single, many = _pair(mb, ctx, multi, width, depth, ptr, item, pref)
    U = width.shape[0]
    users = rng.permutation(np.concatenate([rng.choice(U, 300, replace=False), rng.choice(U, 40)]))
    users[7] = users[3] = users[200]
    _check_all(single, many, ptr, item, users, 50, 0.05, pairs=_pairs(rng, U, np.unique(item), 777))
    many.close()
    single.close()


def test_fewer_queries_than_gpus_and_none(mb, ctx, multi):
    rng = np.random.Generator(np.random.PCG64(6))
    width, depth, ptr, item, pref = _edge_model(rng)
    single, many = _pair(mb, ctx, multi, width, depth, ptr, item, pref)
    G = multi.n_gpus
    users = np.array([17, 3, 40][: max(G - 1, 1)], np.int64)      # q < G when G > 1: some GPUs get nothing
    _check_all(single, many, ptr, item, users, 12, -np.inf, pairs=(users, np.array([5, 9, 17][: users.shape[0]])))
    st = many.stats()
    assert sum(st["work"]) == users.shape[0]
    empty = np.zeros(0, np.int64)
    idx, sim, cnt = many.neighborhood(empty, 12)
    assert idx.shape == (0, 12) and sim.shape == (0, 12) and cnt.shape == (0,)
    assert many.stats()["work"] == [0] * G
    items, vals, c = many.recommend_users(empty, 12, -np.inf, *_data(ptr, item), 10)
    assert items.shape == (0, 10) and c.shape == (0,)
    assert many.estimate_prefs(empty, empty, 12).shape == (0,)
    many.close()
    single.close()


def test_edge_model(mb, ctx, multi):
    """one-pref users, users that cancel to NaN, negative prefs; finite and -inf thresholds; how_many 1 and 1024"""
    rng = np.random.Generator(np.random.PCG64(2))
    width, depth, ptr, item, pref = _edge_model(rng)
    single, many = _pair(mb, ctx, multi, width, depth, ptr, item, pref)
    U = width.shape[0]
    users = np.arange(U)
    pairs = _pairs(rng, U, np.unique(item), 400)
    for n, ms in ((80, -np.inf), (5, -0.25), (3, 0.3)):
        idx, sim, cnt = _check_all(single, many, ptr, item, users, n, ms, how_many=(1, 1024), pairs=pairs)
        if ms == -np.inf:
            assert (sim[idx >= 0] < 0).any() and cnt[4] == 0
    est = many.estimate_prefs(*pairs, 80)
    assert np.isnan(est).any() and (~np.isnan(est)).any()
    many.close()
    single.close()


def test_stats_follow_the_split(mb, ctx, multi):
    rng = np.random.Generator(np.random.PCG64(7))
    width, depth, ptr, item, pref = _edge_model(rng)
    _, many = _pair(mb, ctx, multi, width, depth, ptr, item, pref)
    G = multi.n_gpus
    for q in (1, G + 1, 59):
        users = rng.integers(0, width.shape[0], q)
        for call in (lambda: many.neighborhood(users, 7),
                     lambda: many.recommend_users(users, 7, -np.inf, *_data(ptr, item), 5)):
            call()
            st = many.stats()
            assert st["work"] == [len(range(g, q, G)) for g in range(G)]
            assert sum(st["work"]) == q
            assert len(st["seconds"]) == G and all(s >= 0 for s in st["seconds"])
            assert st["wall_s"] >= max(st["seconds"]) * 0.5
    # estimates: the j-th distinct user row (ascending) goes to GPU j mod G with all its pairs
    rows = rng.integers(0, width.shape[0], 300)
    many.estimate_prefs(rows, rng.integers(1, 200, 300), 7)
    uniq = np.unique(rows)
    gpu = np.searchsorted(uniq, rows) % G
    assert many.stats()["work"] == np.bincount(gpu, minlength=G).tolist()
    many.close()


def _launches(multi):
    from mahout_b200 import _native as N
    out = []
    for h in multi.contexts():
        n = C.c_int64()
        N.check(N.lib().mb200_launch_count(h, C.byref(n)))
        out.append(n.value)
    return out


def test_bad_arguments_then_a_good_call(mb, ctx, multi):
    from mahout_b200 import _native as N
    rng = np.random.Generator(np.random.PCG64(4))
    width, depth, ptr, item, pref = _edge_model(rng)
    single, many = _pair(mb, ctx, multi, width, depth, ptr, item, pref)
    U = width.shape[0]
    users = np.arange(U)
    item_ptr, item_col, item_ids = _data(ptr, item)

    def good():
        _check_all(single, many, ptr, item, users, 8, -np.inf, known=(False,),
                   pairs=(users, np.full(U, int(item_ids[0]), np.int64)))

    good()
    before = _launches(multi)
    host_side = [
        lambda: many.neighborhood(users, 0),
        lambda: many.neighborhood(users, 1025),
        lambda: many.neighborhood(users, 8, math.nan),
        lambda: many.recommend_users(users, 8, -np.inf, item_ptr, item_col, item_ids, 0),
        lambda: many.recommend_users(users, 8, -np.inf, item_ptr, item_col, item_ids, 1025),
        lambda: many.recommend_users(users, 0, -np.inf, item_ptr, item_col, item_ids, 10),
        lambda: many.recommend_users(users, 8, -np.inf, np.where(np.arange(U + 1) == 0, 1, item_ptr), item_col,
                                     item_ids, 10),
        lambda: many.recommend_users(users, 8, -np.inf, item_ptr + (np.arange(U + 1) == U), item_col, item_ids, 10),
        lambda: many.recommend_users(users, 8, -np.inf, item_ptr, item_col, item_ids[::-1].copy(), 10),
        lambda: many.estimate_prefs(users, users, 1025),
        lambda: many.estimate_prefs(users, users, 8, math.nan),
    ]
    L = N.lib()
    raw = [  # q < 0 and NULL arrays through the C ABI itself
        lambda: L.mb200_sized_multi_neighborhood(many.handle, None, -1, 8, 0.0, None, None, None),
        lambda: L.mb200_sized_multi_neighborhood(many.handle, None, 5, 8, 0.0, None, None, None),
        lambda: L.mb200_sized_multi_estimate_prefs(many.handle, None, None, 5, 8, 0.0, None),
        lambda: L.mb200_sized_multi_recommend(many.handle, None, 5, 8, 0.0, None, None, 0, None, 0, 10, 0, None, None,
                                              None),
        lambda: L.mb200_sized_multi_recommend(many.handle, None, -1, 8, 0.0, None, None, 0, None, 0, 10, 0, None, None,
                                              None),
    ]
    for call in host_side:
        with pytest.raises(ValueError):
            call()
    for call in raw:
        assert call() == N.ERR_BAD_ARG
    assert _launches(multi) == before                                  # nothing reached a GPU
    good()
    # a query row out of range at position 1: the second worker's share (the first's with one GPU)
    bad_rows = users.copy()
    bad_rows[1] = U
    name = f"GPU {multi.devices[1 % multi.n_gpus]}:"
    with pytest.raises(ValueError, match=name):
        many.neighborhood(bad_rows, 8)
    good()
    with pytest.raises(ValueError, match=name):
        many.recommend_users(bad_rows, 8, -np.inf, item_ptr, item_col, item_ids, 10)
    good()
    many.close()
    single.close()


def test_per_user_config_recommender_with_multi(mb, ctx, multi):
    from mahout_b200.cmconfig import CountMinSketchConfig
    from mahout_b200.cosinecm import CosineCM
    from mahout_b200.recommender import PerUserConfigUserBasedRecommender
    rng = np.random.Generator(np.random.PCG64(9))
    n, users, items = 6000, 80, 300
    user = rng.integers(1, users + 1, n).astype(np.int64) * 3
    item = rng.integers(1, items, n).astype(np.int64) * 5
    pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    ids, counts = np.unique(user, return_counts=True)
    cfg = CountMinSketchConfig(1.0)
    cfg.configure(ids, counts, items)
    cm = CosineCM(user, item, pref, 128, 3, mb.HashFunctionBuilder(SEED), ctx=ctx, config=cfg)
    one = PerUserConfigUserBasedRecommender(cm, 10, -0.5)
    many = PerUserConfigUserBasedRecommender(cm, 10, -0.5, multi=multi)
    assert many.bank is None
    _same(many.neighborhoods(), [x.cpu().numpy() for x in one.neighborhoods()])
    pick = [int(ids[5]), int(ids[41]), int(ids[41]), int(ids[0])]
    _same(many.neighborhoods(pick), [x.cpu().numpy() for x in one.neighborhoods(pick)])
    qu = rng.choice(ids, 500)
    qi = np.where(rng.random(500) < 0.8, rng.integers(1, items, 500) * 5, 7)
    _same([many.estimate_preferences(qu, qi)], [one.estimate_preferences(qu, qi)])
    for known in (False, True):
        _same(many.recommend_all(7, includeKnownItems=known), one.recommend_all(7, includeKnownItems=known))
        _same(many.recommend_all(7, pick, known), one.recommend_all(7, pick, known))
        for u in pick:
            assert many.recommend(u, 7, known) == one.recommend(u, 7, known)
    for u in pick:
        assert (many.getUserNeighborhood(u) == one.getUserNeighborhood(u)).all()
    many.multi_bank.close()
    cm.close()
