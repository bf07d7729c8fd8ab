"""CosineCM with a CountMinSketchConfig on the GPU (csrc/cmsized.cu) against the oracle: the sized bank's sketches,
the pair cosine, NearestNUserNeighborhood lists and doEstimatePreference, all bit for bit."""
import math

import numpy as np
import pytest

import oracle as orc
from oracle import sized as osz

pytestmark = pytest.mark.gpu

SEED = 11


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


@pytest.fixture(scope="module")
def ctx(mb):
    c = mb.Context(0)
    yield c
    c.close()


def _csr(user_rows, item, pref, U):
    order = np.argsort(user_rows, kind="stable")
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum(np.bincount(user_rows, minlength=U), out=ptr[1:])
    return ptr, np.asarray(item, np.int64)[order], np.asarray(pref, np.float32)[order]


def _ml100k(rng, q):
    """MovieLens-100K-shaped synthetic: 943 users x 1682 items, about 10^5 distinct prefs, shapes from the config"""
    from mahout_b200.cmconfig import CountMinSketchConfig
    U, I, n = 943, 1682, 125000
    w_user = rng.lognormal(0.0, 1.0, U)
    u = rng.choice(U, n, p=w_user / w_user.sum())
    pop = 1.0 / (np.arange(I) + 10.0) ** 0.9
    it = rng.choice(I, n, p=pop / pop.sum()) + 1
    pairs = np.unique(u.astype(np.int64) * (I + 1) + it)
    u, it = pairs // (I + 1), pairs % (I + 1)
    missing = np.setdiff1d(np.arange(U), u)                     # every user has a pref
    u = np.concatenate([u, missing])
    it = np.concatenate([it, rng.integers(1, I + 1, missing.shape[0])])
    pref = (rng.integers(1, 11, u.shape[0]) * 0.5).astype(np.float32)
    ptr, item, pref = _csr(u, it, pref, U)
    cfg = CountMinSketchConfig(q)
    cfg.configure(np.arange(U), np.diff(ptr), I)
    wd = [orc.cm_dims(cfg.getDelta(x), cfg.getEpsilon(x)) for x in range(U)]
    return (np.array([x[0] for x in wd], np.int32), np.array([x[1] for x in wd], np.int32), ptr, item, pref)


def _bank(mb, ctx, width, depth, ptr, item, pref, frac_bits=1):
    return mb.SizedBank(width, depth, mb.HashFunctionBuilder(SEED), ptr, item, pref, frac_bits, ctx)


def _check_lists(got, want):
    gi, gs, gc = (np.asarray(x.cpu() if hasattr(x, "cpu") else x) for x in got)
    wi, ws, wc = want
    assert (gc == wc).all()
    assert (gi == wi).all()
    assert gs.tobytes() == ws.tobytes()


def _oracle_lists(bank, width, depth, ptr, item, pref, queries, n, min_sim=-np.inf):
    return osz.sized_neighborhood(width, depth, bank.a, bank.b, ptr, item, pref, queries, n, min_sim)


@pytest.mark.parametrize("q", [1.0, 0.5])
def test_ml100k_neighborhoods_bit_equal(mb, ctx, q):
    rng = np.random.Generator(np.random.PCG64(1))
    width, depth, ptr, item, pref = _ml100k(rng, q)
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    U = width.shape[0]
    # sketches against orc_cm_update
    a, b = bank.a, bank.b
    for u in rng.choice(U, 40, replace=False).tolist() + [int(np.argmax(np.diff(ptr)))]:
        c = np.zeros((depth[u], width[u]))
        orc.cm_update(c, int(width[u]), int(depth[u]), a, b, item[ptr[u]:ptr[u + 1]],
                      pref[ptr[u]:ptr[u + 1]].astype(np.float64))
        assert bank.read(u).tobytes() == c.tobytes()
    allq = np.arange(U)
    _check_lists(bank.neighborhood(allq, 20), _oracle_lists(bank, width, depth, ptr, item, pref, allq, 20))
    sub = rng.choice(U, 77, replace=False)
    _check_lists(bank.neighborhood(sub, 7, 0.3), _oracle_lists(bank, width, depth, ptr, item, pref, sub, 7, 0.3))
    pl = bank.plan()
    assert pl["queries"] == 77 and pl["classes"] == len(set(zip(width.tolist(), depth.tolist())))
    # doEstimatePreference over the neighbourhoods, each neighbour's own sketch
    idx, sim, cnt = bank.neighborhood(allq, 20)
    users = rng.integers(0, U, 5000)
    its = rng.integers(1, 1683, 5000)
    got = bank.estimate_prefs(idx, sim, cnt, users, its)
    want = osz.sized_estimate(width, depth, a, b, ptr, item, pref, idx, sim, cnt, users, its)
    assert got.tobytes() == want.tobytes()
    assert np.isfinite(got).sum() > 100
    bank.close()


def _edge_model(rng):
    """one-pref users (1, 1); users whose prefs cancel in every bucket (NaN, never listed); negative prefs; a
    duplicated user (tied similarities); explicit shapes with w + 1 / d + 1 and depths up to 25"""
    prefs = []
    for u in range(60):
        k = int(rng.integers(1, 30))
        its = rng.choice(200, k, replace=False) + 1
        ps = rng.integers(-6, 11, k) * 0.5
        prefs.append((its, ps))
    prefs[3] = (np.array([17]), np.array([2.0]))                       # one pref
    prefs[4] = (np.array([5, 5]), np.array([1.5, -1.5]))               # cancels everywhere: NaN against anyone
    prefs[5] = (prefs[6][0].copy(), prefs[6][1].copy())                # identical to user 6: tied similarities
    prefs[7] = (np.array([9]), np.array([-3.0]))                       # one negative pref
    U = len(prefs)
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum([len(p[0]) for p in prefs], out=ptr[1:])
    item = np.concatenate([p[0] for p in prefs]).astype(np.int64)
    pref = np.concatenate([p[1] for p in prefs]).astype(np.float32)
    width = rng.integers(1, 40, U).astype(np.int32)
    depth = rng.integers(1, 26, U).astype(np.int32)
    width[3] = depth[3] = width[7] = depth[7] = 1
    width[5], depth[5] = width[6], depth[6]
    depth[10], width[10] = 25, 31        # d up to 25
    depth[11], width[11] = 25, 26
    width[12], depth[12] = 55, 21        # (54, 21) of the config, one wider: cm_dims' w + 1
    width[13], depth[13] = 54, 22        # and d + 1
    return width, depth, ptr, item, pref


def test_edge_cases_bit_equal(mb, ctx):
    rng = np.random.Generator(np.random.PCG64(2))
    width, depth, ptr, item, pref = _edge_model(rng)
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    U = width.shape[0]
    allq = np.arange(U)
    for n, ms in ((5, -np.inf), (80, -np.inf), (80, 0.0), (10, -0.25), (1, -np.inf)):
        got = bank.neighborhood(allq, n, ms)
        want = _oracle_lists(bank, width, depth, ptr, item, pref, allq, n, ms)
        _check_lists(got, want)
        assert 4 not in got[0][:, :].ravel().tolist()                 # NaN never admitted
        assert got[2][4] == 0
    idx, sim, cnt = bank.neighborhood(allq, 80)
    assert (cnt < 80).all()                                            # n beyond the admissible users
    assert (sim[idx >= 0] < 0).any()                                  # negative similarities listed
    # ties: users 5 and 6 are identical, so every query scores them equally; the lower row comes first
    for t in range(U):
        row = idx[t, :cnt[t]].tolist()
        if 5 in row and 6 in row:
            assert row.index(5) < row.index(6)
    # pair cosine: both directions, against the oracle primitives and against the cross cosine of two banks
    u1 = rng.integers(0, U, 400)
    u2 = rng.integers(0, U, 400)
    got = bank.pair_cosine(u1, u2)
    for t in range(400):
        x, y = int(u1[t]), int(u2[t])
        w, d = int(width[y]), int(depth[y])
        cx, cy = np.zeros((d, w)), np.zeros((d, w))
        orc.cm_update(cx, w, d, bank.a, bank.b, item[ptr[x]:ptr[x + 1]], pref[ptr[x]:ptr[x + 1]].astype(np.float64))
        orc.cm_update(cy, w, d, bank.a, bank.b, item[ptr[y]:ptr[y + 1]], pref[ptr[y]:ptr[y + 1]].astype(np.float64))
        s = orc.cm_cosine(cx, cy, w, d)
        s = s if math.isnan(s) else orc.clamp_similarity(s)
        assert np.float64(s).tobytes() == got[t].tobytes()
    hfb = mb.HashFunctionBuilder(SEED)
    for x, y in [(0, 1), (1, 0), (10, 11), (12, 13), (3, 7), (6, 5)]:
        w, d = int(width[y]), int(depth[y])
        ba = mb.SketchBank(1, w, d, hfb, 1, ctx)
        bb = mb.SketchBank(1, w, d, hfb, 1, ctx)
        ba.update(None, item[ptr[x]:ptr[x + 1]], pref[ptr[x]:ptr[x + 1]])
        bb.update(None, item[ptr[y]:ptr[y + 1]], pref[ptr[y]:ptr[y + 1]])
        import ctypes as C
        out = np.zeros(1)
        z = np.zeros(1, np.int64)
        mb._native.check(mb._native.lib().mb200_bank_cross_cosine(
            ba.handle, z.ctypes.data_as(C.c_void_p), bb.handle, z.ctypes.data_as(C.c_void_p), 1,
            out.ctypes.data_as(C.c_void_p), 0), ctx.handle)
        r = out[0] if math.isnan(out[0]) else min(1.0, max(-1.0, out[0]))
        assert np.float64(r).tobytes() == bank.pair_cosine([x], [y]).tobytes()
        ba.close()
        bb.close()
    # estimates, with a neighbourhood row per query
    users = rng.integers(0, U, 2000)
    its = rng.integers(1, 201, 2000)
    got = bank.estimate_prefs(idx, sim, cnt, users, its)
    want = osz.sized_estimate(width, depth, bank.a, bank.b, ptr, item, pref, idx, sim, cnt, users, its)
    assert got.tobytes() == want.tobytes()
    bank.close()


def test_both_accumulator_paths_and_device_memory(mb, ctx, monkeypatch, capfd):
    import torch
    rng = np.random.Generator(np.random.PCG64(3))
    width, depth, ptr, item, pref = _edge_model(rng)
    width[20], depth[20] = 3000, 7                 # 168 KB: beyond the default query-sketch budget
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    U = width.shape[0]
    allq = np.arange(U)
    want = _oracle_lists(bank, width, depth, ptr, item, pref, allq, 12)
    monkeypatch.setenv("MB200_TRACE", "1")
    _check_lists(bank.neighborhood(allq, 12), want)
    pl = bank.plan()
    assert pl["smem_classes"] > 0 and pl["global_classes"] == 1
    err = capfd.readouterr().err
    assert "sized plan: queries=60" in err and "global_classes=1" in err
    monkeypatch.setenv("MB200_SIZED_QSMEM_BYTES", "0")            # every class through the per-CTA global slice
    _check_lists(bank.neighborhood(allq, 12), want)
    pl = bank.plan()
    assert pl["smem_classes"] == 0 and pl["global_classes"] == pl["classes"]
    monkeypatch.setenv("MB200_SIZED_QSMEM_BYTES", "2048")         # tiles of one to a few queries
    _check_lists(bank.neighborhood(allq, 12), want)
    assert bank.plan()["smem_classes"] > 0
    monkeypatch.delenv("MB200_SIZED_QSMEM_BYTES")
    # device memory in and out, and a device-built bank
    dev = f"cuda:{ctx.device}"
    got = bank.neighborhood(torch.from_numpy(allq).to(dev), 12)
    assert all(x.is_cuda for x in got)
    _check_lists(got, want)
    users = torch.from_numpy(rng.integers(0, U, 500)).to(dev)
    its = torch.from_numpy(rng.integers(1, 201, 500)).to(dev)
    e_dev = bank.estimate_prefs(*got, users, its)
    e_host = bank.estimate_prefs(*(x.cpu().numpy() for x in got), users.cpu().numpy(), its.cpu().numpy())
    assert e_dev.cpu().numpy().tobytes() == e_host.tobytes()
    v2 = rng.integers(0, U, 500)
    p_dev = bank.pair_cosine(users, torch.from_numpy(v2).to(dev))
    assert p_dev.cpu().numpy().tobytes() == bank.pair_cosine(users.cpu().numpy(), v2).tobytes()
    bank2 = mb.SizedBank(width, depth, mb.HashFunctionBuilder(SEED), torch.from_numpy(ptr).to(dev),
                         torch.from_numpy(item).to(dev), torch.from_numpy(pref).to(dev), 1, ctx)
    for u in (0, 10, 20):
        assert bank2.read(u).tobytes() == bank.read(u).tobytes()
    bank2.close()
    bank.close()


def test_bad_arguments_inexact_and_range(mb, ctx):
    rng = np.random.Generator(np.random.PCG64(4))
    width, depth, ptr, item, pref = _edge_model(rng)
    hfb = mb.HashFunctionBuilder(SEED)

    def create(w=width, d=depth, p=ptr, i=item, v=pref, f=1):
        return mb.SizedBank(w, d, hfb, p, i, v, f, ctx)

    for w, d in ((np.where(np.arange(60) == 3, 0, width), depth), (width, np.where(np.arange(60) == 3, 0, depth))):
        with pytest.raises(ValueError):
            create(w=w.astype(np.int32), d=d.astype(np.int32))
    with pytest.raises(ValueError):
        create(d=np.where(np.arange(60) == 3, 33, depth).astype(np.int32))
    bad = ptr.copy()
    bad[10], bad[11] = bad[11], bad[10]
    with pytest.raises(ValueError):
        create(p=bad)
    with pytest.raises(ValueError):
        create(p=ptr + 1, i=np.concatenate([item, item[:1]]), v=np.concatenate([pref, pref[:1]]))
    v = pref.copy()
    v[5] = 0.3
    with pytest.raises(mb.InexactError) as e:
        create(v=v)
    assert e.value.code == -4
    with pytest.raises(mb.InexactError) as e:                          # a row's sum of squared quanta >= 2^53
        create(v=np.full_like(pref, 2.0 ** 26), f=1)
    assert e.value.code == -5
    bank = create()
    U = 60
    for qr in ([0, U], [-1]):
        with pytest.raises(ValueError):
            bank.neighborhood(np.array(qr), 5)
    for n in (0, 1025):
        with pytest.raises(ValueError):
            bank.neighborhood(np.arange(3), n)
    with pytest.raises(ValueError):
        bank.pair_cosine([0, 1], [2, U])
    idx, sim, cnt = bank.neighborhood(np.arange(U), 4)
    its = np.arange(1, 4)
    with pytest.raises(ValueError):
        bank.estimate_prefs(idx, sim, cnt, np.array([0, 1, U]), its)
    c2 = cnt.copy()
    c2[1] = 5
    with pytest.raises(ValueError):
        bank.estimate_prefs(idx, sim, c2, np.array([0, 1, 2]), its)
    i2 = idx.copy()
    i2[2, 0] = U + 3
    with pytest.raises(ValueError):
        bank.estimate_prefs(i2, sim, cnt, np.array([0, 1, 2]), its)
    with pytest.raises(ValueError):
        bank.estimate_prefs(idx, sim, cnt, np.array([0, 1, 2]), its, nb_row=np.array([0, 0, U]))
    bank.close()
    # RANGE at query time: own rows are in range, the re-sketch of user 0 at (1, 1) is not
    big = np.float32(3 * 2 ** 23)                                        # 3 * 2^24 quanta at frac_bits 1
    a, b = hfb.params(2)
    x = next(k for k in range(2, 1000) if all(orc.hash_one(a[i], b[i], 2, k) != orc.hash_one(a[i], b[i], 2, 1)
                                              for i in range(2)))
    rb = mb.SizedBank(np.array([2, 1], np.int32), np.array([2, 1], np.int32), hfb, np.array([0, 2, 3]),
                      np.array([1, x, 5]), np.array([big, big, 1.0], np.float32), 1, ctx)
    for call in (lambda: rb.pair_cosine([0], [1]), lambda: rb.neighborhood([0], 1)):
        with pytest.raises(mb.InexactError) as e:
            call()
        assert e.value.code == -5
    assert abs(rb.pair_cosine([1], [0])[0] - 1.0 / math.sqrt(2.0)) < 1e-15
    rb.close()


def test_cosine_cm_and_recommender(mb, ctx):
    from mahout_b200.cmconfig import CountMinSketchConfig
    from mahout_b200.cosinecm import CosineCM
    from mahout_b200.recommender import PerUserConfigUserBasedRecommender
    rng = np.random.Generator(np.random.PCG64(9))
    n, users, items = 6000, 80, 300
    user = rng.integers(1, users + 1, n).astype(np.int64) * 3
    item = rng.integers(1, items, n).astype(np.int64)
    pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    ids, counts = np.unique(user, return_counts=True)
    cfg = CountMinSketchConfig(1.0)
    cfg.configure(ids, counts, items)
    cm = CosineCM(user, item, pref, 128, 3, mb.HashFunctionBuilder(SEED), ctx=ctx, config=cfg)
    sb = cm.sized_bank()
    for r, u in enumerate(ids):
        assert (int(sb.width[r]), int(sb.depth[r])) == orc.cm_dims(cfg.getDelta(u), cfg.getEpsilon(u))
    ptr, it_s, pr_s = _csr(np.searchsorted(ids, user), item, pref, ids.shape[0])
    i1, i2 = rng.choice(ids, 300), rng.choice(ids, 300)
    got = cm.userSimilaritiesPerUserConfig(i1, i2)
    assert got.tobytes() == sb.pair_cosine(np.searchsorted(ids, i1), np.searchsorted(ids, i2)).tobytes()
    assert cm.userSimilarityPerUserConfig(int(i1[0]), int(i2[0])) == got[0] or math.isnan(got[0])
    rec = PerUserConfigUserBasedRecommender(cm, 10)
    widx, wsim, wcnt = osz.sized_neighborhood(sb.width, sb.depth, sb.a, sb.b, ptr, it_s, pr_s,
                                              np.arange(ids.shape[0]), 10)
    for r in (0, 17, 79):
        assert rec.getUserNeighborhood(int(ids[r])).tolist() == ids[widx[r, :wcnt[r]]].tolist()
    _check_lists(rec.neighborhoods(), (widx, wsim, wcnt))
    qu = rng.choice(ids, 400)
    qi = rng.integers(1, items, 400)
    got = rec.estimate_preferences(qu, qi)
    want = osz.sized_estimate(sb.width, sb.depth, sb.a, sb.b, ptr, it_s, pr_s, widx, wsim, wcnt,
                              np.searchsorted(ids, qu), qi)
    assert got.tobytes() == want.tobytes()
    cm.close()
