"""recommend() over per-user sketch sizes on the GPU (mb200_sized_recommend, k_sized_recommend) against the oracle
(oracle.sized_recommend) bit for bit -- items, value bytes, counts -- and every value against
SizedBank.estimate_prefs for the same (user, item) over the same list row."""
import numpy as np
import pytest

import oracle as orc
from oracle import recommend as orec
from oracle import sized as osz
from oracle.sized_recommend import sized_recommend

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
    missing = np.setdiff1d(np.arange(U), u)
    u = np.concatenate([u, missing])
    it = np.concatenate([it, rng.integers(1, I + 1, missing.shape[0])])
    pref = (rng.integers(1, 11, u.shape[0]) * 0.5).astype(np.float32)
    ptr, item, pref = _csr(u, it, pref, U)
    cfg = CountMinSketchConfig(q)
    cfg.configure(np.arange(U), np.diff(ptr), I)
    wd = [orc.cm_dims(cfg.getDelta(x), cfg.getEpsilon(x)) for x in range(U)]
    return (np.array([x[0] for x in wd], np.int32), np.array([x[1] for x in wd], np.int32), ptr, item, pref)


def _edge_model(rng):
    """one-pref users, users whose prefs cancel (NaN similarity and estimates), negative prefs, odd shapes up to
    depth 25"""
    prefs = []
    for u in range(60):
        k = int(rng.integers(1, 30))
        prefs.append((rng.choice(200, k, replace=False) + 1, rng.integers(-6, 11, k) * 0.5))
    prefs[3] = (np.array([17]), np.array([2.0]))
    prefs[4] = (np.array([5, 5]), np.array([1.5, -1.5]))
    prefs[7] = (np.array([9]), np.array([-3.0]))
    U = len(prefs)
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum([len(p[0]) for p in prefs], out=ptr[1:])
    item = np.concatenate([p[0] for p in prefs]).astype(np.int64)
    pref = np.concatenate([p[1] for p in prefs]).astype(np.float32)
    width = rng.integers(1, 40, U).astype(np.int32)
    depth = rng.integers(1, 26, U).astype(np.int32)
    width[3] = depth[3] = width[7] = depth[7] = 1
    return width, depth, ptr, item, pref


def _bank(mb, ctx, width, depth, ptr, item, pref):
    return mb.SizedBank(width, depth, mb.HashFunctionBuilder(SEED), ptr, item, pref, 1, ctx)


def _data(ptr, item):
    U = ptr.shape[0] - 1
    return orec.item_csr(np.repeat(np.arange(U), np.diff(ptr)), item, U)


def _np(x):
    return np.asarray(x.cpu() if hasattr(x, "cpu") else x)


def _check(bank, width, depth, ptr, item, pref, lists, data, users, how_many, known, got=None):
    """the call against the oracle bit for bit, and every value against estimate_prefs over the same list row"""
    idx, sim, cnt = (_np(x) for x in lists)
    item_ptr, item_col, item_ids = data
    if got is None:
        got = bank.recommend(idx, sim, cnt, item_ptr, item_col, item_ids, users, how_many, known)
    gi, gv, gc = (_np(x) for x in got)
    wi, wv, wc = sized_recommend(width, depth, bank.a, bank.b, ptr, item, pref, idx, sim, cnt, item_ptr, item_col,
                                 item_ids, users, how_many, known)
    assert (gc == wc).all()
    assert (gi == wi).all()
    assert gv.tobytes() == wv.tobytes()
    rows, cols = np.nonzero(gi >= 0)
    if rows.shape[0]:
        est = bank.estimate_prefs(idx, sim, cnt, np.asarray(users, np.int64)[rows], gi[rows, cols], nb_row=rows)
        assert est.tobytes() == gv[rows, cols].tobytes()
    return gi, gv, gc


@pytest.mark.parametrize("q", [1.0, 0.5])
def test_ml100k_all_users_bit_equal(mb, ctx, q):
    rng = np.random.Generator(np.random.PCG64(1))
    width, depth, ptr, item, pref = _ml100k(rng, q)
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    users = np.arange(width.shape[0])
    lists = bank.neighborhood(users, 30)
    data = _data(ptr, item)
    for how_many, known in ((10, False), (10, True), (1024, False), (1024, True)):
        _, _, gc = _check(bank, width, depth, ptr, item, pref, lists, data, users, how_many, known)
        assert gc.sum() > 0
    assert bank.recommend_plan()["users"] == users.shape[0]
    bank.close()


def test_edge_model_thresholds_and_short_lists(mb, ctx):
    rng = np.random.Generator(np.random.PCG64(2))
    width, depth, ptr, item, pref = _edge_model(rng)
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    U = width.shape[0]
    users = np.arange(U)
    data = _data(ptr, item)
    for n, ms in ((80, -np.inf), (5, -0.25), (3, 0.3)):
        lists = bank.neighborhood(users, n, ms)
        idx, sim, cnt = lists
        if ms == -np.inf:
            assert (sim[idx >= 0] < 0).any() and cnt[4] == 0
        for how_many, known in ((10, False), (200, True)):
            _check(bank, width, depth, ptr, item, pref, lists, data, users, how_many, known)
    # rows with zero and one neighbour, the user itself listed, a NaN similarity, negative similarities
    idx, sim, cnt = (x.copy() for x in bank.neighborhood(users, 6))
    cnt[0], cnt[1] = 0, 1
    idx[2, 0] = 2
    sim[3, 1] = np.nan
    sim[5, :] = -np.abs(sim[5, :]) - 0.1
    g = _check(bank, width, depth, ptr, item, pref, (idx, sim, cnt), data, users, 50, False)
    assert g[2][0] == 0 and g[2][1] == 0
    bank.close()


def test_hand_checked_infinite_and_negative_estimates(mb, ctx):
    from test_cmsized_recommend_oracle import HAND_WANT, hand_model
    width, depth, a, b, ptr, item, pref, nb_idx, nb_sim, nb_cnt = hand_model()
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    data = _data(ptr, item)
    for known, want in HAND_WANT.items():
        gi, gv, gc = bank.recommend(nb_idx, nb_sim, nb_cnt, *data, [0], 8, known)
        assert gc[0] == len(want)
        assert gi[0, :gc[0]].tolist() == [i for i, _ in want]
        assert gv[0, :gc[0]].tobytes() == np.array([v for _, v in want], np.float32).tobytes()
    bank.close()


def _plan_model(rng):
    """a catalogue past the shared-memory bitmap (about 140 000 rated items), ten heavy users (several candidate
    chunks), and shape classes that land on each read path at a 4 KiB stage: small odd sketches (whole stages), odd
    rows of a sketch too large for a stage (row stages), rows wider than a stage (gathered although streaming would
    be cheaper), and rows wider than four chunks (gathered by bytes).  Odd widths and odd depths put sketches at odd
    offsets."""
    U, I = 160, 1_000_000
    k = rng.integers(5, 120, U)
    k[:10] = 14_000
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum(k, out=ptr[1:])
    item = np.concatenate([rng.choice(I, int(x), replace=False) for x in k]).astype(np.int64) * 7 - 3
    pref = (rng.integers(-4, 11, ptr[-1]) * 0.5).astype(np.float32)
    shapes = [(3, 1), (7, 3), (33, 5), (101, 3), (301, 5), (203, 3), (1001, 1), (1999, 3), (12001, 1), (8193, 2)]
    width = np.array([shapes[u % len(shapes)][0] for u in range(U)], np.int32)
    depth = np.array([shapes[u % len(shapes)][1] for u in range(U)], np.int32)
    return width, depth, ptr, item, pref


def test_plan_paths_in_one_call_and_device_memory(mb, ctx, monkeypatch, capfd):
    import torch
    rng = np.random.Generator(np.random.PCG64(3))
    width, depth, ptr, item, pref = _plan_model(rng)
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    U = width.shape[0]
    off = np.concatenate([[0], np.cumsum(width.astype(np.int64) * depth)])
    assert (off[:-1] % 2 == 1).any() and (width % 2 == 1).all()
    users = np.concatenate([np.arange(0, 10), rng.choice(np.arange(10, U), 30, replace=False)])
    # every list holds one user of each shape class and two heavy users, with similarities of both signs
    m, ld = users.shape[0], 14
    idx = np.full((m, ld), -1, np.int64)
    sim = np.zeros((m, ld))
    for t in range(m):
        row = np.concatenate([rng.choice(np.arange(c, U, 10), 1) for c in range(10)] + [rng.choice(10, 2)])
        idx[t, :12] = rng.permutation(row)
        sim[t, :12] = rng.uniform(-0.6, 1.0, 12)
    cnt = np.full(m, 12, np.int32)
    data = _data(ptr, item)
    monkeypatch.setenv("MB200_TRACE", "1")
    monkeypatch.setenv("MB200_SIZED_REC_STAGE_BYTES", "4096")
    want = _check(bank, width, depth, ptr, item, pref, (idx, sim, cnt), data, users, 1024, False)
    pl = bank.recommend_plan()
    assert data[2].shape[0] > 131072
    assert "bitmap=global" in capfd.readouterr().err
    assert pl["stages"] == 4 and pl["stage_bytes"] == 4096
    assert pl["stream_visits"] > pl["row_visits"] > 0                  # whole-sketch and row stages
    assert pl["gather_visits"] > pl["too_wide_visits"] > 0             # gathered by bytes and too wide to stage
    assert pl["chunks"] > m and pl["candidates_max"] > pl["chunk_candidates"]
    assert pl["stream_bytes"] > 0 and pl["gather_loads"] > 0
    terms = sum(orec.candidates(int(u), idx[t], cnt[t], *data[:2], False).shape[0] * int((idx[t, :12] != u).sum())
                for t, u in enumerate(users))
    assert pl["terms"] == terms and pl["users"] == m
    # the default stages (no row too wide at these shapes): the same results; device memory
    monkeypatch.delenv("MB200_SIZED_REC_STAGE_BYTES")
    dev = f"cuda:{ctx.device}"
    td = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (idx, sim, cnt, *data, users)]
    got = bank.recommend(*td, 1024, False)
    assert all(isinstance(x, torch.Tensor) and x.is_cuda for x in got)
    for g, w in zip(got, want):
        assert _np(g).tobytes() == w.tobytes()
    pl = bank.recommend_plan()
    assert pl["stage_bytes"] > 4096 and pl["too_wide_visits"] == 0 and pl["stream_visits"] > 0
    # no stages at all: everything gathered, the same results
    monkeypatch.setenv("MB200_SIZED_REC_STAGE_BYTES", "0")
    got = bank.recommend(idx, sim, cnt, *data, users, 1024, False)
    for g, w in zip(got, want):
        assert _np(g).tobytes() == w.tobytes()
    assert bank.recommend_plan()["stream_visits"] == 0
    bank.close()


def test_bad_arguments_then_a_good_call(mb, ctx):
    import torch
    rng = np.random.Generator(np.random.PCG64(4))
    width, depth, ptr, item, pref = _edge_model(rng)
    bank = _bank(mb, ctx, width, depth, ptr, item, pref)
    U = width.shape[0]
    users = np.arange(U)
    idx, sim, cnt = bank.neighborhood(users, 8)
    item_ptr, item_col, item_ids = _data(ptr, item)
    want = sized_recommend(width, depth, bank.a, bank.b, ptr, item, pref, idx, sim, cnt, item_ptr, item_col,
                           item_ids, users, 10)

    def good():
        got = bank.recommend(idx, sim, cnt, item_ptr, item_col, item_ids, users, 10)
        for g, w in zip(got, want):
            assert g.tobytes() == w.tobytes()

    def bad(**kw):
        a = dict(nb_idx=idx, nb_sim=sim, nb_cnt=cnt, item_ptr=item_ptr, item_col=item_col, item_ids=item_ids,
                 users=users, how_many=10)
        a.update(kw)
        dev = a.pop("device", False)
        if dev:
            d = f"cuda:{ctx.device}"
            a = {k: (torch.from_numpy(np.ascontiguousarray(v)).to(d) if isinstance(v, np.ndarray) else v)
                 for k, v in a.items()}
        with pytest.raises(ValueError):
            bank.recommend(**a)
        good()

    bad(how_many=0)
    bad(how_many=1025)
    bad(users=np.where(users == 5, U, users))                          # user row out of range
    bad(users=np.where(users == 5, -1, users))
    c = cnt.copy()
    c[3] = 9                                                           # count beyond nb_ld
    bad(nb_cnt=c)
    c[3] = -1
    bad(nb_cnt=c)
    i = idx.copy()
    i[7, 0] = U                                                        # neighbour index out of range
    bad(nb_idx=i)
    p = item_ptr.copy()
    p[0] = 1                                                           # checked on the host
    bad(item_ptr=p)
    p = item_ptr.copy()
    p[U] += 1
    bad(item_ptr=p)
    p = item_ptr.copy()
    p[20] = p[21] + 1                                                  # descending range: counted on the device
    bad(item_ptr=p, device=True)
    p = item_ptr.copy()
    p[U] = p[U] + 1000                                                 # past nnz
    bad(item_ptr=p, device=True)
    col = item_col.copy()
    col[4] = item_ids.shape[0]                                         # item_col entry out of range
    bad(item_col=col)
    col[4] = -1
    bad(item_col=col, device=True)
    ids = item_ids.copy()
    ids[[3, 4]] = ids[[4, 3]]                                          # itemIDs not ascending
    bad(item_ids=ids)
    with pytest.raises(ValueError):                                    # list rows != users
        bank.recommend(idx[:-1], sim[:-1], cnt[:-1], item_ptr, item_col, item_ids, users, 10)
    good()
    bank.close()


def test_recommender_recommend_and_recommend_all(mb, ctx):
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
    sb = cm.sized_bank()
    rows = np.searchsorted(ids, user)
    ptr, it_s, pr_s = _csr(rows, item, pref, ids.shape[0])
    rec = PerUserConfigUserBasedRecommender(cm, 10, -0.5)
    q = np.arange(ids.shape[0])
    widx, wsim, wcnt = osz.sized_neighborhood(sb.width, sb.depth, sb.a, sb.b, ptr, it_s, pr_s, q, 10, -0.5)
    item_ptr, item_col, item_ids = orec.item_csr(rows, item, ids.shape[0])
    for known in (False, True):
        wi, wv, wc = sized_recommend(sb.width, sb.depth, sb.a, sb.b, ptr, it_s, pr_s, widx, wsim, wcnt, item_ptr,
                                     item_col, item_ids, q, 7, known)
        got_ids, gi, gv, gc = rec.recommend_all(7, includeKnownItems=known)
        assert (got_ids == ids).all()
        assert (gc == wc).all() and (gi == wi).all() and gv.tobytes() == wv.tobytes()
        pick = [int(ids[0]), int(ids[41]), int(ids[41]), int(ids[79])]
        got_ids, gi, gv, gc = rec.recommend_all(7, pick, known)
        r = np.searchsorted(ids, pick)
        assert (gc == wc[r]).all() and (gi == wi[r]).all() and gv.tobytes() == wv[r].tobytes()
        for u in pick:
            t = int(np.searchsorted(ids, u))
            assert rec.recommend(u, 7, known) == [(int(i), float(v)) for i, v in zip(wi[t, :wc[t]], wv[t, :wc[t]])]
    assert wc.sum() > 0
    cm.close()
