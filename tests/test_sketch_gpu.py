"""GPU parity of the sketch stage (K1 update, hash, point query, pair cosine) against the CPU
oracle, through the C ABI.  Bar: bit-exact counters / hashes / point queries; FP64 pair cosine
within 1e-12 relative (summation order differs from the reference's sequential loop)."""
import json
import math
import os

import numpy as np
import pytest

import oracle as orc

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


@pytest.fixture(scope="module")
def ctx(mb):
    c = mb.Context(0)
    yield c
    c.close()


def _events(rng, n, E, key_lo, key_hi, halves=True):
    ent = rng.integers(0, E, n).astype(np.int64)
    key = rng.integers(key_lo, key_hi, n).astype(np.int64)
    inc = (rng.integers(1, 11, n) * (0.5 if halves else 1.0)).astype(np.float32)
    return ent, key, inc


def test_hash_matches_oracle_and_survey_anchors(mb, ctx):
    hfb = mb.HashFunctionBuilder(42)
    keys = np.array([0, 1, 2, 1682, 10 ** 12, -1, 2 ** 63 - 1, -2 ** 63, 2 ** 63 - 25, -(2 ** 63 - 25)],
                    np.int64)
    want0 = [671704, 767226, 862723, 888455, 1047010, 576207]
    h0 = hfb.getHashFunction(0, 1 << 20)
    h0._ctx = ctx
    assert h0.hash(keys)[:6].tolist() == want0
    rng = np.random.Generator(np.random.PCG64(11))
    big = rng.integers(-2 ** 63, 2 ** 63 - 1, 100000, dtype=np.int64)
    oa, ob = orc.hash_params(42, 4)
    for i in range(4):
        for w in (1 << 20, 4096, 4099, 1, 2 ** 31 - 1):
            hf = mb.HashFunction(int(oa[i]), int(ob[i]), w, ctx)
            for ks in (keys, big):
                assert (hf.hash(ks) == orc.hash_many(oa[i], ob[i], w, ks)).all()
    # Math.abs(Long.MIN_VALUE) < 0 corner of the parameters
    hf = mb.HashFunction(-2 ** 63, -2 ** 63, 4096, ctx)
    assert (hf.hash(big[:1000]) == orc.hash_many(-2 ** 63, -2 ** 63, 4096, big[:1000])).all()


def test_golden_fixture_counters_bit_exact(mb, ctx):
    g = json.load(open(os.path.join(GOLD, "sketch_small.json")))
    bank = mb.SketchBank(g["E"], g["w"], g["d"], mb.HashFunctionBuilder(g["seed"]), 1, ctx)
    bank.update(np.array(g["entity"]), np.array(g["key"]), np.array(g["inc"], np.float32))
    got = bank.read().ravel()
    want = np.zeros_like(got)
    want[np.array(g["nonzero_cells"])] = g["nonzero_values"]
    assert got.tobytes() == want.tobytes()
    bank.close()


@pytest.mark.parametrize("E,d,w,n", [(1, 4, 1 << 20, 300000), (1, 4, 4096, 100001), (1, 3, 1000, 7),
                                      (1682, 4, 4096, 100000), (37, 5, 129, 50003), (5, 16, 64, 1000)])
def test_update_bit_exact_host_and_device(mb, ctx, E, d, w, n):
    import torch
    rng = np.random.Generator(np.random.PCG64(1000 + E + d + w))
    ent, key, inc = _events(rng, n, E, -1000, 1000000)
    if E == 1:
        # heavy skew: exercises the shared-memory hot-key cache
        key = np.minimum(rng.zipf(1.1, n), 10 ** 7).astype(np.int64)
    a, b = orc.hash_params(42, d)
    want = np.zeros((E, d, w))
    orc.bank_update(want, d, w, a, b, ent if E > 1 else None, key, inc)
    for where in ("host", "device"):
        bank = mb.SketchBank(E, w, d, 42, 1, ctx)
        if where == "host":
            bank.update(ent if E > 1 else None, key, inc)
        else:
            te = torch.from_numpy(ent).cuda() if E > 1 else None
            bank.update(te, torch.from_numpy(key).cuda(), torch.from_numpy(inc).cuda())
        got = bank.read()
        assert got.tobytes() == want.tobytes(), where
        # point queries (DoubleCountMinSketch.get), including keys never inserted
        qk = np.concatenate([key[:500], rng.integers(-50, 50, 100)]).astype(np.int64)
        qe = np.concatenate([ent[:500], rng.integers(0, E, 100)]).astype(np.int64)
        q = bank.query(qe if E > 1 else None, qk)
        assert q.tobytes() == orc.bank_query(want, d, w, a, b, qe if E > 1 else None, qk).tobytes()
        bank.close()


def _zipf_entities(rng, n, E, s=1.2):
    """entity stream with a heavy head (one entity owns a few windows of the grouped update) and empty tails"""
    return (np.minimum(rng.zipf(s, n), E) - 1).astype(np.int64)


@pytest.mark.parametrize("E,d,w,n,keys", [
    (1682, 4, 4096, 300000, "small"),      # one partition level, tile path + sparse path
    (5000, 4, 4096, 400000, "small"),      # two partition levels
    (40000, 1, 512, 500000, "small"),      # d = 1, mostly sparse entities, many empty ones
    (3000, 5, 1000, 200000, "mixed"),      # generic depth, non-power-of-two width, keys outside [0, 2^32)
    (2100, 16, 4096, 150000, "small"),     # the tile (256 KB) does not fit shared memory: direct path on grouped records
    (2, 4, 4096, 200000, "small"),         # every window inside one entity: shared (atomic) tile flushes
    (700, 4, 4099, 150000, "small"),       # d * w not a multiple of 4: scalar flush
])
def test_grouped_update_bit_exact(mb, ctx, E, d, w, n, keys):
    """bank-mode K1 through the device-side grouping (group.cu) == the oracle, bit for bit, on host and
    device inputs; the direct kernel (grouping off) gives the same bank."""
    import torch
    from mahout_b200 import _native as N
    rng = np.random.Generator(np.random.PCG64(77 + E + d))
    ent = _zipf_entities(rng, n, E)
    if keys == "small":
        key = rng.integers(0, 200000, n).astype(np.int64)
        inc = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    else:
        key = rng.integers(-2 ** 40, 2 ** 40, n).astype(np.int64)
        key[::3] = rng.integers(0, 1000, key[::3].shape[0])
        inc = (rng.integers(-20, 21, n) * 0.5).astype(np.float32)
        inc[::7] = 40000.0                                      # |quanta| >= 2^15: the wide path
    a, b = orc.hash_params(42, d)
    want = np.zeros((E, d, w))
    orc.bank_update(want, d, w, a, b, ent, key, inc)
    try:
        for gmin in (0, 1 << 62):
            ctx.set_option(N.OPT_GROUP_MIN_EVENTS, gmin)
            for where in ("device", "host"):
                bank = mb.SketchBank(E, w, d, 42, 1, ctx)
                if where == "host":
                    bank.update(ent, key, inc)
                else:
                    bank.update(torch.from_numpy(ent).cuda(), torch.from_numpy(key).cuda(), torch.from_numpy(inc).cuda())
                    bank.update(torch.from_numpy(ent).cuda()[:1000], torch.from_numpy(key).cuda()[:1000],
                                -torch.from_numpy(inc).cuda()[:1000])      # additive: a second call cancels a prefix
                    bank.update(torch.from_numpy(ent).cuda()[:1000], torch.from_numpy(key).cuda()[:1000],
                                torch.from_numpy(inc).cuda()[:1000])
                bank.check()
                assert bank.read().tobytes() == want.tobytes(), (gmin, where)
                bank.close()
    finally:
        ctx.set_option(N.OPT_GROUP_MIN_EVENTS, 1 << 16)


def test_grouped_csr_update_and_errors(mb, ctx):
    """mb200_bank_update_grouped: one preference array per entity (CosineCM.exportProfile's shape)."""
    import torch
    from mahout_b200 import _native as N
    rng = np.random.Generator(np.random.PCG64(91))
    E, d, w, n = 900, 4, 4096, 250000
    ent = np.sort(_zipf_entities(rng, n, E))
    key = rng.integers(-5, 2 ** 33, n).astype(np.int64)
    inc = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    row_ptr = np.searchsorted(ent, np.arange(E + 1)).astype(np.int64)
    a, b = orc.hash_params(42, d)
    want = np.zeros((E, d, w))
    orc.bank_update(want, d, w, a, b, ent, key, inc)
    for where in ("host", "device"):
        bank = mb.SketchBank(E, w, d, 42, 1, ctx)
        if where == "host":
            bank.update_grouped(row_ptr, key, inc)
        else:
            bank.update_grouped(torch.from_numpy(row_ptr).cuda(), torch.from_numpy(key).cuda(), torch.from_numpy(inc).cuda())
        bank.check()
        assert bank.read().tobytes() == want.tobytes(), where
        bank.close()
    bank = mb.SketchBank(E, w, d, 42, 1, ctx)
    bad = row_ptr.copy()
    bad[10] = bad[11] + 3
    with pytest.raises(ValueError):
        bank.update_grouped(torch.from_numpy(bad).cuda(), torch.from_numpy(key).cuda(), torch.from_numpy(inc).cuda())
    bank.close()
    # grouped path keeps the status words: a bad entity and an inexact increment still surface
    ctx.set_option(N.OPT_GROUP_MIN_EVENTS, 0)
    try:
        bank = mb.SketchBank(50, 64, 2, 42, 1, ctx)
        e = rng.integers(0, 50, 5000).astype(np.int64)
        e[17] = 50
        bank.update(e, np.arange(5000), np.ones(5000, np.float32))
        with pytest.raises(ValueError):
            bank.check()
        bank.close()
        bank = mb.SketchBank(50, 64, 2, 42, 1, ctx)
        v = np.ones(5000, np.float32)
        v[99] = 0.3
        bank.update(rng.integers(0, 50, 5000).astype(np.int64), np.arange(5000), v)
        with pytest.raises(mb.InexactError):
            bank.check()
        bank.close()
    finally:
        ctx.set_option(N.OPT_GROUP_MIN_EVENTS, 1 << 16)


@pytest.mark.parametrize("E", [1, 700])
def test_narrow_wire_format_bit_exact(mb, ctx, E):
    """mb200_bank_update_u8 (u32 keys, one byte of quanta per event) == the (int64, float) update, host and device,
    aligned and not; mb200_bank_read_i32 gives the same counters as quanta."""
    import torch
    rng = np.random.Generator(np.random.PCG64(31 + E))
    n, d, w = 200003, 4, 4096
    key = np.minimum(rng.zipf(1.1, n), 2 ** 32 - 1).astype(np.uint32)
    key[:5] = [0, 1, 2 ** 32 - 1, 2 ** 31, 7]
    ent = rng.integers(0, E, n).astype(np.uint32)
    quanta = rng.integers(0, 256, n).astype(np.uint8)
    a, b = orc.hash_params(42, d)
    want = np.zeros((E, d, w))
    orc.bank_update(want, d, w, a, b, ent.astype(np.int64) if E > 1 else None, key.astype(np.int64),
                    (quanta * 0.5).astype(np.float32))
    for where in ("host", "device", "device_unaligned"):
        bank = mb.SketchBank(E, w, d, 42, 1, ctx)
        if where == "host":
            bank.update_u8(ent if E > 1 else None, key, quanta)
        else:
            o = 1 if where.endswith("unaligned") else 0
            tk = torch.from_numpy(key.view(np.int32)).cuda()[o:]
            te = torch.from_numpy(ent.view(np.int32)).cuda()[o:] if E > 1 else None
            tq = torch.from_numpy(quanta).cuda()[o:]
            bank.update_u8(te, tk, tq)
            if o:
                bank.update_u8(te[:0] if E > 1 else None, tk[:0], tq[:0])
                bank.update_u8(torch.from_numpy(ent.view(np.int32)).cuda()[:1] if E > 1 else None,
                               torch.from_numpy(key.view(np.int32)).cuda()[:1], torch.from_numpy(quanta).cuda()[:1])
        bank.check()
        assert bank.read().tobytes() == want.tobytes(), where
        assert (bank.read_i32() == np.rint(want * 2).astype(np.int32)).all()
        bank.close()


def test_update_unaligned_and_tail(mb, ctx):
    """odd offsets defeat the 16-byte vector loads; n % 4 != 0 exercises the tail."""
    import torch
    rng = np.random.Generator(np.random.PCG64(5))
    n = 4099
    ent, key, inc = _events(rng, n + 1, 9, 0, 500)
    a, b = orc.hash_params(42, 4)
    want = np.zeros((9, 4, 256))
    orc.bank_update(want, 4, 256, a, b, ent[1:], key[1:], inc[1:])
    bank = mb.SketchBank(9, 256, 4, 42, 1, ctx)
    bank.update(torch.from_numpy(ent).cuda()[1:], torch.from_numpy(key).cuda()[1:],
                torch.from_numpy(inc).cuda()[1:])
    assert bank.read().tobytes() == want.tobytes()
    bank.close()


def test_empty_update_and_clear(mb, ctx):
    bank = mb.SketchBank(3, 64, 2, 42, 1, ctx)
    bank.update(np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.float32))
    assert not bank.read().any()
    bank.update(np.array([1]), np.array([5]), np.array([2.5], np.float32))
    assert bank.read().sum() == 5.0
    bank.clear()
    assert not bank.read().any()
    bank.close()


def test_negative_and_f64_increments(mb, ctx):
    rng = np.random.Generator(np.random.PCG64(6))
    n = 20000
    ent = rng.integers(0, 4, n).astype(np.int64)
    key = rng.integers(-30, 30, n).astype(np.int64)
    inc = (rng.integers(-20, 21, n) * 0.125)
    a, b = orc.hash_params(7, 4)
    want = np.zeros((4, 4, 32))
    for e in range(4):
        m = ent == e
        orc.cm_update(want[e], 32, 4, a, b, key[m], inc[m])
    bank = mb.SketchBank(4, 32, 4, 7, 3, ctx)
    bank.update(ent, key, inc.astype(np.float64))
    assert bank.read().tobytes() == want.tobytes()
    bank.close()


def test_inexact_increment_is_an_error_not_a_rounding(mb, ctx):
    bank = mb.SketchBank(1, 64, 2, 42, 1, ctx)
    bank.update(None, np.array([1, 2]), np.array([0.5, 0.3], np.float32))
    with pytest.raises(mb.InexactError):
        bank.check()
    bank.close()


def test_bad_entity_and_bad_args(mb, ctx):
    bank = mb.SketchBank(4, 64, 2, 42, 1, ctx)
    bank.update(np.array([0, 4]), np.array([1, 2]), np.array([1.0, 1.0], np.float32))
    with pytest.raises(ValueError):
        bank.check()
    bank.close()
    with pytest.raises(ValueError):
        mb.SketchBank(4, 0, 2, 42, 1, ctx)
    with pytest.raises(ValueError):
        mb.SketchBank(4, 16, 0, 42, 1, ctx)
    with pytest.raises(mb.CMException):
        mb.DoubleCountMinSketch(0.9, 0.01, mb.HashFunctionBuilder(1))


def test_double_count_min_sketch_api(mb, ctx):
    """Reads like a test of the Java class: update / get / cosine, widths must agree."""
    hfb = mb.HashFunctionBuilder(42)
    x = [0, 2, 0, 0, 8, 3, 0, 6, 0, 1, 2, 2, 0]
    y = [3, 0, 0, 0, 7, 0, 2, 2, 1, 3, 2, 1, 1]
    # wide enough that the 13 keys do not collide in any row -> sketch cosine == exact cosine,
    # which the reference pins (VectorSimilarityMeasuresTest.testCosineSimilarity: 0.769846046)
    cma = mb.DoubleCountMinSketch(1 << 16, 4, hfb, ctx=ctx)
    cmb = mb.DoubleCountMinSketch(1 << 16, 4, hfb, ctx=ctx)
    for k, (xa, xb) in enumerate(zip(x, y)):
        if xa:
            cma.update(k, float(xa))
        if xb:
            cmb.update(k, float(xb))
    assert cma.get(4) == 8.0 and cmb.get(4) == 7.0 and cma.get(0) == 0.0
    cos = mb.DoubleCountMinSketch.cosine(cma, cmb)
    assert abs(cos - 0.769846046) < 1e-6
    assert abs(cos - orc.cm_cosine(cma.counts(), cmb.counts(), 1 << 16, 4)) < 1e-14
    other = mb.DoubleCountMinSketch(1 << 10, 4, hfb, ctx=ctx)
    with pytest.raises(ValueError, match="Widths of a"):
        mb.DoubleCountMinSketch.cosine(cma, other)
    empty = mb.DoubleCountMinSketch(1 << 16, 4, hfb, ctx=ctx)
    assert math.isnan(mb.DoubleCountMinSketch.cosine(cma, empty))


def test_pair_cosine_matches_oracle(mb, ctx):
    rng = np.random.Generator(np.random.PCG64(8))
    E, d, w, n = 20, 4, 512, 30000
    ent, key, inc = _events(rng, n, E - 1, 0, 3000)   # entity E-1 stays empty -> NaN
    a, b = orc.hash_params(42, d)
    ref = np.zeros((E, d, w))
    orc.bank_update(ref, d, w, a, b, ent, key, inc)
    bank = mb.SketchBank(E, w, d, 42, 1, ctx)
    bank.update(ent, key, inc)
    ea = rng.integers(0, E, 200).astype(np.int64)
    eb = rng.integers(0, E, 200).astype(np.int64)
    got = bank.pair_cosine(ea, eb)
    want = np.array([orc.cm_cosine(ref[x], ref[y], w, d) for x, y in zip(ea, eb)])
    assert (np.isnan(got) == np.isnan(want)).all()
    m = ~np.isnan(want)
    assert np.max(np.abs(got[m] - want[m]) / np.abs(want[m])) < 1e-12
    bank.close()


def test_synth_stream_device_equals_numpy(mb, ctx):
    import torch
    from mahout_b200 import synth
    cdf = synth.zipf_cdf(100000, 1.1)
    perm = synth.rank_permutation(100000, 3)
    cd = torch.from_numpy(cdf).cuda()
    pd = torch.from_numpy(perm).cuda()
    u, i, p = synth.events_device(ctx, 20240002, 12345, 200001, 943, cd, pd)
    hu, hi, hp = synth.events_numpy(20240002, 12345, 200001, 943, cdf, perm)
    assert (u.cpu().numpy() == hu).all() and (i.cpu().numpy() == hi).all()
    assert (p.cpu().numpy() == hp).all()
    # Zipf head really is heavy
    top = perm[0]
    assert (hi == top).mean() > 0.05


def test_cosine_cm_user_similarity(mb, ctx):
    """CosineCM.userSimilarity / exported profiles / the point query of doEstimatePreference."""
    from mahout_b200.cosinecm import CosineCM
    rng = np.random.Generator(np.random.PCG64(21))
    n, users, items, w, d = 3000, 40, 300, 256, 3
    user = rng.integers(100, 100 + users, n).astype(np.int64) * 7       # arbitrary (non-dense) user IDs
    item = rng.integers(1, items, n).astype(np.int64)
    pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    cm = CosineCM(user, item, pref, w, d, mb.HashFunctionBuilder(42), ctx=ctx)
    a, b = orc.hash_params(42, d)
    ids = np.unique(user)
    ref = {}
    for u in ids:
        c = np.zeros((d, w))
        m = user == u
        orc.cm_update(c, w, d, a, b, item[m], pref[m].astype(np.float64))
        ref[int(u)] = c
    for u1, u2 in [(ids[0], ids[1]), (ids[3], ids[3]), (ids[5], ids[17])]:
        want = orc.clamp_similarity(orc.cm_cosine(ref[int(u1)], ref[int(u2)], w, d))
        assert abs(cm.userSimilarity(int(u1), int(u2)) - want) < 1e-12
    assert cm.getExportedCMProfile(int(ids[2])).tobytes() == ref[int(ids[2])].tobytes()
    u = int(ids[4])
    it = int(item[user == u][0])
    assert cm.estimatePreference(u, it) == float(np.float32(orc.cm_get(ref[u], w, d, a, b, it)))
    with pytest.raises(KeyError):
        cm.userSimilarity(1, 2)
    with pytest.raises(RuntimeError, match="CountMinSketch error"):
        CosineCM(user, item, pref, 0.9, 0.01, 42, ctx=ctx)
    near, sims = cm.mostSimilarUserIDs(u, 5)
    assert len(near) == 5 and u not in near.tolist() and (np.diff(sims) <= 0).all()
    cm.close()


def test_cosine_cm_per_user_config_and_estimate_preference(mb, ctx):
    """The reference's per-pair sizing (u1's sketch rebuilt with u2's (delta, epsilon), CosineCM.java:84-96)
    with a CountMinSketchConfig, and GenericUserBasedRecommender.doEstimatePreference (:134-184) over a
    neighbourhood -- against the oracle's sketches."""
    import math
    from mahout_b200.cmconfig import CountMinSketchConfig
    from mahout_b200.cosinecm import CosineCM
    rng = np.random.Generator(np.random.PCG64(33))
    n, users, items = 2500, 30, 200
    user = rng.integers(1, users + 1, n).astype(np.int64)
    item = rng.integers(1, items, n).astype(np.int64)
    pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    ids, counts = np.unique(user, return_counts=True)
    cfg = CountMinSketchConfig(1.0)
    cfg.configure(ids, counts, items)
    hfb = mb.HashFunctionBuilder(7)
    cm = CosineCM(user, item, pref, 128, 3, hfb, ctx=ctx, config=cfg)
    for u1, u2 in [(1, 2), (5, 9), (9, 5), (3, 3)]:
        w, d = orc.cm_dims(cfg.getDelta(u2), cfg.getEpsilon(u2))
        a, b = orc.hash_params(7, d)
        c1, c2 = np.zeros((d, w)), np.zeros((d, w))
        orc.cm_update(c1, w, d, a, b, item[user == u1], pref[user == u1].astype(np.float64))
        orc.cm_update(c2, w, d, a, b, item[user == u2], pref[user == u2].astype(np.float64))
        want = orc.cm_cosine(c1, c2, w, d)
        want = want if math.isnan(want) else orc.clamp_similarity(want)
        got = cm.userSimilarityPerUserConfig(u1, u2)
        assert (math.isnan(got) and math.isnan(want)) or abs(got - want) < 1e-12
    # doEstimatePreference over the shared-size bank
    w, d = 128, 3
    a, b = orc.hash_params(7, d)
    ref = {}
    for u in ids:
        c = np.zeros((d, w))
        orc.cm_update(c, w, d, a, b, item[user == u], pref[user == u].astype(np.float64))
        ref[int(u)] = c
    the_user, nb, it = 4, [2, 4, 6, 8, 10, 12], int(item[user == 6][0])
    preference = total = 0.0
    count = 0
    for u in nb:
        if u == the_user:
            continue
        p = float(np.float32(orc.cm_get(ref[u], w, d, a, b, it)))
        if p == 0.0:
            continue
        s = orc.clamp_similarity(orc.cm_cosine(ref[the_user], ref[u], w, d))
        if not math.isnan(s):
            preference += s * p
            total += s
            count += 1
    want = math.nan if count <= 1 else float(np.float32(preference / total))
    got = cm.doEstimatePreference(the_user, nb, it)
    assert (math.isnan(got) and math.isnan(want)) or got == want
    assert math.isnan(cm.doEstimatePreference(the_user, [], it))
    assert math.isnan(cm.doEstimatePreference(the_user, [the_user], it))
    cm.close()


def test_full_size_properties_config2(mb, ctx):
    """Size-independent properties at BASELINE config-2 scale (2^28 device-generated Zipf events,
    d=4 x W=2^20): every sketch row holds exactly the total mass, the update is linear (two halves
    into one sketch == sum of two sketches), and a prefix agrees bit for bit with the oracle."""
    import torch
    from mahout_b200 import synth
    n, d, w = 1 << 28, 4, 1 << 20
    cdf = synth.zipf_cdf(10_000_000, 1.1)
    cd = torch.from_numpy(cdf).cuda()
    _, item, pref = synth.events_device(ctx, 20240002, 0, n, 1_000_000, cd, None, want_user=False)
    whole = mb.SketchBank(1, w, d, 42, 1, ctx)
    whole.update(None, item, pref)
    whole.check()
    c = whole.counters_tensor()                                   # int64 quanta [1, d, w]
    total = int((pref.double() * 2).sum().item())
    assert c.sum(dim=2).flatten().tolist() == [total] * d         # mass conservation per row
    h1 = mb.SketchBank(1, w, d, 42, 1, ctx)
    h2 = mb.SketchBank(1, w, d, 42, 1, ctx)
    h1.update(None, item[: n // 2], pref[: n // 2])
    h2.update(None, item[n // 2:], pref[n // 2:])
    assert torch.equal(h1.counters_tensor() + h2.counters_tensor(), c)   # linearity
    # point queries never under-estimate (count-min property) on the hottest keys
    keys = torch.arange(1, 1001, device="cuda")
    est = torch.from_numpy(whole.query(None, keys.cpu().numpy()))
    true = torch.zeros(1001, dtype=torch.float64, device="cuda").index_add_(
        0, item.clamp(max=1000), torch.where(item <= 1000, pref.double(), torch.zeros_like(pref).double()))[1:]
    assert (est >= true.cpu() - 1e-9).all()
    m = 1 << 22
    a, b = orc.hash_params(42, d)
    ref = np.zeros((1, d, w))
    orc.bank_update(ref, d, w, a, b, None, item[:m].cpu().numpy(), pref[:m].cpu().numpy(), nthreads=orc.max_threads())
    pre = mb.SketchBank(1, w, d, 42, 1, ctx)
    pre.update(None, item[:m], pref[:m])
    assert pre.read().tobytes() == ref.tobytes()
    for bk in (whole, h1, h2, pre):
        bk.close()


def test_context_stats(mb, ctx):
    st = ctx.stats()
    assert st["num_sms"] >= 100 and st["launches"] >= 0 and "B200" in st["device_name"]
    bank = mb.SketchBank(300, 256, 2, 42, 1, ctx)
    bank.update(np.arange(300), np.arange(300), np.ones(300, np.float32))
    bank.cosine_topk(5)
    st2 = ctx.stats()
    assert st2["launches"] > st["launches"] and st2["workspace_bytes"] > 0 and st2["cosine_job_active"] == 0
    bank.close()


def test_bank_dump_and_load_round_trip(mb, ctx, tmp_path):
    """checkpoint: a loaded bank has the dumped counters, hash family and quantum, keeps accepting updates, and a
    truncated or foreign file is refused"""
    rng = np.random.Generator(np.random.PCG64(44))
    E, d, w, n = 37, 3, 1000, 20000
    ent, key, inc = _events(rng, n, E, -50, 100000)
    bank = mb.SketchBank(E, w, d, 1234, 1, ctx)
    bank.update(ent, key, inc)
    path = str(tmp_path / "bank.mb200")
    bank.dump(path)
    back = mb.SketchBank.load(path, ctx)
    assert (back.E, back.d, back.w, back.frac_bits) == (E, d, w, 1)
    assert back.a.tolist() == bank.a.tolist() and back.b.tolist() == bank.b.tolist()
    assert back.read().tobytes() == bank.read().tobytes()
    bank.update(ent[:500], key[:500], inc[:500])
    back.update(ent[:500], key[:500], inc[:500])
    assert back.read().tobytes() == bank.read().tobytes()
    q = rng.integers(-50, 100000, 300).astype(np.int64)
    qe = rng.integers(0, E, 300).astype(np.int64)
    assert back.query(qe, q).tobytes() == bank.query(qe, q).tobytes()
    raw = open(path, "rb").read()
    open(path, "wb").write(raw[:len(raw) // 2])
    with pytest.raises(ValueError, match="truncated"):
        mb.SketchBank.load(path, ctx)
    open(path, "wb").write(b"not a dump at all" * 100)
    with pytest.raises(ValueError, match="not a bank dump"):
        mb.SketchBank.load(path, ctx)
    st = ctx.stats()
    assert st["events_updated"] > 0 and st["h2d_bytes"] > 0 and st["d2h_bytes"] > 0
    bank.close()
    back.close()


def test_single_sketch_update_bit_exact(mb, ctx):
    """The single-sketch K1 (2-way shared-memory cache in one 1024-thread CTA per SM) gives the oracle's counters on
    a Zipf stream with keys outside the 32-bit tag range, keys equal to 2^32 - 1, negative increments and the n % 4
    tail, from host and from device memory."""
    import torch
    rng = np.random.Generator(np.random.PCG64(71))
    n, d, w = 400003, 4, 1 << 16
    key = np.minimum(rng.zipf(1.1, n), 10 ** 7).astype(np.int64)
    key[::50] = rng.integers(-2 ** 62, 2 ** 62, key[::50].shape[0])
    key[1::97] = 2 ** 32 - 1
    inc = (rng.integers(-6, 11, n) * 0.5).astype(np.float32)
    a, b = orc.hash_params(42, d)
    want = np.zeros((1, d, w))
    orc.bank_update(want, d, w, a, b, None, key, inc)
    for dev in (False, True):
        bank = mb.SketchBank(1, w, d, 42, 1, ctx)
        if dev:
            bank.update(None, torch.from_numpy(key).cuda(), torch.from_numpy(inc).cuda())
        else:
            bank.update(None, key, inc)
        bank.check()
        assert bank.read().tobytes() == want.tobytes(), dev
        bank.close()


def test_set_option_rejects_unknown_options(mb):
    """Option 3 (the removed single-sketch kernel selector) is unknown: mb200_set_option fails with
    MB200_ERR_BAD_ARG.  Options 1 (GROUP_MIN_EVENTS), 2 (GROUP_PREFETCH) and 4 (MAX_FALLBACK_ROWS) still take
    values."""
    from mahout_b200 import _native as N
    c = mb.Context(0)
    try:
        for val in (0, 1, 2):
            assert N.lib().mb200_set_option(c.handle, 3, val) == N.ERR_BAD_ARG
            assert "unknown option" in N.last_error(c.handle)
            with pytest.raises(ValueError, match="unknown option"):
                c.set_option(3, val)
        c.set_option(N.OPT_GROUP_MIN_EVENTS, 0)
        c.set_option(N.OPT_GROUP_MIN_EVENTS, 1 << 16)
        c.set_option(N.OPT_GROUP_PREFETCH, 0)
        c.set_option(N.OPT_MAX_FALLBACK_ROWS, 64)
        c.set_option(N.OPT_MAX_FALLBACK_ROWS, -1)
    finally:
        c.close()
