"""GPU recommender (csrc/recommend.cu): mb200_bank_estimate_prefs and mb200_bank_recommend against the numpy
restatement oracle/recommend.py with the GPU's own neighbourhood lists, so that estimates (bit for bit), item lists
and counts are compared on identical inputs.  Every estimation path the kernel can choose is witnessed through its
MB200_TRACE plan line."""
import math
import re

import numpy as np
import pytest

import oracle as orc
from oracle import recommend as orec

pytestmark = pytest.mark.gpu

PLAN_RE = re.compile(r"recommend plan: users=(\d+) stream=(\d+) gather=(\d+) chunks=(\d+) stages=(\d+) chunk=(\d+)")


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


@pytest.fixture(scope="module")
def ctx(mb):
    c = mb.Context(0)
    yield c
    c.close()


class Case:
    """a bank of user sketches on the GPU, the same bank in the oracle, the data model and the neighbourhoods"""

    def __init__(self, mb, ctx, seed, U, n_items, n, w, d, k, item_step=3, shift=0.0, rows=None, items=None):
        rng = np.random.Generator(np.random.PCG64(seed))
        self.rows = rng.integers(0, U, n) if rows is None else rows
        self.items = (rng.integers(0, n_items, n) * item_step + 5) if items is None else items
        self.pref = (rng.integers(1, 11, self.rows.shape[0]) * 0.5 + shift).astype(np.float32)
        self.U, self.w, self.d = U, w, d
        self.bank = mb.SketchBank(U, w, d, mb.HashFunctionBuilder(seed), frac_bits=1, ctx=ctx)
        self.bank.update(self.rows, self.items, self.pref)
        self.bank.check()
        self.a, self.b = orc.hash_params(seed, d)
        self.ob = np.zeros((U, d, w))
        orc.bank_update(self.ob, d, w, self.a, self.b, self.rows, self.items, self.pref)
        self.csr = orec.item_csr(self.rows, self.items, U)
        self.nb = self.bank.cosine_topk(k, precision="rescored")

    def recommend(self, users, how_many, include_known=False, nb=None):
        nb = self.nb if nb is None else nb
        return self.bank.recommend(*nb, *self.csr, users, how_many, include_known)

    def oracle(self, users, how_many, include_known=False, nb=None):
        nb = self.nb if nb is None else nb
        return orec.recommend(self.ob, self.a, self.b, *nb, *self.csr, users, how_many, include_known)


def _same(got, want):
    gi, gv, gc = (np.asarray(x) for x in got)
    wi, wv, wc = want
    assert (gc == wc).all(), np.nonzero(gc != wc)[0][:10]
    assert (gi == wi).all()
    assert (gv.view(np.int32) == wv.view(np.int32)).all()      # bit-identical floats, 0 in the unused slots


def _plan(capfd):
    found = PLAN_RE.findall(capfd.readouterr().err)
    assert found, "no recommend plan line in the trace output"
    users, stream, gather, chunks, stages, chunk = map(int, found[-1])
    return dict(users=users, stream=stream, gather=gather, chunks=chunks, stages=stages, chunk=chunk)


def test_recommend_streaming_matches_oracle(mb, ctx, capfd, monkeypatch):
    """W = 256: users with more than W/4 candidates stream their neighbours' rows; with and without the known
    items, how_many larger than some users' candidate counts, and users without neighbours"""
    monkeypatch.setenv("MB200_TRACE", "1")
    c = Case(mb, ctx, 21, 300, 2000, 30000, 256, 3, 12)
    users = np.arange(c.U)
    c.nb[2][::17] = 0                                         # users with no neighbours
    for include_known in (False, True):
        for how_many in (10, 700):
            capfd.readouterr()
            got = c.recommend(users, how_many, include_known)
            plan = _plan(capfd)
            assert plan["stream"] > 0 and plan["stages"] >= 2, plan
            _same(got, c.oracle(users, how_many, include_known))
    got = c.recommend(users, 700)
    assert (got[2] < 700).any() and (got[2][::17] == 0).all()


def test_recommend_several_chunks(mb, ctx, capfd, monkeypatch):
    """24 000 items, every user rates most of them: each user's candidates take several chunks, each re-streaming
    the neighbours' rows"""
    monkeypatch.setenv("MB200_TRACE", "1")
    rng = np.random.Generator(np.random.PCG64(4))
    U, I = 24, 24000
    rows = np.repeat(np.arange(U), 14000)
    items = np.concatenate([rng.choice(I, 14000, replace=False) for _ in range(U)]) * 2 + 1
    c = Case(mb, ctx, 8, U, I, 0, 256, 3, 8, rows=rows, items=items)
    users = np.arange(U)
    got = c.recommend(users, 50)
    plan = _plan(capfd)
    assert plan["stream"] == U and plan["chunks"] >= 3 * U, plan
    _same(got, c.oracle(users, 50))


def test_recommend_gather_and_large_catalogue(mb, ctx, capfd, monkeypatch):
    """few candidates per user at W = 4096 gather single counters; 150 000 items put the candidate bitmap in a
    per-CTA global slice"""
    monkeypatch.setenv("MB200_TRACE", "1")
    for n_items, seed in ((400, 3), (150000, 5)):
        c = Case(mb, ctx, seed, 200, n_items, 3000, 4096, 3, 6, item_step=1)
        users = np.arange(c.U)
        capfd.readouterr()
        got = c.recommend(users, 10)
        plan = _plan(capfd)
        assert plan["gather"] == c.U and plan["stream"] == 0, plan
        _same(got, c.oracle(users, 10))


def test_recommend_rows_too_wide_to_stage(mb, ctx, capfd, monkeypatch):
    """W = 2^16: a row (512 KiB) does not fit shared memory: every user gathers, whatever its candidate count"""
    monkeypatch.setenv("MB200_TRACE", "1")
    c = Case(mb, ctx, 9, 60, 30000, 40000, 1 << 16, 2, 10)
    users = np.arange(c.U)
    capfd.readouterr()
    got = c.recommend(users, 20)
    plan = _plan(capfd)
    assert plan["stages"] == 0 and plan["gather"] == c.U and plan["stream"] == 0, plan
    _same(got, c.oracle(users, 20))


def test_estimate_prefs_equals_do_estimate_preference(mb, ctx):
    """random (user, neighbourhood, item) triples: neighbourhoods containing the user, empty ones, items no
    neighbour has; against CosineCM.doEstimatePreference and the oracle, bit for bit"""
    from mahout_b200.cosinecm import CosineCM
    rng = np.random.Generator(np.random.PCG64(33))
    n, users = 4000, 40
    user = rng.integers(1, users + 1, n).astype(np.int64) * 10
    item = rng.integers(1, 300, n).astype(np.int64)
    pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    cm = CosineCM(user, item, pref, 128, 3, mb.HashFunctionBuilder(7), ctx=ctx)
    U, ld = cm.user_ids.shape[0], 7
    nb_idx = rng.integers(0, U, (U, ld))
    nb_cnt = rng.integers(0, ld + 1, U).astype(np.int32)
    nb_cnt[:3] = 0
    nb_sim = cm.bank.pair_cosine(np.repeat(np.arange(U), ld), nb_idx.ravel()).reshape(U, ld)
    q = 600
    qu = rng.integers(0, U, q)
    qi = rng.integers(1, 320, q)                              # items 300..319: no neighbour has them
    got = cm.bank.estimate_prefs(nb_idx, nb_sim, nb_cnt, qu, qi)
    a, b = orc.hash_params(7, 3)
    ob = np.zeros((U, 3, 128))
    orc.bank_update(ob, 3, 128, a, b, np.searchsorted(cm.user_ids, user), item, pref)
    for t in range(q):
        u = int(qu[t])
        want = orec.estimate(ob, a, b, u, nb_idx[u], nb_sim[u], nb_cnt[u], qi[t:t + 1])[0]
        ref = cm.doEstimatePreference(int(cm.user_ids[u]), cm.user_ids[nb_idx[u, :nb_cnt[u]]], int(qi[t]))
        for w in (want, ref):
            assert (math.isnan(got[t]) and math.isnan(w)) or np.float32(got[t]).view(np.int32) == np.float32(w).view(np.int32)
    assert np.isnan(got).any() and (~np.isnan(got)).any()
    cm.close()


def test_ties_lower_item_first(mb, ctx):
    """users whose neighbours rated many items alike: equal float estimates come out lower itemID first"""
    rng = np.random.Generator(np.random.PCG64(2))
    U = 30
    rows = np.repeat(np.arange(U), 40)
    items = np.concatenate([rng.choice(60, 40, replace=False) for _ in range(U)]) * 5 + 100
    c = Case(mb, ctx, 12, U, 0, 0, 4096, 3, 6, rows=rows, items=items)
    c.pref[:] = 2.0
    c.bank.clear()
    c.bank.update(c.rows, c.items, c.pref)
    c.ob[:] = 0
    orc.bank_update(c.ob, c.d, c.w, c.a, c.b, c.rows, c.items, c.pref)
    c.nb = c.bank.cosine_topk(6, precision="rescored")
    users = np.arange(U)
    got = c.recommend(users, 25)
    _same(got, c.oracle(users, 25))
    gi, gv, gc = got
    ties = 0
    for u in range(U):
        for t in range(1, gc[u]):
            if gv[u, t] == gv[u, t - 1]:
                ties += 1
                assert gi[u, t] > gi[u, t - 1]
    assert ties > 0


def test_negative_increments_and_similarities(mb, ctx):
    """rating shift: negative counters, point queries of exactly 0 (skipped), negative similarities"""
    rng = np.random.Generator(np.random.PCG64(6))
    U, n = 80, 6000
    rows = rng.integers(0, U, n)
    items = rng.integers(0, 500, n) * 7 + 3
    # +x then -x for the same (user, item): a counter of exactly 0
    rows = np.concatenate([rows, rows[:500]])
    items = np.concatenate([items, items[:500]])
    c = Case(mb, ctx, 14, U, 0, 0, 4096, 3, 10, rows=rows, items=items, shift=-2.5)
    c.pref[n:] = -c.pref[:500]
    c.bank.clear()
    c.bank.update(c.rows, c.items, c.pref)
    c.ob[:] = 0
    orc.bank_update(c.ob, c.d, c.w, c.a, c.b, c.rows, c.items, c.pref)
    users = np.arange(U)
    # neighbourhoods with negative similarities: random lists, similarities from the pair cosine
    nb_idx = rng.integers(0, U, (U, 10))
    nb_sim = c.bank.pair_cosine(np.repeat(users, 10), nb_idx.ravel()).reshape(U, 10)
    assert (nb_sim < 0).any()
    nb = (nb_idx, nb_sim, np.full(U, 10, np.int32))
    for include_known in (False, True):
        _same(c.recommend(users, 40, include_known, nb=nb), c.oracle(users, 40, include_known, nb=nb))
    _same(c.recommend(users, 40), c.oracle(users, 40))


def test_device_and_host_memory_agree(mb, ctx):
    import torch
    c = Case(mb, ctx, 23, 150, 900, 12000, 256, 3, 8)
    users = np.arange(0, c.U, 2)
    host = c.recommend(users, 15)
    dev = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (*c.nb, *c.csr, users)]
    got = c.bank.recommend(*dev[:6], dev[6], 15)
    for h, g in zip(host, got):
        assert g.is_cuda and (g.cpu().numpy() == h).all()
    qi = c.items[:300]
    eh = c.bank.estimate_prefs(*c.nb, c.rows[:300], qi)
    ed = c.bank.estimate_prefs(*dev[:3], torch.from_numpy(c.rows[:300]).cuda(), torch.from_numpy(qi).cuda())
    assert (ed.cpu().numpy().view(np.int32) == eh.view(np.int32)).all()


def test_recommender_single_user_equals_batch(mb, ctx):
    from mahout_b200.cosinecm import CosineCM
    from mahout_b200.recommender import GenericUserBasedRecommender
    rng = np.random.Generator(np.random.PCG64(8))
    n = 20000
    user = rng.integers(1, 301, n).astype(np.int64) * 3
    item = rng.integers(1, 1500, n).astype(np.int64) * 11
    pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    cm = CosineCM(user, item, pref, 256, 3, 42, ctx=ctx)
    rec = GenericUserBasedRecommender(cm, 15)
    ids, items, vals, cnt = rec.recommend_all(8)
    assert (cnt > 0).sum() > 0.9 * ids.shape[0]
    for r in (0, 5, 77, ids.shape[0] - 1):
        one = rec.recommend(int(ids[r]), 8)
        assert [i for i, _ in one] == items[r, :cnt[r]].tolist()
        assert [v for _, v in one] == vals[r, :cnt[r]].tolist()
    # the neighbourhood is the re-scored top-15, and estimate_preferences equals doEstimatePreference over it
    nbh = rec.getUserNeighborhood(int(ids[5]))
    assert 0 < len(nbh) <= 15 and int(ids[5]) not in nbh.tolist()
    e = rec.estimate_preferences(np.full(5, ids[5]), items[5, :5].clip(min=11))
    for t in range(5):
        ref = cm.doEstimatePreference(int(ids[5]), nbh, int(items[5, :5].clip(min=11)[t]))
        assert (math.isnan(e[t]) and math.isnan(ref)) or np.float32(e[t]) == np.float32(ref)
    with pytest.raises(KeyError):
        rec.recommend(2, 5)
    cm.close()


def test_bad_arguments(mb, ctx):
    c = Case(mb, ctx, 31, 50, 200, 2000, 256, 3, 5)
    users = np.arange(c.U)
    for how_many in (0, 1025):
        with pytest.raises(ValueError, match="how_many"):
            c.recommend(users, how_many)
    with pytest.raises(ValueError, match="out of range"):
        c.recommend(np.array([0, c.U]), 5)                                     # user row
    idx, sim, cnt = (x.copy() for x in c.nb)
    idx[3, 0], cnt[3] = c.U + 7, max(cnt[3], 1)
    with pytest.raises(ValueError, match="out of range"):
        c.recommend(users, 5, nb=(idx, sim, cnt))                             # neighbour index
    with pytest.raises(ValueError, match="out of range"):
        c.bank.estimate_prefs(idx, sim, cnt, np.array([3]), np.array([5]))
    ptr, col, ids = c.csr
    col = col.copy()
    col[4] = ids.shape[0]
    with pytest.raises(ValueError, match="out of range"):
        c.bank.recommend(*c.nb, ptr, col, ids, users, 5)                       # item_col
    with pytest.raises(ValueError):
        c.bank.recommend(*c.nb, ptr[:-1], c.csr[1], ids, users, 5)            # item_ptr of the wrong length
    with pytest.raises(ValueError):
        c.bank.recommend(*c.nb, ptr, c.csr[1][:-1], ids, users, 5)            # nnz != item_ptr[E]
    with pytest.raises(ValueError):
        c.bank.estimate_prefs(*c.nb, np.array([1, 2]), np.array([5]))          # user / item lengths
    # the context still works after the rejected calls
    _same(c.recommend(users, 5), c.oracle(users, 5))
