"""GPU item-based recommender (csrc/recommend.cu, k_itembased) against the numpy restatement oracle/itembased.py on
the GPU's own item top-k lists, for both measures: items, counts and float bits must be equal.  Every accumulator
path is witnessed through the MB200_TRACE plan line, so a change to the selection fails here instead of dropping
coverage."""
import re

import numpy as np
import pytest

from oracle import itembased as oib

pytestmark = pytest.mark.gpu

PLAN_RE = re.compile(r"itembased plan: users=(\d+) smem=(\d+) dense=(\d+) entries=(\d+) entries_max=(\d+) "
                     r"pruned=(\d+) candidates_max=(\d+)")


@pytest.fixture(scope="module")
def ctx():
    import mahout_b200 as mb
    c = mb.Context(0)
    yield c
    c.close()


def _plan(capfd):
    found = PLAN_RE.findall(capfd.readouterr().err)
    assert found, "no itembased plan line in the trace output"
    keys = ("users", "smem", "dense", "entries", "entries_max", "pruned", "candidates_max")
    return dict(zip(keys, map(int, found[-1])))


class Case:
    """de-duplicated prefs of a random population, the GPU's top-k lists of one measure, the user CSR"""

    def __init__(self, ctx, seed, n_items=400, n_users=300, max_n=40, k=20, shift=0.0, exact=False,
                 boolean_data=False, equal_prefs=0):
        from mahout_b200 import similarity as sim
        rng = np.random.Generator(np.random.PCG64(seed))
        rows, users, prefs = [], [], []
        for u in range(n_users):
            n = int(rng.integers(1, max_n + 1))
            r = rng.choice(n_items, n, replace=False)
            if boolean_data:
                p = np.ones(n, np.float32)
            elif u < equal_prefs:
                p = np.full(n, 3.0, np.float32)                           # equal prefs: tied predictions
            elif u % 23 == 5:
                p = np.zeros(n, np.float32)                               # no considered pref
            else:
                p = (rng.integers(0, 11, n) * 0.5 + shift).astype(np.float32)   # ties at T, zeros
            rows.append(r)
            users.append(np.full(n, 10 ** 6 + 7 * u, np.int64))         # row u = user u
            prefs.append(p)
        self.row, self.user, self.pref = np.concatenate(rows), np.concatenate(users), np.concatenate(prefs)
        # the lists come from the pref-weighted vectors (1.0 for boolean data); zero prefs do not enter the bank
        nzp = self.pref != 0
        r, u, p = self.row[nzp], self.user[nzp], self.pref[nzp]
        if exact:
            self.lists = sim.exact_item_similarity(r, u, p, n_items, k=k, ctx=ctx)
        else:
            self.lists = sim.item_similarity(r, u, p, n_items, k=k, width=512, depth=3, ctx=ctx)
        self.item_ids = rng.permutation(n_items).astype(np.int64) * 13 + 2        # not ascending in row order
        self.uids, self.ptr, self.prow, self.pval = oib.user_csr(self.row, self.user, self.pref)
        self.ctx = ctx

    def run(self, users=None, how_many=10, max_prefs=10, boolean_data=False, allowed_ids=None, device=False):
        from mahout_b200 import itembased as ib
        users = np.arange(self.uids.shape[0]) if users is None else np.asarray(users)
        mask = None if allowed_ids is None else ib.allowed_mask(self.item_ids, allowed_ids)
        uv = ib.UserVectors(self.uids, self.ptr, self.prow, self.pval)
        lists, item_ids = self.lists, self.item_ids
        if device:
            import torch
            t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()   # noqa: E731
            lists = tuple(t(x) for x in lists)
            uv = ib.UserVectors(t(self.uids), t(self.ptr), t(self.prow), t(self.pval))
            users, item_ids = t(users), t(item_ids)
            mask = None if mask is None else t(mask.view(np.int32))
        got = ib.recommend(lists, uv, item_ids, users, how_many, max_prefs, boolean_data, mask, ctx=self.ctx)
        return tuple(x.cpu().numpy() if hasattr(x, "cpu") else x for x in got)

    def oracle(self, users=None, how_many=10, max_prefs=10, boolean_data=False, allowed_ids=None):
        users = np.arange(self.uids.shape[0]) if users is None else np.asarray(users)
        allowed = None if allowed_ids is None else np.isin(self.item_ids, list(allowed_ids))
        return oib.recommend(*self.lists, self.ptr, self.prow, self.pval, self.item_ids, users, how_many, max_prefs,
                             boolean_data, allowed)

    def check(self, **kw):
        got, want = self.run(**kw), self.oracle(**kw)
        _same(got, want)
        return got


def _same(got, want):
    gi, gv, gc = got
    wi, wv, wc = want
    assert (gc == wc).all(), np.nonzero(gc != wc)[0][:10]
    assert (gi == wi).all()
    assert (gv.view(np.int32) == wv.view(np.int32)).all()      # bit-identical floats, 0 in the unused slots


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("shift", [0.0, -2.5])
def test_table_path_matches_oracle(ctx, capfd, monkeypatch, exact, shift):
    """k = 20, P = 10: every user's entries fit the shared-memory table; users over, at and under P with ties at T,
    zero prefs, users with no considered pref, rating shift (predictions <= 0 dropped)"""
    monkeypatch.setenv("MB200_TRACE", "1")
    c = Case(ctx, 3 + int(exact), shift=shift, exact=exact)
    capfd.readouterr()
    got = c.check()
    plan = _plan(capfd)
    assert plan["smem"] == c.uids.shape[0] and plan["dense"] == 0 and plan["pruned"] > 0, plan
    assert (got[2] > 0).sum() > c.uids.shape[0] // 2
    assert (got[2][5::23] == 0).all()                      # the users whose prefs are all zero


@pytest.mark.parametrize("exact", [False, True])
def test_dense_path_matches_oracle(ctx, capfd, monkeypatch, exact):
    """k = 100 and P unlimited: users with many prefs exceed the table and take dense slices; the others stay in
    the table in the same launch"""
    monkeypatch.setenv("MB200_TRACE", "1")
    c = Case(ctx, 8 + int(exact), n_items=3000, n_users=400, max_n=200, k=100, exact=exact)
    for max_prefs in (2 ** 31 - 1, 50):
        capfd.readouterr()
        c.check(max_prefs=max_prefs, how_many=50)
        plan = _plan(capfd)
        assert plan["dense"] > 0 and plan["smem"] > 0 and plan["entries_max"] > 1024, plan


@pytest.mark.parametrize("exact", [False, True])
def test_boolean_data(ctx, capfd, monkeypatch, exact):
    monkeypatch.setenv("MB200_TRACE", "1")
    c = Case(ctx, 12, boolean_data=True, exact=exact)
    capfd.readouterr()
    got = c.check(boolean_data=True, how_many=20)
    plan = _plan(capfd)
    assert plan["pruned"] > 0, plan                         # users over P ...
    unlimited = c.run(boolean_data=True, how_many=20, max_prefs=2 ** 31 - 1)
    for g, u in zip(got, unlimited):                        # ... keep every pref: all tie at T
        assert (g == u).all()
    assert (got[2] > 0).any()


def test_ties_lower_item_id_first(ctx):
    """users whose prefs are all equal: many equal predictions; itemIDs are not ascending in row order"""
    c = Case(ctx, 14, equal_prefs=150, exact=True)
    gi, gv, gc = c.check(how_many=60)
    ties = 0
    for u in range(c.uids.shape[0]):
        for t in range(1, gc[u]):
            if gv[u, t] == gv[u, t - 1]:
                ties += 1
                assert gi[u, t] > gi[u, t - 1]
    assert ties > 0


def test_allowed_items_user_subset_and_how_many(ctx):
    c = Case(ctx, 15)
    U = c.uids.shape[0]
    allowed = set(c.item_ids[::4].tolist())
    got = c.check(allowed_ids=allowed, how_many=15)
    assert all(i in allowed for i in got[0][got[0] >= 0].tolist()) and (got[2] > 0).any()
    sub = np.array([U - 1, 0, 17, 17, 100])
    c.check(users=sub)
    one = c.check(how_many=1)
    assert (one[2] <= 1).all() and (one[2] == 1).any()
    full = c.check(how_many=1024, max_prefs=40)
    assert (full[2] < 1024).all() and full[2].max() > 60     # more slots than candidates


def test_host_and_device_memory_agree(ctx):
    c = Case(ctx, 16)
    allowed = set(c.item_ids[::3].tolist())
    host = c.run(how_many=12, allowed_ids=allowed)
    dev = c.run(how_many=12, allowed_ids=allowed, device=True)
    for h, d in zip(host, dev):
        assert (np.asarray(h) == np.asarray(d)).all()
    _same(host, c.oracle(how_many=12, allowed_ids=allowed))


def test_bad_arguments(ctx):
    from mahout_b200 import itembased as ib
    c = Case(ctx, 17, n_users=60)
    U = c.uids.shape[0]
    users = np.arange(U)
    idx, sim, cnt = c.lists

    def call(lists=None, ptr=None, prow=None, users_=None, **kw):
        uv = ib.UserVectors(c.uids, c.ptr if ptr is None else ptr, c.prow if prow is None else prow, c.pval)
        return ib.recommend(c.lists if lists is None else lists, uv, c.item_ids, users if users_ is None else users_,
                            ctx=ctx, **kw)

    for kw in ({"how_many": 0}, {"how_many": 1025}, {"max_prefs_per_user": 0}):
        with pytest.raises(ValueError):
            call(**kw)
    with pytest.raises(ValueError, match="out of range"):
        call(users_=np.array([0, U]))                                          # user row
    with pytest.raises(ValueError, match="out of range"):
        call(users_=np.array([-1]))
    ptr = c.ptr.copy()
    ptr[5] = ptr[6] + 1                                                        # user_ptr not monotone
    with pytest.raises(ValueError, match="out of range"):
        call(ptr=ptr)
    ptr = c.ptr.copy()
    ptr[-1] = c.prow.shape[0] + 5                                              # beyond nnz
    with pytest.raises(ValueError, match="out of range"):
        call(ptr=ptr)
    u = int(np.argmax(np.diff(c.ptr)))
    lo = int(c.ptr[u])
    for bad_row in (idx.shape[0], -3):
        prow = c.prow.copy()
        prow[lo] = bad_row                                                     # pref_row out of range
        with pytest.raises(ValueError, match="out of range"):
            call(prow=prow)
    prow = c.prow.copy()
    prow[lo], prow[lo + 1] = prow[lo + 1], prow[lo]                            # not ascending
    with pytest.raises(ValueError, match="ascending"):
        call(prow=prow)
    j = int(c.prow[lo + int(np.argmax(c.pval[lo:int(c.ptr[u + 1])] != 0))])   # a list the user considers
    bcnt = cnt.copy()
    bcnt[j] = idx.shape[1] + 1                                                 # count beyond the lists' width
    with pytest.raises(ValueError, match="out of range"):
        call(lists=(idx, sim, bcnt), max_prefs_per_user=10 ** 6)
    bidx = idx.copy()
    bidx[j, 0], bcnt = idx.shape[0] + 9, cnt.copy()
    bcnt[j] = max(bcnt[j], 1)
    with pytest.raises(ValueError, match="out of range"):
        call(lists=(bidx, sim, bcnt), max_prefs_per_user=10 ** 6)            # list entry
    _same(c.run(), c.oracle())                                                 # the context still works


def _write_input(path, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    n = 6000
    u = rng.integers(1, 301, n) * 3
    i = rng.integers(1, 400, n) * 11
    p = rng.integers(1, 11, n) * 0.5
    path.write_text("".join(f"{a},{b},{c}\n" for a, b, c in zip(u, i, p)))


@pytest.mark.parametrize("measure", ["SIMILARITY_COSINE", "SIMILARITY_SKETCH_COSINE"])
def test_job_output_equals_oracle_formatting(ctx, tmp_path, measure):
    """the job's file, byte for byte, against the oracle run on the lists and user vectors the same calls produce"""
    from mahout_b200 import ingest, similarity as sim
    from mahout_b200.recommenditembased import RecommenderJob, format_line
    inp, out = tmp_path / "in.csv", tmp_path / "out.txt"
    _write_input(inp, 21)
    users_file, items_file = tmp_path / "users.txt", tmp_path / "items.txt"
    users_file.write_text("".join(f"{3 * u}\n" for u in range(1, 301, 2)))
    items_file.write_text("".join(f"{11 * i}\n" for i in range(1, 400, 3)))
    for extra, how_many in (([], 10), (["--numRecommendations", "25", "--maxPrefsPerUser", "5",
                                        "--usersFile", str(users_file), "--itemsFile", str(items_file)], 25)):
        assert RecommenderJob().run(["--input", str(inp), "--output", str(out), "-s", measure, "-m", "30",
                                     "--sketchWidth", "1024", "--sketchDepth", "3"] + extra) == 0
        ev = ingest.Events.parse_file(str(inp))
        prep = ev.prepare(1)
        ev.close()
        if measure == "SIMILARITY_COSINE":
            lists = sim.exact_item_similarity(prep.row, prep.user, prep.pref, prep.num_items, k=30,
                                              ucol=prep.ucol, num_users=prep.num_users)
        else:
            lists = sim.item_similarity(prep.row, prep.user, prep.pref, prep.num_items, k=30, width=1024, depth=3)
        uids, ptr, prow, pval = oib.user_csr(*(x.cpu().numpy() for x in (prep.row, prep.user, prep.pref)))
        rows = np.arange(uids.shape[0])
        allowed = None
        if extra:
            rows = rows[np.isin(uids, np.arange(3, 901, 6))]
            allowed = np.isin(prep.item_id, np.arange(11, 4400, 33))
        wi, wv, wc = oib.recommend(*lists, ptr, prow, pval, prep.item_id, rows, how_many, 5 if extra else 10,
                                   False, allowed)
        want = "".join(format_line(uids[r], wi[t, :wc[t]], wv[t, :wc[t]]) for t, r in enumerate(rows) if wc[t])
        prep.close()
        assert want and out.read_text() == want


def test_job_hand_checked_answers(tmp_path):
    from mahout_b200.recommenditembased import RecommenderJob
    cases = [("1,1,5\n1,2,3\n2,1,4\n2,2,2\n2,3,5\n3,2,1\n3,3,4\n4,1,2\n4,3,1\n", [],
              "1\t[3:3.9341865]\n3\t[1:2.0673192]\n4\t[2:1.6134744]\n"),
             ("2,1,1\n1,2,1\n3,4,1\n1,3,2\n2,3,1\n", ["--booleanData", "true"],
              "1\t[1:0.70710677]\n2\t[2:0.70710677]\n"),
             ("2,1,1\n1,2,1\n3,4,1\n1,3,2\n2,3,1\n", [], "")]
    for text, extra, want in cases:
        inp, out = tmp_path / "in.csv", tmp_path / "out.txt"
        inp.write_text(text)
        assert RecommenderJob().run(["-i", str(inp), "-o", str(out), "-s", "SIMILARITY_COSINE"] + extra) == 0
        assert out.read_text() == want
