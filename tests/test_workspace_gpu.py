"""The context's named workspaces, host-argument staging and status words (csrc/runtime.cu): host-memory calls
interleaved on one context return the bytes each returns alone on a fresh context, also after
mb200_release_workspace, and mb200_get_stats counts the buffers those calls keep."""
import ctypes as C

import numpy as np
import pytest

from oracle import itembased as oib
from oracle import recommend as orec

pytestmark = pytest.mark.gpu

SEED = 31
U, N_ITEMS, W, D = 300, 2000, 256, 3


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


class Data:
    """host inputs of every call; the neighbourhood and item lists come from one set-up context, so each call under
    test sees the same arguments on every context"""

    def __init__(self, mb):
        from mahout_b200 import similarity as sim
        rng = np.random.Generator(np.random.PCG64(SEED))
        rows = rng.integers(0, U, 30000)
        items = rng.integers(0, N_ITEMS, rows.shape[0]) * 3 + 5
        self.ptr, self.col, self.item_ids = orec.item_csr(rows, items, U)
        self.rows = np.repeat(np.arange(U), np.diff(self.ptr))
        self.items = self.item_ids[self.col]
        self.pref = (rng.integers(1, 11, self.rows.shape[0]) * 0.5).astype(np.float32)
        self.width = rng.choice([31, 64, 100, 257], U).astype(np.int32)
        self.depth = rng.choice([2, 3, 5], U).astype(np.int32)
        self.users = rng.permutation(U)[:200]
        self.q_user = rng.integers(0, U, 5000)
        self.q_item = self.item_ids[rng.integers(0, self.item_ids.shape[0], 5000)]
        self.pair = rng.integers(0, U, (2, 3000))
        # mb200_bank_update_grouped: 64 entities, events grouped by entity
        self.g_ptr = np.concatenate([[0], np.cumsum(rng.integers(0, 3000, 64))]).astype(np.int64)
        n = int(self.g_ptr[-1])
        self.g_key = rng.integers(0, 10 ** 6, n)
        self.g_inc = (rng.integers(-4, 9, n) * 0.5).astype(np.float32)
        # a single-sketch update large enough for the key table once its threshold is lowered
        self.kt_key = np.minimum(rng.zipf(1.1, 300001), 10 ** 7).astype(np.int64)
        self.kt_inc = (rng.integers(-4, 9, self.kt_key.shape[0]) * 0.5).astype(np.float32)
        self.route_row = rng.integers(0, 1000, 100003)
        ctx = mb.Context(0)
        bank, sized = self.banks(mb, ctx)
        self.nb = bank.cosine_topk(12, precision="rescored")
        self.snb = sized.neighborhood(self.users, 20)
        for h in (bank, sized):
            h.close()
        # two item-based populations of different num_items, both with users on the dense slices
        self.ib = []
        for n_items in (3000, 2000):
            r, u, p = [], [], []
            for x in range(400):
                k = int(rng.integers(1, 201))
                r.append(rng.choice(n_items, k, replace=False))
                u.append(np.full(k, 10 ** 6 + 7 * x, np.int64))
                p.append((rng.integers(1, 11, k) * 0.5).astype(np.float32))
            r, u, p = np.concatenate(r), np.concatenate(u), np.concatenate(p)
            lists = sim.exact_item_similarity(r, u, p, n_items, k=100, ctx=ctx)
            item_ids = rng.permutation(n_items).astype(np.int64) * 13 + 2
            self.ib.append((tuple(np.asarray(x) for x in lists), oib.user_csr(r, u, p), item_ids))
        ctx.close()

    def banks(self, mb, ctx):
        bank = mb.SketchBank(U, W, D, mb.HashFunctionBuilder(SEED), frac_bits=1, ctx=ctx)
        bank.update(self.rows, self.items, self.pref)
        bank.check()
        sized = mb.SizedBank(self.width, self.depth, mb.HashFunctionBuilder(SEED), self.ptr, self.items, self.pref,
                             ctx=ctx)
        return bank, sized


def _itembased(x, ctx, which):
    from mahout_b200 import itembased as ib
    lists, (uids, ptr, prow, pval), item_ids = x.ib[which]
    got = ib.recommend(lists, ib.UserVectors(uids, ptr, prow, pval), item_ids, None, 50, 2 ** 31 - 1, ctx=ctx)
    assert ib.itembased_plan(ctx)["dense_users"] > 0
    return got


def _update_grouped(mb, x, ctx):
    bank = mb.SketchBank(64, 512, 4, 42, 1, ctx)
    bank.update_grouped(x.g_ptr, x.g_key, x.g_inc)
    return bank.read()


def _keytable(mb, x, ctx):
    bank = mb.SketchBank(1, 1 << 16, 4, 42, 1, ctx)
    bank.update(None, x.kt_key, x.kt_inc)
    return bank.read()


def _route_count(x, ctx):
    import torch
    from mahout_b200 import _native as N
    row = torch.from_numpy(x.route_row).cuda(ctx.device)
    counts = np.zeros(8, np.int64)
    N.check(N.lib().mb200_route_count(ctx.handle, C.c_void_p(row.data_ptr()), row.numel(), 8,
                                      counts.ctypes.data_as(C.c_void_p)), ctx.handle)
    return counts


CALLS = {
    "bank_recommend": lambda mb, x, c, b, s: b.recommend(*x.nb, x.ptr, x.col, x.item_ids, x.users, 10),
    "bank_estimate_prefs": lambda mb, x, c, b, s: b.estimate_prefs(*x.nb, x.q_user, x.q_item),
    "sized_neighborhood": lambda mb, x, c, b, s: s.neighborhood(x.users, 20),
    "sized_recommend": lambda mb, x, c, b, s: s.recommend(*x.snb, x.ptr, x.col, x.item_ids, x.users, 10),
    "sized_pair_cosine": lambda mb, x, c, b, s: s.pair_cosine(x.pair[0], x.pair[1]),
    "itembased_3000": lambda mb, x, c, b, s: _itembased(x, c, 0),
    "itembased_2000": lambda mb, x, c, b, s: _itembased(x, c, 1),
    "bank_query": lambda mb, x, c, b, s: b.query(x.q_user, x.q_item),
    "bank_read": lambda mb, x, c, b, s: b.read(),
    "bank_update_grouped": lambda mb, x, c, b, s: _update_grouped(mb, x, c),
    "route_count": lambda mb, x, c, b, s: _route_count(x, c),
    "keytable": lambda mb, x, c, b, s: _keytable(mb, x, c),
}

SEQUENCE = ["bank_recommend", "itembased_3000", "sized_neighborhood", "bank_query", "keytable", "bank_update_grouped",
            "sized_recommend", "itembased_2000", "bank_estimate_prefs", "route_count", "sized_pair_cosine",
            "itembased_3000", "bank_read", "keytable", "bank_recommend", "sized_neighborhood"]


def _bytes(out):
    if isinstance(out, tuple):
        return tuple(_bytes(o) for o in out)
    return np.ascontiguousarray(np.asarray(out)).tobytes()


def test_interleaved_calls_equal_calls_alone(mb, monkeypatch):
    """each call alone on a fresh context, then all of them interleaved on one context, then again after
    mb200_release_workspace (the key table and the item-based dense slices must come back zeroed)"""
    from mahout_b200 import _native as N
    monkeypatch.setenv("MB200_K1_KEYTABLE_MIN_EVENTS", "0")
    x = Data(mb)
    alone = {}
    for name, call in CALLS.items():
        ctx = mb.Context(0)
        b, s = x.banks(mb, ctx)
        alone[name] = _bytes(call(mb, x, ctx, b, s))
        for h in (b, s, ctx):
            h.close()
    ctx = mb.Context(0)
    b, s = x.banks(mb, ctx)
    for rnd in range(2):
        for name in SEQUENCE:
            assert _bytes(CALLS[name](mb, x, ctx, b, s)) == alone[name], (rnd, name)
        N.check(N.lib().mb200_release_workspace(ctx.handle), ctx.handle)
    for h in (b, s, ctx):
        h.close()


def test_stats_count_named_workspaces_and_staging(mb):
    """a host-memory mb200_bank_recommend on a fresh context (bank built from device memory) keeps named workspaces
    and at least its staged arguments' bytes; mb200_release_workspace returns every workspace"""
    import torch
    from mahout_b200 import _native as N
    rng = np.random.Generator(np.random.PCG64(SEED + 1))
    rows = rng.integers(0, U, 20000)
    items = rng.integers(0, N_ITEMS, rows.shape[0]) * 3 + 5
    ptr, col, item_ids = orec.item_csr(rows, items, U)
    rows = np.repeat(np.arange(U), np.diff(ptr))
    pref = (rng.integers(1, 11, rows.shape[0]) * 0.5).astype(np.float32)
    ctx = mb.Context(0)
    bank = mb.SketchBank(U, W, D, mb.HashFunctionBuilder(SEED), frac_bits=1, ctx=ctx)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda(ctx.device)   # noqa: E731
    bank.update(cuda(rows), cuda(item_ids[col]), cuda(pref))
    nb = bank.cosine_topk(12, precision="rescored")
    N.check(N.lib().mb200_release_workspace(ctx.handle), ctx.handle)    # what cosine_topk kept
    users, how_many = np.arange(U), 10
    st0 = ctx.stats()
    assert st0["workspace_bytes"] == 0 and st0["staging_bytes"] == 0, st0
    got = bank.recommend(*nb, ptr, col, item_ids, users, how_many)
    staged = sum(a.nbytes for a in (*nb, ptr, col, item_ids, users, *got))
    st = ctx.stats()
    assert st["workspace_bytes"] > 0 and st["staging_bytes"] >= staged, (st, staged)
    N.check(N.lib().mb200_release_workspace(ctx.handle), ctx.handle)
    assert ctx.stats()["workspace_bytes"] == 0
    bank.close()
    ctx.close()
