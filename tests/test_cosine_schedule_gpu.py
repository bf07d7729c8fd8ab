"""K3 (k_cosine) and the K5 merge (k_merge) at the schedules they run at scale.

At the few thousand items of test_cosine_gpu.py the host planner (job_push_locked) always makes a small uniform
launch: no persistent CTA reaches a second work item, a candidate list never fills, there is no tail plan.  Here
the banks are large enough (and MB200_COS_CHUNKS / MB200_COS_MAIN push the planner) for more work items than SMs,
tail plans (`main < num_m`), chunks of 4+ tiles (a list passes LCAP - HALF entries and takes the forced threshold
raise), many lists per row in k_merge, and the strided item form of the fused pull-gather.  Every case reads the
plan the library chose from its MB200_TRACE line and asserts the property it was written for, so that a change of
the cost model fails loudly instead of silently dropping the coverage.

Bars:
  * TENSOR: idx, sim and cnt equal, bit for bit, the top-k of the kernel's own dense values (want_dense) under
    (value desc, index asc) -- candidates are the columns c != r with a value that is not NaN, > 0 and >= threshold.
    This tests selection and merge independently of the MMA's precision.
  * RESCORED: idx, sim and cnt bit-equal to the oracle.
  * CERTIFIED: the oracle's top-k sets, values within 1e-3 relative of the oracle's.
"""
import ctypes as C
import re

import numpy as np
import pytest

import oracle as orc
from oracle import fast

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3
W = 256
PLAN_RE = re.compile(r"\[mb200 trace\] plan: num_m=(\d+) T=(\d+) main=(\d+) blocks x (\d+) chunks, tail x (\d+) chunks")
LANES = (0, 31, 32, 63, 64, 95, 96, 127)   # first and last lane of every TMEM lane quarter

# (name, planner overrides, what the plan must reach): "waves" = more work items than SMs, "tail" = a tail plan
# (main < num_m), "long" = a column chunk of 4+ tiles
PLANNER = ("planner", {}, ("waves", "tail", "long"))
CHUNKS1 = ("chunks=1", {"MB200_COS_CHUNKS": "1"}, ("long",))
CHUNKS3 = ("chunks=3", {"MB200_COS_CHUNKS": "3"}, ("waves", "long"))
CHUNKS16 = ("chunks=16", {"MB200_COS_CHUNKS": "16"}, ("waves",))
MAIN2 = ("main=2", {"MB200_COS_MAIN": "2"}, ("waves", "tail", "long"))
MAIN4 = ("main=4", {"MB200_COS_MAIN": "4"}, ("waves", "tail", "long"))


@pytest.fixture(scope="module")
def mb():
    import mahout_b200
    return mahout_b200


@pytest.fixture(scope="module")
def ctx(mb):
    c = mb.Context(0)
    yield c
    c.close()


class Bank:
    """a device bank with its oracle counters (preference units) and quanta (frac_bits = 1)"""

    def __init__(self, mb, ctx, E, d, item, user, pref):
        self.E, self.d = E, d
        self.sk = mb.SketchBank(E, W, d, 42, 1, ctx)
        self.sk.update(item, user, pref)
        a, b = orc.hash_params(42, d)
        self.ref = np.zeros((E, d, W))
        orc.bank_update(self.ref, d, W, a, b, item, user, pref)
        assert self.sk.read().tobytes() == self.ref.tobytes(), "counters differ from the oracle"
        self.q = np.rint(self.ref * 2).astype(np.int64)
        self.rows, self.valid = self.sk.normalize()

    def oracle(self, rows, k):
        return fast.bank_rows_topk(self.q, rows, k, threads=orc.max_threads())


def _events(E, seed, users, empty):
    """_make_bank's shape (test_cosine_gpu.py): Zipf items spread over the index range, half-unit prefs, 50 events
    per item on average; `empty` items get none"""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = 50 * E
    item = (np.minimum(rng.zipf(1.2, n), E) - 1).astype(np.int64)
    item = (item * 7919) % E
    item = item[~np.isin(item, np.array(empty))]
    user = rng.integers(1, users + 1, item.shape[0]).astype(np.int64)
    pref = (rng.integers(1, 11, item.shape[0]) * 0.5).astype(np.float32)
    return item, user, pref


@pytest.fixture(scope="module")
def bank_a(mb, ctx):
    """12 000 items, d = 2: 94 row blocks (the last one partial, with an empty item), 47 column tiles"""
    E = 12000
    b = Bank(mb, ctx, E, 2, *_events(E, 1, 3000, empty=(5, 4097, 11990)))
    yield b
    b.sk.close()


@pytest.fixture(scope="module")
def bank_b(mb, ctx):
    """20 000 items, d = 1: 157 row blocks, more than one full wave of 148 SMs"""
    E = 20000
    b = Bank(mb, ctx, E, 1, *_events(E, 2, 3000, empty=(11, 19990)))
    yield b
    b.sk.close()


@pytest.fixture(scope="module")
def bank_ties(mb, ctx):
    """boolean data (every preference 1.0), 2 events per item from 40 users: large groups of identical sketches
    (and of equal similarities) spread over every chunk, item and wave; the last 5 items stay empty"""
    E = 12000
    rng = np.random.Generator(np.random.PCG64(12))
    item = np.repeat(np.arange(E - 5), 2).astype(np.int64)
    user = rng.integers(1, 41, item.shape[0]).astype(np.int64)
    b = Bank(mb, ctx, E, 2, item, user, np.ones(item.shape[0], np.float32))
    yield b
    b.sk.close()


@pytest.fixture(scope="module")
def bank_mixed(mb, ctx):
    """negative increments (test_mixed_sign_counters_exact_sets) at bank A's shape"""
    E = 12000
    rng = np.random.Generator(np.random.PCG64(99))
    n = 50 * E
    item = rng.integers(0, E, n).astype(np.int64)
    user = rng.integers(1, 2000, n).astype(np.int64)
    pref = (rng.integers(-10, 11, n) * 0.5).astype(np.float32)
    b = Bank(mb, ctx, E, 2, item, user, pref)
    assert (b.ref < 0).any()
    yield b
    b.sk.close()


def _sample_rows(E):
    """lanes 0, 31, 32, 63, 64, 95, 96, 127 of every full 128-row block, every row of the last partial one"""
    full = E // 128 * 128
    return np.array([m + l for m in range(0, full, 128) for l in LANES] + list(range(full, E)), np.int64)


@pytest.fixture(scope="module")
def oracle_a(bank_a):
    """all rows of bank A at k = 300; the top-100 is its prefix"""
    return bank_a.oracle(np.arange(bank_a.E), 300)


@pytest.fixture(scope="module")
def oracle_b(bank_b):
    rows = _sample_rows(bank_b.E)
    return rows, bank_b.oracle(rows, 100)


@pytest.fixture(scope="module")
def oracle_ties(bank_ties):
    return bank_ties.oracle(np.arange(bank_ties.E), 50)


def _prefix(o, k):
    idx, sim, cnt = o
    return np.ascontiguousarray(idx[:, :k]), np.ascontiguousarray(sim[:, :k]), np.minimum(cnt, k)


def _dense(ctx, bank, block_n=0):
    """the kernel's own tensor values [E, E] (float32, device; NaN = no comparable depth row), written by whole-row
    sweeps: a schedule that skips tiles cannot hide the same tiles from the reference"""
    from mahout_b200.sketch import cosine_topk_blocks
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("MB200_COS_CHUNKS", "1")
        mp.delenv("MB200_COS_MAIN", raising=False)
        *_, dense = cosine_topk_blocks(ctx, bank.rows, bank.valid, bank.rows.unsqueeze(0), bank.valid.unsqueeze(0),
                                       bank.d, W, 8, b_id=(1, bank.E), precision="tensor", block_n=block_n,
                                       want_dense=True)
    return dense[:, :bank.E]


@pytest.fixture(scope="module")
def dense_a(ctx, bank_a):
    return _dense(ctx, bank_a)


@pytest.fixture(scope="module")
def dense_ties(ctx, bank_ties):
    return _dense(ctx, bank_ties)


def _tensor_ref(dense, k, threshold=None, exclude_self=True, block=1024):
    """top-k of every row of `dense` under (value desc, index asc) over the admissible columns, in the output
    convention of k_merge (unused slots: idx -1, sim 0).  Synchronises on return: the library works on its own
    stream, and memory the caching allocator hands it must not still be written by the sort's temporaries."""
    import torch
    E = dense.shape[0]
    idx, sim, cnt = [], [], []
    for r0 in range(0, E, block):
        r1 = min(E, r0 + block)
        v = dense[r0:r1]
        keep = v > 0                                       # (NaN compares false)
        if threshold is not None:
            keep &= v.double() >= threshold
        if exclude_self:
            r = torch.arange(r1 - r0, device=v.device)
            keep[r, r + r0] = False
        v = torch.where(keep, v, torch.full_like(v, float("-inf")))
        val, order = torch.sort(v, dim=1, descending=True, stable=True)     # stable: equal values by index asc
        val, order = val[:, :k], order[:, :k]
        ok = torch.isfinite(val)
        idx.append(torch.where(ok, order, -1))
        sim.append(torch.where(ok, val.double(), 0.0))
        cnt.append(ok.sum(dim=1, dtype=torch.int32))
    out = torch.cat(idx), torch.cat(sim), torch.cat(cnt)
    torch.cuda.synchronize()
    return out


def _use_plan(monkeypatch, env):
    monkeypatch.setenv("MB200_TRACE", "1")
    for name in ("MB200_COS_CHUNKS", "MB200_COS_MAIN"):
        monkeypatch.delenv(name, raising=False)
    for name, value in env.items():
        monkeypatch.setenv(name, value)


def _witness(capfd, ctx, case, wants, label=""):
    """the plan of the first K3 launch since the last call (its MB200_TRACE line), checked against what the case
    claims to reach; returns the plan line for assertion messages"""
    err = capfd.readouterr().err
    found = PLAN_RE.findall(err)
    assert found, f"{case}: no plan line in the trace output"
    num_m, T, main, s_main, s_tail = map(int, found[0])
    items, longest = 0, 0
    for blocks, S in ((main, s_main), (num_m - main, s_tail)):    # emit(): ct = ceil(T/S), Sr = ceil(T/ct)
        if blocks > 0:
            ct = -(-T // S)
            items += blocks * -(-T // ct)
            longest = max(longest, ct)
    sms = ctx.stats()["num_sms"]
    plan = (f"num_m={num_m} T={T} main={main} x {s_main} + tail x {s_tail}: {items} items on {sms} SMs, "
            f"longest chunk {longest} tiles")
    print(f"[plan] {label}{case}: {plan}")
    if "waves" in wants:
        assert items > sms, f"{case}: meant to give more work items than SMs, got {plan}"
    if "tail" in wants:
        assert main < num_m, f"{case}: meant to be a tail plan, got {plan}"
    if "long" in wants:
        assert longest >= 4, f"{case}: meant to sweep chunks of 4+ tiles (full candidate lists), got {plan}"
    return plan


def _same(got, want, what):
    import torch
    gi, gs, gc = got
    wi, ws, wc = want
    assert torch.equal(gc, wc), f"{what}: {int((gc != wc).sum())} counts differ"
    assert torch.equal(gi, wi), f"{what}: {int((gi != wi).sum())} index mismatches"
    assert torch.equal(gs.view(torch.int64), ws.view(torch.int64)), f"{what}: similarities are not bit-equal"


def _equal_oracle(got, want, what):
    idx, sim, cnt = got
    oidx, osim, ocnt = want
    assert (cnt == ocnt).all(), f"{what}: {(cnt != ocnt).sum()} counts differ"
    assert (idx == oidx).all(), f"{what}: {(idx != oidx).any(axis=1).sum()} rows with index mismatches"
    assert sim.tobytes() == osim.tobytes(), f"{what}: re-scored similarities are not bit-equal to the oracle"


def _sets_oracle(got, want, what):
    """CERTIFIED: the oracle's sets, each value within REL_TOL of the oracle's value for that index"""
    idx, sim, cnt = got
    oidx, osim, ocnt = want
    assert (cnt == ocnt).all(), f"{what}: {(cnt != ocnt).sum()} counts differ"
    big = np.iinfo(np.int64).max
    g = np.argsort(np.where(idx >= 0, idx, big), axis=1, kind="stable")
    o = np.argsort(np.where(oidx >= 0, oidx, big), axis=1, kind="stable")
    gi, gs = np.take_along_axis(idx, g, 1), np.take_along_axis(sim, g, 1)
    oi, os_ = np.take_along_axis(oidx, o, 1), np.take_along_axis(osim, o, 1)
    assert (gi == oi).all(), f"{what}: {(gi != oi).any(axis=1).sum()} rows with a different top-k set"
    m = oi >= 0
    rel = np.abs(gs[m] - os_[m]) / np.abs(os_[m])
    assert rel.max(initial=0.0) <= REL_TOL, f"{what}: relative error {rel.max()}"


def _stats(ctx):
    from mahout_b200.sketch import last_band_rows, last_fallback_rows
    return f"fallback rows {last_fallback_rows(ctx)}, band rows {last_band_rows(ctx)}"


# --- 1. the schedule does not change the answer (tensor precision) ---------------------------------------------

@pytest.mark.parametrize("k,threshold,exclude_self", [(5, None, True), (50, None, True), (100, None, True),
                                                      (192, None, True), (100, 0.3, True), (100, None, False)])
def test_every_plan_gives_the_dense_topk(ctx, bank_a, dense_a, monkeypatch, capfd, k, threshold, exclude_self):
    """k = 5: ksel 32, optional raises from 128 entries, rationed away in bulk; k = 192: ksel = CAP - 64, raises from
    384 entries, lists that pass LCAP - HALF take the forced raise.  chunks=1: 47-tile whole-row sweeps (the most
    forced raises); chunks=16: ~10 items per CTA, 32 lists per row in k_merge; main=2 / main=4: tail plans."""
    from mahout_b200.sketch import cosine_topk_blocks
    b = bank_a
    want = _tensor_ref(dense_a, k, threshold, exclude_self)
    for case, env, wants in (PLANNER, CHUNKS1, CHUNKS3, CHUNKS16, MAIN2, MAIN4):
        _use_plan(monkeypatch, env)
        capfd.readouterr()
        got = cosine_topk_blocks(ctx, b.rows, b.valid, b.rows.unsqueeze(0), b.valid.unsqueeze(0), b.d, W, k,
                                 b_id=(1, b.E), threshold=threshold, exclude_self=exclude_self, precision="tensor")
        plan = _witness(capfd, ctx, case, wants, f"A k={k} threshold={threshold} exclude_self={exclude_self} ")
        _same(got, want, f"{case} ({plan})")


# --- 2. exact precisions against the oracle --------------------------------------------------------------------

@pytest.mark.parametrize("precision", ["rescored", "certified"])
@pytest.mark.parametrize("which", ["A", "B"])
def test_exact_precisions_at_scale(ctx, bank_a, bank_b, oracle_a, oracle_b, monkeypatch, capfd, which, precision):
    k = 100
    if which == "A":
        b, rows, want = bank_a, np.arange(bank_a.E), _prefix(oracle_a, k)
    else:
        b, (rows, want) = bank_b, oracle_b
    for case, env, wants in (PLANNER, CHUNKS1, CHUNKS16):
        _use_plan(monkeypatch, env)
        capfd.readouterr()
        idx, sim, cnt = b.sk.cosine_topk(k, precision=precision)
        plan = _witness(capfd, ctx, case, wants, f"{which} {precision} ")
        got = (idx[rows], sim[rows], cnt[rows])
        what = f"{which} {case} ({plan}; {_stats(ctx)})"
        (_equal_oracle if precision == "rescored" else _sets_oracle)(got, want, what)


@pytest.mark.parametrize("precision", ["rescored", "certified"])
def test_multipass_large_k_at_scale(ctx, bank_a, oracle_a, monkeypatch, capfd, precision):
    """k = 300 > CAP - 64: the candidates are collected 128 ranks at a time (row ceilings) over the tail plan"""
    _use_plan(monkeypatch, {})
    capfd.readouterr()
    got = bank_a.sk.cosine_topk(300, precision=precision)
    plan = _witness(capfd, ctx, *PLANNER[::2], f"A {precision} k=300 ")
    (_equal_oracle if precision == "rescored" else _sets_oracle)(got, oracle_a, f"k=300 ({plan}; {_stats(ctx)})")


# --- 3. tie groups across chunks and items ---------------------------------------------------------------------

@pytest.mark.parametrize("precision", ["tensor", "rescored", "certified"])
@pytest.mark.parametrize("k", [10, 50])
def test_tie_groups_across_chunks_and_items(ctx, bank_ties, oracle_ties, dense_ties, monkeypatch, capfd, k, precision):
    """Groups of equal values straddle the column chunks of a row, its work items and the waves: a list cuts a large
    group by index (warp_compact_list) and publishes row_thr = k-th value - 1 ulp, so that the row's other lists
    still admit the tie; the lower index must win, as in the oracle."""
    b = bank_ties
    want = _prefix(oracle_ties, k)
    if precision == "tensor":
        from mahout_b200.sketch import cosine_topk_blocks
        want_t = _tensor_ref(dense_ties, k)
    for case, env, wants in (PLANNER, CHUNKS1, CHUNKS16):
        _use_plan(monkeypatch, env)
        capfd.readouterr()
        if precision == "tensor":
            got = cosine_topk_blocks(ctx, b.rows, b.valid, b.rows.unsqueeze(0), b.valid.unsqueeze(0), b.d, W, k,
                                     b_id=(1, b.E), precision="tensor")
            plan = _witness(capfd, ctx, case, wants, f"ties k={k} tensor ")
            _same(got, want_t, f"{case} ({plan})")
            continue
        idx, sim, cnt = b.sk.cosine_topk(k, precision=precision)
        plan = _witness(capfd, ctx, case, wants, f"ties k={k} {precision} ")
        what = f"{case} ({plan}; {_stats(ctx)})"
        if precision == "rescored":
            _equal_oracle((idx, sim, cnt), want, what)
        else:
            assert (cnt == want[2]).all() and (idx == want[0]).all(), f"{what}: {(idx != want[0]).sum()} index mismatches"


# --- 4. mixed-sign counters ------------------------------------------------------------------------------------

def test_mixed_sign_counters_at_scale(ctx, bank_mixed, monkeypatch, capfd):
    """similarities cluster around zero and almost every column passes the initial threshold: every list fills"""
    k = 100
    b = bank_mixed
    want = b.oracle(np.arange(b.E), k)
    for case, env, wants in (PLANNER, CHUNKS1):
        _use_plan(monkeypatch, env)
        capfd.readouterr()
        got = b.sk.cosine_topk(k, precision="rescored")
        plan = _witness(capfd, ctx, case, wants, "mixed-sign rescored ")
        assert b.sk.sign_info()
        _equal_oracle(got, want, f"{case} ({plan}; {_stats(ctx)})")


# --- 5. block_n = 128 ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("k", [5, 192])
def test_block_n_128_plans(ctx, bank_a, monkeypatch, capfd, k):
    """BN = 128: HALF = 64, forced raises from LCAP - HALF = 448 entries.  (The values of a BN = 128 sweep are only
    compared with the dense values of a BN = 128 sweep.)"""
    from mahout_b200.sketch import cosine_topk_blocks
    b = bank_a
    dense = _dense(ctx, b, block_n=128)
    want = _tensor_ref(dense, k)
    del dense
    for case, env, wants in (("planner", {}, ("waves", "long")), CHUNKS1,
                             ("chunks=32", {"MB200_COS_CHUNKS": "32"}, ("waves",))):
        _use_plan(monkeypatch, env)
        capfd.readouterr()
        got = cosine_topk_blocks(ctx, b.rows, b.valid, b.rows.unsqueeze(0), b.valid.unsqueeze(0), b.d, W, k,
                                 b_id=(1, b.E), precision="tensor", block_n=128)
        plan = _witness(capfd, ctx, case, wants, f"A BN=128 k={k} ")
        _same(got, want, f"{case} ({plan})")


# --- 6. incremental job ----------------------------------------------------------------------------------------

def _shards(mb, ctx, bank, G):
    """shard banks (owner = index % G) of one bank -> rows [G,d,per,ld], valid [G,d,vw], counters [G,per,d,w]"""
    import torch
    E, d = bank.E, bank.d
    counters = bank.sk.counters_tensor()
    per = E // G
    rows, valid, cnts = [], [], []
    for g in range(G):
        sh = mb.SketchBank(per, W, d, 42, 1, ctx)
        sh.counters_tensor().copy_(counters[g::G])
        torch.cuda.synchronize()
        r, v = sh.normalize()
        rows.append(r)
        valid.append(v)
        cnts.append(sh.counters_tensor().clone())
        sh.close()
    out = torch.stack(rows), torch.stack(valid), torch.stack(cnts)
    torch.cuda.synchronize()                           # (read on the library's stream)
    return out


@pytest.mark.parametrize("precision", ["tensor", "rescored"])
@pytest.mark.parametrize("plan_case", [("chunks=1", {"MB200_COS_CHUNKS": "1"}, ("long",)),
                                       ("chunks=12", {"MB200_COS_CHUNKS": "12"}, ("waves",))], ids=lambda p: p[0])
def test_incremental_job_at_scale(mb, ctx, bank_a, monkeypatch, capfd, precision, plan_case):
    """3 shards of bank A, the B side pushed as row chunks of 1024 of all blocks: the carry merge after pushes of
    full lists (chunks=1: 12-tile sweeps) or of many items (chunks=12) gives the one-shot result bit for bit"""
    import torch
    from mahout_b200.sketch import CosineJob, cosine_topk_blocks
    k, G = 100, 3
    d, E = bank_a.d, bank_a.E
    b_rows, b_valid, b_cnt = _shards(mb, ctx, bank_a, G)
    per = E // G
    case, env, wants = plan_case
    _use_plan(monkeypatch, env)
    for g in range(G):
        kw = dict(a_counters=b_cnt[g], b_counters=b_cnt) if precision == "rescored" else {}
        capfd.readouterr()
        one = cosine_topk_blocks(ctx, b_rows[g], b_valid[g], b_rows, b_valid, d, W, k, a_id=(G, g), b_id=(G, 1),
                                 precision=precision, **kw)
        _witness(capfd, ctx, case, wants, f"A/3 shard {g} one-shot {precision} ")
        job = CosineJob(ctx, b_rows[g], b_valid[g], d, W, k, a_id=(G, g), precision=precision)
        for c0 in range(0, per, 1024):
            c1 = min(per, c0 + 1024)
            rows_c = b_rows[:, :, c0:c1].contiguous()
            valid_c = b_valid[:, :, c0 // 32:(c1 + 31) // 32].contiguous()
            vw = int(mb._native.lib().mb200_valid_words(c1 - c0))
            vpad = torch.zeros((G, d, vw), dtype=torch.int32, device=valid_c.device)
            vpad[:, :, :valid_c.shape[2]] = valid_c
            torch.cuda.synchronize()                   # (the job reads them on the library's stream)
            capfd.readouterr()
            job.push(rows_c, vpad, id_mul=G, id_add=1, id_base=c0 * G)
            _witness(capfd, ctx, case, wants, f"A/3 shard {g} push rows {c0}:{c1} {precision} ")
        torch.cuda.synchronize()
        got = job.finish(b_id=(G, 1), **kw)
        _same(got, one, f"shard {g}, {case}, {precision}")


# --- 7. the strided item form of the fused pull-gather, on one GPU ---------------------------------------------

@pytest.mark.parametrize("precision", ["tensor", "rescored"])
@pytest.mark.parametrize("plan_case", [("planner", {}, ("long",)),
                                       ("chunks=8", {"MB200_COS_CHUNKS": "8"}, ("waves",))], ids=lambda p: p[0])
def test_fused_pull_gather_schedule_on_one_gpu(mb, ctx, bank_b, monkeypatch, capfd, precision, plan_case):
    """G = 4 shards of bank B emulated on one GPU: the "peer" buffers are device tensors, mb200_gather_pull stages them
    and publishes the arrival flags, K3 sweeps the staged operand in the strided item form (chunk sI takes every
    Sr-th tile, the blocks rotated to start at first_block = g).  The pulls are waited for before the push: this test
    is about the tile order, the rotation and the flag reads, not about a copy overlapping the persistent kernel.
    Result == the unfused call over the same blocks, bit for bit."""
    import torch
    from mahout_b200 import _native as N
    from mahout_b200.sketch import CosineJob, cosine_topk_blocks
    k, G = 100, 4
    d = bank_b.d
    b_rows, b_valid, b_cnt = _shards(mb, ctx, bank_b, G)
    case, env, wants = plan_case
    _use_plan(monkeypatch, env)
    staging_rows, staging_valid = torch.empty_like(b_rows), torch.empty_like(b_valid)
    peer_rows = (C.c_void_p * G)(*[b_rows[g].data_ptr() for g in range(G)])
    peer_valid = (C.c_void_p * G)(*[b_valid[g].data_ptr() for g in range(G)])
    rows_bytes, valid_bytes = b_rows[0].numel() * b_rows.element_size(), b_valid[0].numel() * b_valid.element_size()
    lib = N.lib()
    for g in range(G):
        kw = dict(a_counters=b_cnt[g], b_counters=b_cnt) if precision == "rescored" else {}
        capfd.readouterr()
        one = cosine_topk_blocks(ctx, b_rows[g], b_valid[g], b_rows, b_valid, d, W, k, a_id=(G, g), b_id=(G, 1),
                                 precision=precision, **kw)
        unfused = _witness(capfd, ctx, case, (), f"B/4 shard {g} unfused {precision} ")
        staging_rows.zero_()
        staging_valid.zero_()
        torch.cuda.synchronize()
        flags, epoch = C.c_void_p(), C.c_uint32()
        N.check(lib.mb200_gather_pull(ctx.handle, C.c_void_p(staging_rows.data_ptr()),
                                      C.c_void_p(staging_valid.data_ptr()), C.cast(peer_rows, C.c_void_p),
                                      C.cast(peer_valid, C.c_void_p), G, g, rows_bytes, valid_bytes,
                                      C.byref(flags), C.byref(epoch)), ctx.handle)
        N.check(lib.mb200_gather_wait(ctx.handle), ctx.handle)
        job = CosineJob(ctx, b_rows[g], b_valid[g], d, W, k, a_id=(G, g), precision=precision)
        capfd.readouterr()
        job.push(staging_rows, staging_valid, id_mul=G, id_add=1, ready=(flags.value, epoch.value), first_block=g)
        plan = _witness(capfd, ctx, case, wants, f"B/4 shard {g} fused {precision} ")
        torch.cuda.synchronize()
        if precision == "rescored":
            got = job.finish(b_id=(G, 1), resident_b=(staging_rows, staging_valid), **kw)
        else:
            got = job.finish()
        _same(got, one, f"shard {g}, fused {plan} vs unfused {unfused}, {precision}")
