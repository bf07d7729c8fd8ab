#!/usr/bin/env python
"""Small end-to-end pass over every kernel family, meant to run under compute-sanitizer (SURVEY.md section 5):

    compute-sanitizer --tool memcheck  python tools/sanitize_small.py all
    compute-sanitizer --tool racecheck python tools/sanitize_small.py k1        # shared-memory hazards of K1 / grouping / routing

Checks its results against the oracle as it goes (a sanitizer run that computes garbage proves nothing)."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mahout_b200 as mb
from mahout_b200 import _native as N
import oracle as orc

what = sys.argv[1] if len(sys.argv) > 1 else "all"
ctx = mb.Context(0)
rng = np.random.Generator(np.random.PCG64(1))

# ---- K1 single sketch
n, d, w = 30011, 4, 4096
key = np.minimum(rng.zipf(1.1, n), 10 ** 6).astype(np.int64)
inc = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
a, b = orc.hash_params(42, d)
want = np.zeros((1, d, w))
orc.bank_update(want, d, w, a, b, None, key, inc)
bank = mb.SketchBank(1, w, d, 42, 1, ctx)
bank.update(None, key, inc)
assert bank.read().tobytes() == want.tobytes()
bank.close()
bank = mb.SketchBank(1, w, d, 42, 1, ctx)
bank.update_u8(None, key.astype(np.uint32), (inc * 2).astype(np.uint8))
assert bank.read().tobytes() == want.tobytes()
bank.close()
print("K1 single: ok", flush=True)

# ---- K1 bank mode: direct, grouped (one and two partition levels), CSR
for E in (300, 1500):
    n = 40000
    ent = (np.minimum(rng.zipf(1.2, n), E) - 1).astype(np.int64)
    key = rng.integers(0, 5000, n).astype(np.int64)
    key[::11] = -7
    inc = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
    want = np.zeros((E, d, 256))
    orc.bank_update(want, d, 256, a, b, ent, key, inc)
    for gmin in (0, 1 << 62):
        ctx.set_option(N.OPT_GROUP_MIN_EVENTS, gmin)
        bank = mb.SketchBank(E, 256, d, 42, 1, ctx)
        bank.update(ent, key, inc)
        assert bank.read().tobytes() == want.tobytes(), (E, gmin)
        bank.close()
    order = np.argsort(ent, kind="stable")
    rp = np.searchsorted(ent[order], np.arange(E + 1)).astype(np.int64)
    bank = mb.SketchBank(E, 256, d, 42, 1, ctx)
    bank.update_grouped(rp, key[order], inc[order])
    assert bank.read().tobytes() == want.tobytes()
    bank.close()
ctx.set_option(N.OPT_GROUP_MIN_EVENTS, 1 << 16)
print("K1 bank: ok", flush=True)

# ---- routing (one shard set on one GPU: every destination is local memory)
import ctypes as C
import torch
G, n = 4, 20000
row = torch.from_numpy(rng.integers(0, 1000, n).astype(np.int64)).cuda()
usr = torch.from_numpy(rng.integers(0, 99999, n).astype(np.int64)).cuda()
prf = torch.from_numpy((rng.integers(1, 11, n) * 0.5).astype(np.float32)).cuda()
cnt = np.zeros(G, np.int64)
N.check(N.lib().mb200_route_count(ctx.handle, C.c_void_p(row.data_ptr()), n, G, cnt.ctypes.data_as(C.c_void_p)), ctx.handle)
assert cnt.tolist() == np.bincount(row.cpu().numpy() % G, minlength=G).tolist()
dst = [[torch.empty(int(c), dtype=t, device="cuda") for c in cnt] for t in (torch.int64, torch.int64, torch.float32)]
ptrs = [(C.c_void_p * G)(*[x.data_ptr() for x in col]) for col in dst]
off = np.zeros(G, np.int64)
N.check(N.lib().mb200_route_scatter(ctx.handle, C.c_void_p(row.data_ptr()), C.c_void_p(usr.data_ptr()), C.c_void_p(prf.data_ptr()),
                                    n, G, C.cast(ptrs[0], C.c_void_p), C.cast(ptrs[1], C.c_void_p), C.cast(ptrs[2], C.c_void_p),
                                    off.ctypes.data_as(C.c_void_p)), ctx.handle)
ctx.sync()
for g in range(G):
    m = (row % G) == g
    got = sorted(zip(dst[0][g].cpu().tolist(), dst[1][g].cpu().tolist(), dst[2][g].cpu().tolist()))
    exp = sorted(zip((row[m] // G).cpu().tolist(), usr[m].cpu().tolist(), prf[m].cpu().tolist()))
    assert got == exp, g
print("route: ok", flush=True)
if what == "k1":
    sys.exit(0)

# ---- cosine stage: K2, K3, K5 in the three precisions, band pass and exact path, ingest
E, d, w, k = 400, 2, 256, 20
n = 50 * E
item = rng.integers(0, E, n).astype(np.int64)
user = rng.integers(1, 200, n).astype(np.int64)
pref = (rng.integers(1, 11, n) * 0.5).astype(np.float32)
a2, b2 = orc.hash_params(42, d)
ref = np.zeros((E, d, w))
orc.bank_update(ref, d, w, a2, b2, item, user, pref)
oidx, osim, ocnt = orc.bank_cosine_topk(ref, k)
bank = mb.SketchBank(E, w, d, 42, 1, ctx)
bank.update(item, user, pref)
for precision in ("tensor", "certified", "rescored"):
    for dtype in ("f16", "bf16"):
        idx, sim, cnt_ = bank.cosine_topk(k, dtype=dtype, precision=precision)
        assert (cnt_ == ocnt).all()
        if precision == "rescored":
            assert (idx == oidx).all() and sim.tobytes() == osim.tobytes()
os.environ["MB200_NO_BAND"] = "1"
idx, sim, cnt_ = bank.cosine_topk(k, dtype="bf16", precision="rescored")
assert (idx == oidx).all() and sim.tobytes() == osim.tobytes()
del os.environ["MB200_NO_BAND"]
bank.close()
from mahout_b200 import ingest
lines = [f"{u},{i},{p}" for u, i, p in zip(user[:3000].tolist(), item[:3000].tolist(), pref[:3000].tolist())]
ev = ingest.Events.parse("\n".join(lines) + "\n", ctx=ctx)
pm = ev.prepare(2)
pm.close()
ev.close()
ctx.close()
print("cosine + ingest: ok", flush=True)
