"""CosineCM with a CountMinSketchConfig on one GPU: NearestNUserNeighborhood over per-user sketch sizes
(mb200_sized_neighborhood), with oracle parity on sampled queries.

Populations (each user's (w, d) = cm_dims of CountMinSketchConfig(q = 1.0), hash seed 42, n = 100 neighbours):
  ml100k   MovieLens-100K shape: 943 users x 1682 items, about 10^5 prefs (user activity lognormal(0, 1), item popularity (r + 10)^-0.9); all users
  config3  the config-3 population with the roles swapped: 138 493 users x 26 744 items, 2 * 10^7 events of
           mahout_b200.synth (users uniform, items Zipf(1.1)), one pref per (user, item); 4096 sampled queries and
           all users
  zipf     the same with users drawn Zipf(1.0): shapes spread to large n, so the per-CTA global slice runs at scale;
           4096 sampled queries (all users too when --all-zipf)

Per call: time (best of --repeats, device-synchronised, after one warm-up call), pair FMAs from the shape model (sum
over candidate users v != query of d_v * w_v), FMA/s, the plan (mb200_sized_last_plan) and bit parity of the lists
with orc_sized_neighborhood on --parity sampled queries.  Prints one JSON line with the GPU's name and power limit.
--dry prints the shape model only (no GPU).

Recommend leg (config3, --recommend-populations): recommend(user, 10) over the users' n = 100 neighbourhoods
(mb200_sized_recommend) for the 4096 sampled users, then all users.  Per call: time (best of --repeats after a
warm-up, device-synchronised), users/s, neighbour terms/s (sum over users of candidates x listed neighbours other than
the user), the plan (mb200_sized_recommend_last_plan), the bytes model (streamed bytes + 32 B per gathered counter)
over the time as a share of 7.7 TB/s of HBM, the neighbourhood time of the same users beside it, and bit parity with
oracle.sized_recommend on --parity sampled users.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED, N_NB = 42, 100


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return name, power
    except Exception as e:        # the JSON line still says what could not be read
        return f"unknown ({e})", "unknown"


def _model(user, item, pref, U):
    """one pref per (user, item) -- the first -- as CSR by user row"""
    key = user.astype(np.int64) * (1 << 32) + item.astype(np.int64)
    _, first = np.unique(key, return_index=True)
    first.sort()
    user, item, pref = user[first], item[first], pref[first]
    order = np.argsort(user, kind="stable")
    ptr = np.zeros(U + 1, np.int64)
    np.cumsum(np.bincount(user, minlength=U), out=ptr[1:])
    return ptr, item[order].astype(np.int64), pref[order].astype(np.float32)


def population(name):
    from mahout_b200 import synth
    if name == "ml100k":
        rng = np.random.Generator(np.random.PCG64(SEED))
        U, I = 943, 1682
        w = rng.lognormal(0.0, 1.0, U)
        user = np.concatenate([np.arange(U), rng.choice(U, 125_000 - U, p=w / w.sum())])
        pop = 1.0 / (np.arange(I) + 10.0) ** 0.9
        item = rng.choice(I, user.shape[0], p=pop / pop.sum()) + 1
        pref = (rng.integers(1, 11, user.shape[0]) * 0.5).astype(np.float32)
        return U, I, _model(user, item, pref, U)
    U, I, n = 138_493, 26_744, 20_000_000
    user, item, pref = synth.events_numpy(SEED, 0, n, U, synth.zipf_cdf(I, 1.1), synth.rank_permutation(I, SEED))
    user = user - 1                                       # userIDs 1..U -> rows
    if name == "zipf":
        cdf = synth.zipf_cdf(U, 1.0)
        r = np.random.Generator(np.random.PCG64(SEED + 1)).random(n)
        user = np.minimum(np.searchsorted(cdf, r), U - 1)
    return U, I, _model(user.astype(np.int64), item, pref, U)


def shapes(ptr, I):
    from mahout_b200.cmconfig import CountMinSketchConfig
    import oracle as orc
    U = ptr.shape[0] - 1
    n = np.diff(ptr)
    cfg = CountMinSketchConfig(1.0)
    cfg.configure(np.arange(U), n, I)
    dims = {}
    w = np.empty(U, np.int32)
    d = np.empty(U, np.int32)
    for u in range(U):
        k = (cfg.getDelta(u), cfg.getEpsilon(u))
        if k not in dims:
            dims[k] = orc.cm_dims(*k)
        w[u], d[u] = dims[k]
    return w, d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--populations", default="ml100k,config3,zipf")
    ap.add_argument("--queries", type=int, default=4096)
    ap.add_argument("--parity", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--all-zipf", action="store_true", help="also time all users on the zipf population")
    ap.add_argument("--dry", action="store_true", help="shape model only, no GPU")
    ap.add_argument("--recommend-populations", default="config3", help="populations of the recommend leg ('' = none)")
    ap.add_argument("--how-many", type=int, default=10)
    args = ap.parse_args()
    out = {"tool": "cmsized_perf", "n": N_NB, "q": 1.0}
    if not args.dry:
        out["gpu"], out["power_limit"] = _gpu_info()
    for name in args.populations.split(","):
        U, I, (ptr, item, pref) = population(name)
        w, d = shapes(ptr, I)
        cells = w.astype(np.int64) * d
        rec = {"users": U, "items": I, "prefs": int(ptr[-1]), "classes": len(set(zip(w.tolist(), d.tolist()))),
               "cells": int(cells.sum()), "max_cells": int(cells.max()), "max_prefs": int(np.diff(ptr).max())}
        calls = [("all", np.arange(U))]
        if U > 4096:
            sample = np.sort(np.random.Generator(np.random.PCG64(SEED)).choice(U, args.queries, replace=False))
            calls = [("sample", sample)] + ([] if name == "zipf" and not args.all_zipf else calls)
        rec["calls"] = {}
        for label, qrows in calls:
            fmas = int(qrows.shape[0] * cells.sum() - cells[qrows].sum())
            rec["calls"][label] = {"queries": int(qrows.shape[0]), "pair_fmas": fmas}
        if not args.dry:
            run(rec, name, w, d, ptr, item, pref, calls, args)
            if name in args.recommend_populations.split(","):
                run_recommend(rec, w, d, ptr, item, pref, calls, args)
        out[name] = rec
        print(json.dumps({name: rec}), file=sys.stderr, flush=True)
    print(json.dumps(out))


def run(rec, name, w, d, ptr, item, pref, calls, args):
    import torch
    import mahout_b200 as mb
    from oracle import sized as osz
    ctx = mb.Context(0)
    dev = f"cuda:{ctx.device}"
    t0 = time.perf_counter()
    bank = mb.SizedBank(w, d, mb.HashFunctionBuilder(SEED), ptr, item, pref, 1, ctx)
    ctx.sync()
    rec["build_s"] = time.perf_counter() - t0
    for label, qrows in calls:
        c = rec["calls"][label]
        q = torch.from_numpy(qrows).to(dev)
        res = bank.neighborhood(q, N_NB)        # warm-up
        torch.cuda.synchronize(ctx.device)
        best = float("inf")
        for _ in range(args.repeats):
            t = time.perf_counter()
            res = bank.neighborhood(q, N_NB)
            torch.cuda.synchronize(ctx.device)
            best = min(best, time.perf_counter() - t)
        c["time_s"] = best
        c["fma_per_s"] = c["pair_fmas"] / best
        c["plan"] = bank.plan()
        pick = np.random.Generator(np.random.PCG64(SEED + 7)).choice(qrows.shape[0], min(args.parity,
                                                                                         qrows.shape[0]),
                                                                     replace=False)
        t = time.perf_counter()
        oi, osim, oc = osz.sized_neighborhood(w, d, bank.a, bank.b, ptr, item, pref, qrows[pick], N_NB)
        c["oracle_s"] = time.perf_counter() - t
        gi, gs, gc = (x.cpu().numpy()[pick] for x in res)
        c["parity_queries"] = int(pick.shape[0])
        c["parity"] = bool((gc == oc).all() and (gi == oi).all() and gs.tobytes() == osim.tobytes())
    bank.close()
    ctx.close()


HBM_BYTES_PER_S = 7.7e12   # HGX B200 data sheet, one GPU


def run_recommend(rec, w, d, ptr, item, pref, calls, args):
    import torch
    import mahout_b200 as mb
    from oracle import recommend as orec
    from oracle.sized_recommend import sized_recommend
    ctx = mb.Context(0)
    dev = f"cuda:{ctx.device}"
    U = w.shape[0]
    bank = mb.SizedBank(w, d, mb.HashFunctionBuilder(SEED), ptr, item, pref, 1, ctx)
    data = orec.item_csr(np.repeat(np.arange(U), np.diff(ptr)), item, U)
    data_d = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in data]
    rec["recommend"] = {}
    for label, qrows in calls:
        c = {"users": int(qrows.shape[0]), "how_many": args.how_many}
        q = torch.from_numpy(qrows).to(dev)
        t = time.perf_counter()
        lists = bank.neighborhood(q, N_NB)
        torch.cuda.synchronize(ctx.device)
        c["neighborhood_s"] = time.perf_counter() - t
        res = bank.recommend(*lists, *data_d, q, args.how_many)        # warm-up
        torch.cuda.synchronize(ctx.device)
        best = float("inf")
        for _ in range(args.repeats):
            t = time.perf_counter()
            res = bank.recommend(*lists, *data_d, q, args.how_many)
            torch.cuda.synchronize(ctx.device)
            best = min(best, time.perf_counter() - t)
        pl = bank.recommend_plan()
        c["time_s"] = best
        c["users_per_s"] = qrows.shape[0] / best
        c["terms_per_s"] = pl["terms"] / best
        c["plan"] = pl
        c["model_bytes"] = pl["stream_bytes"] + 32 * pl["gather_loads"]
        c["hbm_share"] = c["model_bytes"] / best / HBM_BYTES_PER_S
        pick = np.sort(np.random.Generator(np.random.PCG64(SEED + 9)).choice(qrows.shape[0], min(args.parity,
                                                                                                qrows.shape[0]),
                                                                             replace=False))
        idx, sim, cnt = (x.cpu().numpy()[pick] for x in lists)
        t = time.perf_counter()
        wi, wv, wc = sized_recommend(w, d, bank.a, bank.b, ptr, item, pref, idx, sim, cnt, *data, qrows[pick],
                                     args.how_many)
        c["oracle_s"] = time.perf_counter() - t
        gi, gv, gc = (x.cpu().numpy()[pick] for x in res)
        c["parity_users"] = int(pick.shape[0])
        c["parity"] = bool((gc == wc).all() and (gi == wi).all() and gv.tobytes() == wv.tobytes())
        rec["recommend"][label] = c
    bank.close()
    ctx.close()


if __name__ == "__main__":
    main()
