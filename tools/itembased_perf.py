"""Item-based recommendation (RecommenderJob's aggregate-and-recommend phase, k_itembased) at the config-3 population.

Workload: synthetic events (mahout_b200.synth, Zipf(1.1) items), 26 744 items, 138 493 users, 2 * 10^7 events, seed
42, prepared on the device (last pref of a (user, item) wins).  Item lists: the sketch measure, d = 4, W = 4096,
k = 100, re-scored, device-resident.  Then recommend(howMany = 10) for every user, with maxPrefsPerUser = 10 (the
default) and unlimited, so that both accumulator paths run: users whose considered lists hold at most 1024 entries
accumulate in the shared-memory table, the others in dense slices (ties at the pruning threshold can lift a user
with P = 10 over that bound).

Prints one JSON line: card name and power limit; per maxPrefsPerUser setting the call time (host clock around a
synchronising call, best of --repeats after a warm-up) and K_RECOMMEND time from the library's device events, users/s
and partial products/s (list entries visited, from the plan), the plan split; the phase times (prepare, similarity,
recommend); bit parity with oracle/itembased.py on --parity sampled users of each setting.
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


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return name, power
    except Exception as e:        # the JSON line still says what could not be read
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=26_744)
    ap.add_argument("--users", type=int, default=138_493)
    ap.add_argument("--events", type=int, default=20_000_000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--how-many", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--parity", type=int, default=64, help="sampled users compared with the oracle per setting")
    args = ap.parse_args()

    import torch
    import mahout_b200 as mb
    from mahout_b200 import _native as N
    from mahout_b200 import ingest, itembased as ib, similarity as sim, synth
    from oracle import itembased as oib

    SEED, W, D = 42, 4096, 4
    name, power = _gpu_info()
    ctx = mb.Context(0)
    cdf = torch.from_numpy(synth.zipf_cdf(args.items, 1.1)).cuda()
    perm = torch.from_numpy(synth.rank_permutation(args.items, SEED)).cuda()
    user, item, pref = synth.events_device(ctx, SEED, 0, args.events, args.users, cdf, perm)

    torch.cuda.synchronize()
    t = time.perf_counter()
    ev = ingest.Events.from_arrays(user, item, pref, ctx=ctx)
    prep = ev.prepare(1)
    ev.close()
    uv = ib.user_vectors(prep.row, prep.user, prep.pref)
    torch.cuda.synchronize()
    prepare_s = time.perf_counter() - t

    t = time.perf_counter()
    lists = sim.item_similarity(prep.row, prep.user, prep.pref, prep.num_items, k=args.k, width=W, depth=D,
                                seed=SEED, ctx=ctx, device=True)
    torch.cuda.synchronize()
    similarity_s = time.perf_counter() - t

    item_id = torch.from_numpy(prep.item_id).cuda()
    users = torch.arange(uv.num_users, dtype=torch.int64, device="cuda")
    host = dict(idx=lists[0].cpu().numpy(), sim=lists[1].cpu().numpy(), cnt=lists[2].cpu().numpy(),
                ptr=uv.user_ptr.cpu().numpy(), prow=uv.pref_row.cpu().numpy(), pval=uv.pref_val.cpu().numpy())
    sample = np.linspace(0, uv.num_users - 1, min(args.parity, uv.num_users)).astype(np.int64)

    runs = {}
    for label, P in (("maxPrefsPerUser_10", 10), ("maxPrefsPerUser_unlimited", 2 ** 31 - 1)):
        ib.recommend(lists, uv, item_id, users[:4096], args.how_many, P, ctx=ctx)          # warm-up
        ctx.set_profiling(True)
        ctx.reset_profile()
        times = []
        for _ in range(args.repeats):
            torch.cuda.synchronize()
            t = time.perf_counter()
            out = ib.recommend(lists, uv, item_id, users, args.how_many, P, ctx=ctx)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t)
        k_ms, k_n = ctx.kernel_time(N.K_RECOMMEND)
        ctx.set_profiling(False)
        plan = ib.itembased_plan(ctx)
        call_s = min(times)
        gi, gv, gc = (x.cpu().numpy() for x in out)
        wi, wv, wc = oib.recommend(host["idx"], host["sim"], host["cnt"], host["ptr"], host["prow"], host["pval"],
                                   prep.item_id, sample, args.how_many, P)
        parity = bool((gc[sample] == wc).all() and (gi[sample] == wi).all()
                      and (gv[sample].view(np.int32) == wv.view(np.int32)).all())
        runs[label] = {
            "call_s": round(call_s, 5), "k_recommend_ms_per_call": round(k_ms / args.repeats, 3),
            "k_recommend_launches_per_call": k_n // args.repeats,
            "users_per_s": round(uv.num_users / call_s, 1),
            "partial_products_per_s": round(plan["entries"] / call_s, 1),
            "partial_products": plan["entries"], "entries_max": plan["entries_max"],
            "smem_users": plan["smem_users"], "dense_users": plan["dense_users"], "pruned_users": plan["pruned_users"],
            "candidates_max": plan["candidates_max"], "dense_slices": plan["dense_slices"],
            "users_with_recommendations": int((gc > 0).sum()),
            "oracle_parity_users": int(sample.shape[0]), "parity": parity,
        }
    res = {
        "bench": "itembased_perf", "gpu": name, "power_limit": power,
        "items": int(prep.num_items), "users": int(uv.num_users), "prefs": int(prep.n), "events": args.events,
        "measure": "sketch", "width": W, "depth": D, "k": args.k, "how_many": args.how_many,
        "phase_s": {"prepare": round(prepare_s, 4), "similarity": round(similarity_s, 4),
                    "recommend_maxPrefsPerUser_10": runs["maxPrefsPerUser_10"]["call_s"]},
        **runs,
        "parity": all(r["parity"] for r in runs.values()),
    }
    print(json.dumps(res), flush=True)
    prep.close()
    ctx.close()
    return 0 if res["parity"] else 1


if __name__ == "__main__":
    sys.exit(main())
