"""User-based recommendation at the config-3 population with the roles swapped (users are the sketched entities):
K_RECOMMEND and the batched doEstimatePreference on one GPU, with oracle parity on sampled users.

Workload: synthetic events (mahout_b200.synth.events_numpy, Zipf(1.1) items), U = 138 493 users, I = 26 744 items,
2 * 10^7 events, bank entity = user, key = item, d = 4, W = 4096, hash seed 42.  90 % of the events build the bank and
the data model, 10 % are held out for estimate_preferences.

  1. neighbourhoods: cosine_topk(n = 100, rescored), device-resident;
  2. recommend_all(howMany = 10) over --users evenly spaced users (after a warm-up), device-synchronised;
  3. estimate_preferences over the held-out pairs.

Prints one JSON line: GPU name and power limit, users/s, candidate estimates/s, candidate counts, the stream / gather
split, K_RECOMMEND ms, the bytes model (streamed users: rows x W x 8 bytes per candidate chunk; gathered users:
candidates x neighbours x d x 32-byte sectors) over the 6544 GB/s HBM copy rate measured on B200, bit parity with
oracle/recommend.py on --parity users, and a CPU stand-in: the numpy restatement on all cores over the same sampled
users, extrapolated to the population (labelled as such).
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

HBM_COPY_GBPS = 6544.0   # device-to-device copy rate measured on B200 (DESIGN.md section 6)

_ORC = {}


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return name, power
    except Exception as e:        # the JSON line still says what could not be read
        return f"unknown ({e})", "unknown"


def _oracle_user(t):
    from oracle import recommend as orec
    o = _ORC
    u = int(o["users"][t])
    return orec.recommend(o["bank"], o["a"], o["b"], o["nb_idx"], o["nb_sim"], o["nb_cnt"], o["ptr"], o["col"],
                          o["ids"], [u], o["how_many"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, default=4096, help="users timed in recommend_all")
    ap.add_argument("--parity", type=int, default=64, help="users compared with the oracle")
    ap.add_argument("--events", type=int, default=20_000_000)
    ap.add_argument("--neighbours", type=int, default=100)
    ap.add_argument("--how-many", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()

    import torch
    import mahout_b200 as mb
    from mahout_b200 import _native as N
    from mahout_b200 import synth
    from mahout_b200.cosinecm import CosineCM
    from mahout_b200.recommender import GenericUserBasedRecommender

    U, I, W, D, SEED = 138_493, 26_744, 4096, 4, 42
    name, power = _gpu_info()
    cdf = synth.zipf_cdf(I, 1.1)
    user, item, pref = synth.events_numpy(SEED, 0, args.events, U, cdf, synth.rank_permutation(I, SEED))
    held = np.random.Generator(np.random.PCG64(SEED)).random(args.events) < 0.1
    ctx = mb.Context(0)
    t0 = time.perf_counter()
    cm = CosineCM(user[~held], item[~held], pref[~held], W, D, SEED, ctx=ctx)
    rec = GenericUserBasedRecommender(cm, args.neighbours)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    n_users = cm.user_ids.shape[0]
    sample = cm.user_ids[np.linspace(0, n_users - 1, min(args.users, n_users)).astype(np.int64)]

    rec.recommend_all(args.how_many, sample[:256])                      # warm-up
    ctx.set_profiling(True)
    ctx.reset_profile()
    times = []
    for _ in range(args.repeats):
        torch.cuda.synchronize()
        t = time.perf_counter()
        ids, items, vals, cnt = rec.recommend_all(args.how_many, sample)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t)
    k_ms, k_n = ctx.kernel_time(N.K_RECOMMEND)
    plan = cm.bank.recommend_plan()
    k_ms_call = k_ms / max(k_n, 1)
    bytes_model = plan["stream_rows"] * W * 8 + plan["gather_loads"] * 32
    call_s = min(times)

    # held-out pairs: doEstimatePreference over the recommender's neighbourhoods
    hu, hi = user[held], item[held]
    known = np.isin(hu, cm.user_ids)
    hu, hi = hu[known], hi[known]
    rec.estimate_preferences(hu[:1000], hi[:1000])
    ctx.reset_profile()
    torch.cuda.synchronize()
    t = time.perf_counter()
    est = rec.estimate_preferences(hu, hi)
    torch.cuda.synchronize()
    est_s = time.perf_counter() - t
    est_k_ms, _ = ctx.kernel_time(N.K_RECOMMEND)
    ctx.set_profiling(False)

    # parity with the oracle on sampled users, over an oracle bank of those users and their neighbours
    import oracle as orc
    from oracle import recommend as orec
    from multiprocessing import get_context
    par = sample[np.linspace(0, sample.shape[0] - 1, min(args.parity, sample.shape[0])).astype(np.int64)]
    prow = cm._rows(par)
    nb_idx, nb_sim, nb_cnt = (x.cpu().numpy() for x in (rec.nb_idx, rec.nb_sim, rec.nb_cnt))
    need = np.unique(np.concatenate([prow] + [nb_idx[r, :nb_cnt[r]] for r in prow]))
    remap = np.full(n_users, -1, np.int64)
    remap[need] = np.arange(need.shape[0])
    rows_all = np.searchsorted(cm.user_ids, user[~held])
    keep = remap[rows_all] >= 0
    a, b = orc.hash_params(SEED, D)
    bank = np.zeros((need.shape[0], D, W))
    orc.bank_update(bank, D, W, a, b, remap[rows_all[keep]], item[~held][keep], pref[~held][keep],
                    nthreads=orc.max_threads())
    sub_idx = np.where(nb_idx[need] >= 0, remap[np.maximum(nb_idx[need], 0)], -1)
    ptr, col, ids_o = orec.item_csr(remap[rows_all[keep]], item[~held][keep], need.shape[0])
    _ORC.update(bank=bank, a=a, b=b, nb_idx=sub_idx, nb_sim=nb_sim[need], nb_cnt=nb_cnt[need], ptr=ptr, col=col,
                ids=ids_o, users=remap[prow], how_many=args.how_many)
    workers = max(1, min(os.cpu_count() or 1, par.shape[0]))
    t = time.perf_counter()
    with get_context("fork").Pool(workers) as pool:
        res = pool.map(_oracle_user, range(par.shape[0]))
    cpu_s = time.perf_counter() - t
    got_i, got_v, got_c = (x[np.searchsorted(sample, par)] for x in (items, vals, cnt))
    mismatch = 0
    for t, (wi, wv, wc) in enumerate(res):
        ok = (got_c[t] == wc[0] and (got_i[t] == wi[0]).all() and (got_v[t].view(np.int32) == wv[0].view(np.int32)).all())
        mismatch += not ok

    out = {
        "bench": "recommend_perf", "gpu": name, "power_limit": power,
        "users_total": int(n_users), "items": I, "events_in_bank": int((~held).sum()), "width": W, "depth": D,
        "neighbours": args.neighbours, "how_many": args.how_many, "setup_s": round(setup_s, 2),
        "recommend_users_timed": int(sample.shape[0]), "recommend_call_s": round(call_s, 4),
        "users_per_s": round(sample.shape[0] / call_s, 1),
        "candidate_estimates_per_s": round(plan["candidates"] / call_s, 1),
        "candidates_mean": round(plan["candidates"] / sample.shape[0], 1), "candidates_max": plan["candidates_max"],
        "stream_users": plan["stream_users"], "gather_users": plan["gather_users"], "chunks": plan["chunks"],
        "stages": plan["stages"], "chunk_candidates": plan["chunk_candidates"],
        "k_recommend_ms_per_call": round(k_ms_call, 3),
        "bytes_model_GB": round(bytes_model / 1e9, 3),
        "bytes_model_GBps": round(bytes_model / (k_ms_call * 1e-3) / 1e9, 1),
        "bytes_model_fraction_of_hbm_copy": round(bytes_model / (k_ms_call * 1e-3) / 1e9 / HBM_COPY_GBPS, 3),
        "all_users_extrapolated_s": round(n_users * call_s / sample.shape[0], 1),
        "estimate_pairs": int(hu.shape[0]), "estimate_s": round(est_s, 4),
        "estimate_pairs_per_s": round(hu.shape[0] / est_s, 1), "estimate_kernel_ms": round(est_k_ms, 3),
        "estimate_nan_fraction": round(float(np.isnan(est).mean()), 4),
        "oracle_parity_users": int(par.shape[0]), "oracle_parity_mismatches": int(mismatch),
        "cpu_standin": f"numpy restatement (oracle/recommend.py), {workers} processes, {par.shape[0]} users, "
                       "extrapolated to all users",
        "cpu_standin_users_per_s": round(par.shape[0] / cpu_s, 2),
        "cpu_standin_all_users_extrapolated_s": round(n_users * cpu_s / par.shape[0], 1),
    }
    print(json.dumps(out), flush=True)
    cm.close()
    ctx.close()
    return 0 if mismatch == 0 else 1


if __name__ == "__main__":
    sys.exit(main())
