"""Item-based recommendation on all GPUs of the process (mb200_itembased_multi_*) at the config-3 population.

Workload: tools/itembased_perf.py's -- synthetic events (mahout_b200.synth, Zipf(1.1) items), 26 744 items, 138 493
users, 2 * 10^7 events, seed 42, prepared on GPU 0; item lists of the sketch measure, d = 4, W = 4096, k = 100,
re-scored, on GPU 0; recommend(howMany = 10) for every user at maxPrefsPerUser = 10 and unlimited.

For G = 1, 2, 4 and 8 (those that are visible), in one process:
  create_s      mb200_itembased_multi_create: the host lists, user CSR and itemIDs copied to every GPU in parallel
  call_s        one mb200_itembased_multi_recommend for all users per maxPrefsPerUser setting
each the best of --repeats after one warm-up call; the calls take and return host arrays, so they end
device-synchronised.  Per timed call: the per-GPU worker seconds of the best run and the imbalance max / mean; the
speed-up against G = 1; a byte-for-byte check of every output array against G = 1's (and G = 1's against
itembased.recommend on one context); bit parity with oracle/itembased.py on --parity sampled users.  Then the whole
job, `recommenditembased` on the same events written as text, without --numGpus and with --numGpus G: its phase times
(RecommenderJob.phase_s) and whether its file equals the single-GPU job's.  Prints one JSON line with every GPU's name
and power limit, read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED, W, D = 42, 4096, 4
SETTINGS = (("maxPrefsPerUser_10", 10), ("maxPrefsPerUser_unlimited", 2 ** 31 - 1))


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return [[x.strip() for x in line.split(",")] for line in out]
    except Exception as e:        # the JSON line still says what could not be read
        return [[f"unknown ({e})", "unknown"]]


def _best(fn, repeats, seconds):
    """best wall time of `repeats` calls after a warm-up, the per-GPU seconds of that call, its output"""
    fn()                                                    # warm-up
    best, per, out = float("inf"), None, None
    for _ in range(repeats):
        t = time.perf_counter()
        out = fn()
        dt = time.perf_counter() - t
        if dt < best:
            best, per = dt, seconds()
    return best, per, out


def _text(user, item, pref) -> bytes:
    """`user,item,pref` lines, zero-padded to fixed width (Long.parseLong reads the leading zeros); the synthetic
    prefs are multiples of 0.5 in [0.5, 5]"""
    def digits(v, w):
        v = v.astype(np.int64)
        return np.stack([(v // 10 ** (w - 1 - j)) % 10 + 48 for j in range(w)], 1).astype(np.uint8)
    uw, iw = len(str(int(user.max()))), len(str(int(item.max())))
    half = np.rint(pref.astype(np.float64) * 2).astype(np.int64)
    cols = [digits(user, uw), np.full((user.shape[0], 1), 44, np.uint8), digits(item, iw),
            np.full((user.shape[0], 1), 44, np.uint8), digits(half // 2, 1), np.full((user.shape[0], 1), 46, np.uint8),
            np.where(half % 2 == 1, 53, 48).astype(np.uint8)[:, None], np.full((user.shape[0], 1), 10, np.uint8)]
    return np.ascontiguousarray(np.concatenate(cols, 1)).tobytes()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=26_744)
    ap.add_argument("--users", type=int, default=138_493)
    ap.add_argument("--events", type=int, default=20_000_000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--how-many", type=int, default=10)
    ap.add_argument("--gpus", default="1,2,4,8", help="G values, limited to the visible GPUs")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--parity", type=int, default=64, help="sampled users compared with the oracle")
    ap.add_argument("--no-job", action="store_true", help="skip the recommenditembased runs")
    args = ap.parse_args()

    import torch
    import mahout_b200 as mb
    from mahout_b200 import ingest, itembased as ib, similarity as sim, synth
    from mahout_b200.multi import MultiGpu
    from mahout_b200.recommenditembased import RecommenderJob
    from oracle import itembased as oib

    res = {"bench": "itembased_multi_perf", "gpus": _gpu_info(), "gpus_visible": torch.cuda.device_count(),
           "events": args.events, "measure": "sketch", "width": W, "depth": D, "k": args.k,
           "how_many": args.how_many}
    ctx = mb.Context(0)
    cdf = torch.from_numpy(synth.zipf_cdf(args.items, 1.1)).cuda()
    perm = torch.from_numpy(synth.rank_permutation(args.items, SEED)).cuda()
    user, item, pref = synth.events_device(ctx, SEED, 0, args.events, args.users, cdf, perm)
    ev = ingest.Events.from_arrays(user, item, pref, ctx=ctx)
    prep = ev.prepare(1)
    ev.close()
    uv = ib.user_vectors(prep.row, prep.user, prep.pref)
    lists = sim.item_similarity(prep.row, prep.user, prep.pref, prep.num_items, k=args.k, width=W, depth=D,
                                seed=SEED, ctx=ctx, device=True)
    host_lists = tuple(x.cpu().numpy() for x in lists)
    host_uv = ib.UserVectors(*(x.cpu().numpy() for x in (uv.user_ids, uv.user_ptr, uv.pref_row, uv.pref_val)))
    item_id = prep.item_id
    U = host_uv.num_users
    res.update(items=int(prep.num_items), users=U, prefs=int(prep.n),
               replica_bytes=int(sum(x.nbytes for x in host_lists) + host_uv.user_ptr.nbytes
                                 + host_uv.pref_row.nbytes + host_uv.pref_val.nbytes + item_id.nbytes))
    sample = np.linspace(0, U - 1, min(args.parity, U)).astype(np.int64)
    oracle = {label: oib.recommend(*host_lists, host_uv.user_ptr, host_uv.pref_row, host_uv.pref_val, item_id, sample,
                                   args.how_many, P) for label, P in SETTINGS}
    single = {label: tuple(x.cpu().numpy() for x in ib.recommend(lists, uv, torch.from_numpy(item_id).cuda(), None,
                                                                 args.how_many, P, ctx=ctx))
              for label, P in SETTINGS}

    Gs = [g for g in (int(x) for x in args.gpus.split(",")) if g <= res["gpus_visible"]]
    ref, runs = None, {}
    for G in Gs:
        multi = MultiGpu(G)
        r = {"G": G}
        made = []

        def create():
            made.append(multi.item_based(host_lists, host_uv, item_id))
            if len(made) > 1:
                made.pop(0).close()
        r["create_s"], r["create_gpu_s"], _ = _best(create, args.repeats, lambda: made[-1].stats()["seconds"])
        many = made[-1]
        outs = {}
        for label, P in SETTINGS:
            s, per, out = _best(lambda: many.recommend(None, args.how_many, P), args.repeats,
                                lambda: many.stats()["seconds"])
            outs[label] = out
            gi, gv, gc = out
            wi, wv, wc = oracle[label]
            r[label] = {"call_s": s, "gpu_s": per, "imbalance": float(np.max(per) / np.mean(per)),
                        "work": many.stats()["work"],
                        "parity": bool((gc[sample] == wc).all() and (gi[sample] == wi).all()
                                       and (gv[sample].view(np.int32) == wv.view(np.int32)).all())}
        if ref is None:
            ref = (outs, r)
            r["bytes_equal_single_context"] = all(a.tobytes() == b.tobytes() for label, _ in SETTINGS
                                                  for a, b in zip(outs[label], single[label]))
        r["bytes_equal_g1"] = all(a.tobytes() == b.tobytes() for label, _ in SETTINGS
                                  for a, b in zip(outs[label], ref[0][label]))
        r["create_speedup"] = ref[1]["create_s"] / r["create_s"]
        for label, _ in SETTINGS:
            r[label]["speedup"] = ref[1][label]["call_s"] / r[label]["call_s"]
        many.close()
        multi.close()
        runs[str(G)] = r
        print(json.dumps(r), file=sys.stderr, flush=True)
    res["runs"] = runs
    res["parity"] = all(r[label]["parity"] for r in runs.values() for label, _ in SETTINGS)
    res["bytes_equal"] = all(r["bytes_equal_g1"] for r in runs.values()) and \
        bool(runs and runs[str(Gs[0])]["bytes_equal_single_context"])

    if not args.no_job:
        u, i, p = (x.cpu().numpy() for x in (user, item, pref))
        job = {}
        with tempfile.TemporaryDirectory() as td:
            inp = os.path.join(td, "prefs.csv")
            with open(inp, "wb") as f:
                f.write(_text(u, i, p))
            base = ["-i", inp, "-s", "SIMILARITY_SKETCH_COSINE", "-m", str(args.k), "--sketchWidth", str(W),
                    "--sketchDepth", str(D), "--sketchSeed", str(SEED), "--precision", "rescored",
                    "--numRecommendations", str(args.how_many)]
            want = None
            for G in [None] + Gs:
                out = os.path.join(td, f"out{G}.txt")
                j = RecommenderJob()
                t = time.perf_counter()
                rc = j.run(base + ["-o", out] + ([] if G is None else ["--numGpus", str(G)]))
                entry = {"rc": rc, "total_s": time.perf_counter() - t, "phase_s": j.phase_s}
                data = open(out, "rb").read() if rc == 0 else None
                if G is None:
                    want = data
                else:
                    entry["file_equal_single"] = data is not None and data == want
                job["single" if G is None else f"G{G}"] = entry
                print(json.dumps({"job": G, **entry}), file=sys.stderr, flush=True)
        res["job"] = job
    print(json.dumps(res), flush=True)
    prep.close()
    ctx.close()
    return 0 if res["parity"] and res["bytes_equal"] else 1


if __name__ == "__main__":
    sys.exit(main())
