"""CosineCM with a CountMinSketchConfig on all GPUs of the process (mb200_sized_multi_*): the config-3 population
with the roles swapped (tools/cmsized_perf.py's `config3`: 138 493 users x 26 744 items, 2 * 10^7 events, every
user's (w, d) from CountMinSketchConfig(q = 1.0), hash seed 42), all users, n = 100 neighbours, how_many = 10, at
G = 1, 2, 4 and 8 GPUs (those that are visible).

For each G, in one process:
  create_s          mb200_sized_multi_create: one sized bank per GPU, built in parallel
  neighborhood_s    mb200_sized_multi_neighborhood for all users
  recommend_s       mb200_sized_multi_recommend for all users (each GPU computes its users' neighbourhoods, then
                    recommends over them: the neighbourhood time is part of it)
each the best of --repeats after one warm-up call; the calls return host arrays, so they end device-synchronised.
Per timed call: the per-GPU worker seconds of the best run and the imbalance max / mean; the speed-up against G = 1;
a byte-for-byte check of every output array against G = 1's; and bit parity with the oracle (oracle.sized,
oracle.sized_recommend) on --parity sampled users.  The bank's device bytes per GPU (one full replica each) are
counted from the shapes.  Prints one JSON line with every GPU's name and power limit; --dry prints the shape model
only (no GPU).
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from cmsized_perf import N_NB, SEED, population, shapes  # noqa: E402


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return [[x.strip() for x in line.split(",")] for line in out]
    except Exception as e:        # the JSON line still says what could not be read
        return [[f"unknown ({e})", "unknown"]]


def bank_bytes(w, d, nnz):
    """device bytes of one sized bank (mb200_sized_bank_create's allocations): counters (cells + 2 cells of
    padding), per-row sums of squares, quanta, hash residues [max depth][nnz], and per user width, depth (int32),
    counter / row / pref offsets (int64, U + 1 each) and the class member list (int32)"""
    U = w.shape[0]
    cells = int((w.astype(np.int64) * d).sum())
    rows = int(d.astype(np.int64).sum())
    return {"counters": (cells + 2) * 8, "sumsq": rows * 8, "quanta": nnz * 8, "hash_residues": nnz * int(d.max()) * 8,
            "per_user": 4 * U * 3 + 8 * (U + 1) * 3}


def _best(fn, repeats, seconds):
    """best wall time of `repeats` calls after a warm-up, the per-GPU seconds of that call, its output"""
    fn()                                                    # warm-up
    best, per = float("inf"), None
    for _ in range(repeats):
        t = time.perf_counter()
        out = fn()
        dt = time.perf_counter() - t
        if dt < best:
            best, per = dt, seconds()
    return best, per, out


def _equal(a, b):
    """integers by value, floats byte for byte (NaN slots included)"""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind == "f" or b.dtype.kind == "f":
        return a.dtype == b.dtype and a.tobytes() == b.tobytes()
    return a.shape == b.shape and bool((a == b).all())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,4,8", help="G values, limited to the visible GPUs")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--parity", type=int, default=64)
    ap.add_argument("--how-many", type=int, default=10)
    ap.add_argument("--dry", action="store_true", help="population, shapes and bank bytes only (no GPU)")
    args = ap.parse_args()
    U, I, (ptr, item, pref) = population("config3")
    w, d = shapes(ptr, I)
    nnz = int(ptr[-1])
    bb = bank_bytes(w, d, nnz)
    out = {"tool": "cmsized_multi_perf", "population": "config3", "users": U, "items": I, "prefs": nnz, "n": N_NB,
           "how_many": args.how_many, "q": 1.0, "bank_bytes_per_gpu": sum(bb.values()), "bank_bytes": bb}
    if args.dry:
        print(json.dumps(out))
        return
    import torch
    import mahout_b200 as mb
    from mahout_b200.multi import MultiGpu
    from oracle import recommend as orec
    from oracle import sized as osz
    from oracle.sized_recommend import sized_recommend
    out["gpus"] = _gpu_info()
    visible = torch.cuda.device_count()
    out["gpus_visible"] = visible
    Gs = [g for g in (int(x) for x in args.gpus.split(",")) if g <= visible]
    users = np.arange(U, dtype=np.int64)
    data = orec.item_csr(np.repeat(np.arange(U), np.diff(ptr)), item, U)
    hfb = mb.HashFunctionBuilder(SEED)
    pick = np.sort(np.random.Generator(np.random.PCG64(SEED + 9)).choice(U, min(args.parity, U), replace=False))
    ref, oracle_out, runs = None, None, {}
    for G in Gs:
        multi = MultiGpu(G)
        r = {"G": G}
        banks = []

        def create():
            banks.append(multi.sized_bank(w, d, hfb, ptr, item, pref, 1))
            if len(banks) > 1:
                banks.pop(0).close()
        r["create_s"], r["create_gpu_s"], _ = _best(create, args.repeats, lambda: banks[-1].stats()["seconds"])
        many = banks[-1]
        secs = lambda: many.stats()["seconds"]                                  # noqa: E731
        r["neighborhood_s"], r["neighborhood_gpu_s"], nb = _best(lambda: many.neighborhood(users, N_NB),
                                                                 args.repeats, secs)
        r["neighborhood_work"] = many.stats()["work"]
        r["recommend_s"], r["recommend_gpu_s"], rec = _best(
            lambda: many.recommend_users(users, N_NB, -np.inf, *data, args.how_many), args.repeats, secs)
        for k in ("create", "neighborhood", "recommend"):
            s = np.asarray(r[f"{k}_gpu_s"])
            r[f"{k}_imbalance"] = float(s.max() / s.mean())
        if ref is None:
            ref = (nb, rec, r)
            t = time.perf_counter()
            oi, osim, oc = osz.sized_neighborhood(w, d, many.a, many.b, ptr, item, pref, users[pick], N_NB)
            wi, wv, wc = sized_recommend(w, d, many.a, many.b, ptr, item, pref, oi, osim, oc, *data, users[pick],
                                         args.how_many)
            oracle_out = ((oi, osim, oc), (wi, wv, wc))
            out["oracle_s"] = time.perf_counter() - t
        r["bytes_equal_g1"] = all(a.tobytes() == b.tobytes() for a, b in zip(nb + rec, ref[0] + ref[1]))
        r["oracle_parity_users"] = int(pick.shape[0])
        r["oracle_parity"] = all(_equal(a[pick], b) for a, b in zip(nb + rec, oracle_out[0] + oracle_out[1]))
        for k in ("create", "neighborhood", "recommend"):
            r[f"{k}_speedup"] = ref[2][f"{k}_s"] / r[f"{k}_s"]
        many.close()
        multi.close()
        runs[str(G)] = r
        print(json.dumps(r), file=sys.stderr, flush=True)
    out["runs"] = runs
    print(json.dumps(out))


if __name__ == "__main__":
    main()
