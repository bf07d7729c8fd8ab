"""Single-sketch K1 (k_update_single_v2): the direct path against the key-table path, A/B in one process.

Workload: config 2 of bench.py -- device-resident synthetic events (mahout_b200.synth, seed 20240002, 10^7 items),
Zipf 1.1 and 1.5, one d = 4 x W = 2^20 sketch, 10^9 events per launch.  The path is chosen per call through the
MB200_K1_KEYTABLE_MIN_EVENTS override (0 = table, huge = direct).  For each Zipf exponent, after two warm-up calls
of each path, --reps repetitions alternate --launches timed calls of the direct path and of the table path on the same
resident events (CUDA events around the launches, stream-ordered); the two banks then receive the same events the
same number of times and their counters must be equal.  One extra call of each path runs with MB200_TRACE set, and
its trace line gives the L2 reductions per event.

--sweep also times both paths on prefixes of the Zipf 1.1 events (2^20 .. 2^28 events): the crossover that sets
KT_MIN_EVENTS in sketch.cu.

Prints JSON lines: the card's name and power limit, then one line per Zipf exponent (ms per launch of every
repetition, G events/s of the best, speed-up, reductions per event, counters equal) and one per sweep size.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ENV = "MB200_K1_KEYTABLE_MIN_EVENTS"
NEVER = str(2 ** 63 - 1)
PATHS = {"direct": NEVER, "table": "0"}


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return name, power
    except Exception as e:        # the JSON line still says what could not be read
        return f"unknown ({e})", "unknown"


def _traced(fn):
    """run fn() with MB200_TRACE set and return the library's k1 trace line (read from fd 2)"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as f:
        os.dup2(f.fileno(), 2)
        os.environ["MB200_TRACE"] = "1"
        try:
            fn()
        finally:
            del os.environ["MB200_TRACE"]
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read().decode(errors="replace")
    lines = [ln for ln in text.splitlines() if "k1: path=" in ln]
    if not lines:
        raise RuntimeError(f"no k1 trace line in: {text!r}")
    kv = dict(re.findall(r"(\w+)=(\S+)", lines[-1]))
    return {k: (v if k == "path" else float(v)) for k, v in kv.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=float, default=1e9)
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--zipf", type=float, nargs="+", default=[1.1, 1.5])
    ap.add_argument("--sweep", action="store_true")
    args = ap.parse_args()

    import torch
    import mahout_b200 as mb
    from mahout_b200 import synth

    name, power = _gpu_info()
    print(json.dumps({"gpu": name, "power_limit": power}), flush=True)
    ctx = mb.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    n = int(args.events)

    def run(bank, path, item, pref):
        os.environ[ENV] = PATHS[path]
        bank.update(None, item, pref)

    def timed(bank, path, item, pref, launches):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(launches):
            run(bank, path, item, pref)
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / launches

    for s in args.zipf:
        cdf = torch.from_numpy(synth.zipf_cdf(10_000_000, s)).cuda()
        _, item, pref = synth.events_device(ctx, 20240002, 0, n, 1_000_000, cdf, None, want_user=False)
        banks = {p: mb.SketchBank(1, 1 << 20, 4, 42, 1, ctx) for p in PATHS}
        for p in PATHS:
            for _ in range(2):
                run(banks[p], p, item, pref)
        ms = {p: [] for p in PATHS}
        for _ in range(args.reps):
            for p in PATHS:
                ms[p].append(timed(banks[p], p, item, pref, args.launches))
        trace = {p: _traced(lambda p=p: run(banks[p], p, item, pref)) for p in PATHS}
        for b in banks.values():
            b.check()
        equal = bool(torch.equal(banks["direct"].counters_tensor(), banks["table"].counters_tensor()))
        best = {p: min(v) for p, v in ms.items()}
        print(json.dumps({
            "zipf": s, "events_per_launch": n, "launches_per_rep": args.launches, "gpu": name, "power_limit": power,
            "ms_per_launch": ms, "G_events_per_s": {p: n / best[p] / 1e6 for p in PATHS},
            "speedup": best["direct"] / best["table"],
            "reds_per_event": {p: trace[p]["reds_per_event"] for p in PATHS}, "trace": trace,
            "counters_equal": equal}), flush=True)
        for b in banks.values():
            b.close()
        if args.sweep and s == args.zipf[0]:
            for lg in range(20, 29):
                m = 1 << lg
                if m > n:
                    break
                k = max(args.launches, min(200, (1 << 30) // m))
                sb = {p: mb.SketchBank(1, 1 << 20, 4, 42, 1, ctx) for p in PATHS}
                for p in PATHS:
                    timed(sb[p], p, item[:m], pref[:m], 2)
                r = {p: [] for p in PATHS}
                for _ in range(args.reps):
                    for p in PATHS:
                        r[p].append(timed(sb[p], p, item[:m], pref[:m], k))
                eq = bool(torch.equal(sb["direct"].counters_tensor(), sb["table"].counters_tensor()))
                print(json.dumps({"sweep_events": m, "launches_per_rep": k, "ms_per_launch": r,
                                  "table_over_direct": min(r["table"]) / min(r["direct"]), "counters_equal": eq}),
                      flush=True)
                for b in sb.values():
                    b.close()
        del item, pref
        torch.cuda.empty_cache()
    os.environ.pop(ENV, None)
    ctx.close()


if __name__ == "__main__":
    main()
