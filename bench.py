#!/usr/bin/env python
"""bench.py -- headline benchmark of the sketch-similarity hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

Workload (BASELINE.json configs[1]): count-min sketch update of synthetic Zipf(1.1)
(user, item, pref) events over 10^7 items into one depth-4 x width-2^20 sketch; one step = one
pass of K1 over one HBM-resident batch of 10^9 events (12 B/event read: item key + pref).
Prints ONE JSON line (see DESIGN.md "Measurement" for every field).

N > 1 (launched by torchrun, one rank per GPU): every rank streams its own 10^9-event slice
into a private replica sketch (weak scaling, no data-path collective) and one NCCL all-reduce
of the 32 MiB counter array per step produces the single global sketch (SURVEY.md 8e).

--impl reference times the reference's CPU algorithm (oracle/ C port, all host threads) on a
bounded sample of the same event stream; the Java itself cannot run here (no JVM in the image).

--dump-outputs DIR writes what the timed steps computed, as float64 DIR/<name>.npy (rank 0, under 64 MB):
sketch.npy, the [depth, width] sketch after the last step (the all-reduced one at N > 1), and, unless --no-cosine,
cosine_<precision>_{idx,sim,cnt}.npy of the cosine stage's last step for a fixed sample of rows whose global item
ids are cosine_rows.npy.  The inputs depend only on the arguments, so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree the benchmark runs from may be read-only: no caches next to the sources

SEED = 20240002           # SURVEY.md 8d: 20240001 + config number (config 2 -> ...0003 is 1-based; fixed here)
SKETCH_SEED = 42
DEPTH, WIDTH = 4, 1 << 20
ITEMS, USERS, ZIPF_S = 10_000_000, 1_000_000, 1.1
# SURVEY.md 8d's algorithmic model: event read + d x (8 B read + 8 B write) per FP64 counter RMW.  The single-sketch
# kernel reads 12 B per event (8 B key + 4 B preference; no entity column), a bank-mode event is 20 B.
ALGO_BYTES_PER_EVENT = 12 + DEPTH * 16
BANK_BYTES_PER_EVENT = 20 + DEPTH * 16
# ncu --set full of k_update_single_v2 on this workload (profiles/r2_k_update_single_v2_ncu.txt, one launch of 2.5e8
# events): 3.05 GB of DRAM traffic and 286.7 M RED requests -- the physical side of the roofline object
K1_DRAM_BYTES_PER_EVENT = 12.21
K1_REDS_PER_EVENT = 1.147
C3_USERS, C3_ITEMS, C3_EVENTS, C3_WIDTH, C3_DEPTH, C3_K = 138_493, 26_744, 20_000_000, 4096, 4, 50
C3_SEED = 20240003
C3_CHUNKS = 4              # all-gather chunks per step of the pipelined multi-GPU cosine form
METRIC = "sketch_updates_per_sec"
UNIT = "events/s"
DUMP_ROWS = 4096           # cosine-stage rows written by --dump-outputs (a seeded sample)
DUMP_MAX_BYTES = 64_000_000


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=float(j["hbm_gbs"]), bf16=float(j.get("bf16_tflops_sustained", j["bf16_tflops"])),
                    bf16_burst=float(j["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, bf16=1400.0, bf16_burst=1590.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index: int, period: float = 0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def _write_dump(path: str, arrays: dict):
    """--dump-outputs: every array as float64 DIR/<name>.npy"""
    arrays = {name: np.ascontiguousarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def _host_threads() -> int:
    """all host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle's OpenMP
    regions take an explicit thread count)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def _physical_gpu_index(local: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on host cores
# ------------------------------------------------------------------------------------------------
def _cpu_update_rate(item, pref, threads: int):
    """events/s of the reference algorithm (oracle C port) on the given events."""
    import oracle as orc
    a, b = orc.hash_params(SKETCH_SEED, DEPTH)
    bank = np.zeros((1, DEPTH, WIDTH))
    t0 = time.perf_counter()
    orc.bank_update(bank, DEPTH, WIDTH, a, b, None, item, pref, nthreads=threads)
    dt = time.perf_counter() - t0
    return item.shape[0] / dt, dt, bank


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle as orc
    from mahout_b200 import synth
    threads = _host_threads()
    cdf = synth.zipf_cdf(ITEMS, ZIPF_S)
    _, item, pref = synth.events_numpy(SEED, 0, 1 << 22, USERS, cdf)
    rate, _, _ = _cpu_update_rate(item, pref, threads)           # calibration
    per_step = int(min(max(rate * 4.0, 1 << 25), 1 << 27))       # ~4 s of CPU work per step
    _, item, pref = synth.events_numpy(SEED, 0, per_step, USERS, cdf)
    for w in range(args.warmup):
        m = min(per_step, 1 << 22)
        _cpu_update_rate(item[:m], pref[:m], threads)
    t = 0.0
    for s in range(args.steps):
        _, dt, _ = _cpu_update_rate(item, pref, threads)
        t += dt
    value = per_step * args.steps / t
    sample = (f"first {per_step} events of the config-2 stream (Zipf({ZIPF_S}) over {ITEMS} items) per step, "
              f"d={DEPTH}, W=2^20")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": _config(args.gpus, per_step),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference Java cannot run (no JVM in image): oracle/ C port of HashFunction.hash + "
                "DoubleCountMinSketch.update, OpenMP over event slices with private sketches.  Each step times a "
                f"PREFIX of {per_step} events of the config-2 stream, not the 1e9 of the GPU arm: a rate measured on a "
                "bounded sample of the same workload (same generator, seed, sketch shape)",
        "sample_is_prefix_of_config": True,
    }
    if not args.no_cosine:
        line["cosine"] = _reference_cosine(threads)
    print(json.dumps(line), flush=True)


def _reference_cosine(threads: int):
    """configs[2] on the host cores: oracle sketch build (all 2e7 events) + DoubleCountMinSketch.cosine
    + top-k for a bounded sample of rows, all threads."""
    import oracle as orc
    from mahout_b200 import synth
    cdf = synth.zipf_cdf(C3_ITEMS, ZIPF_S)
    perm = synth.rank_permutation(C3_ITEMS, 3) - 1
    user, item, pref = synth.events_numpy(C3_SEED, 0, C3_EVENTS, C3_USERS, cdf, perm)
    a, b = orc.hash_params(SKETCH_SEED, C3_DEPTH)
    bank = np.zeros((C3_ITEMS, C3_DEPTH, C3_WIDTH))
    t0 = time.perf_counter()
    orc.bank_update(bank, C3_DEPTH, C3_WIDTH, a, b, item, user, pref, nthreads=1)
    build_s = time.perf_counter() - t0
    rows = threads * 16
    _, _, _, cpu_s = _cpu_cosine_rows(bank, list(range(rows)), C3_K, threads)
    value = rows * C3_ITEMS / cpu_s
    return {"metric": "item_pair_cosine_sims_per_sec", "value": value, "unit": "pairs/s",
            "config": {"workload": "configs[2]: MovieLens-20M-shaped synthetic, sketch d=4 x W=4096, cosine top-50",
                       "items": C3_ITEMS, "depth": C3_DEPTH, "width": C3_WIDTH, "k": C3_K},
            "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port",
                             "sample": f"{rows} rows x all {C3_ITEMS} columns, {cpu_s:.1f} s"},
            "sketch_build": {"events_per_s": C3_EVENTS / build_s, "events": C3_EVENTS, "s": build_s, "cores": 1},
            "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def _config(n_gpus: int, events_per_step: int):
    return {"workload": "configs[1]: count-min sketch update, synthetic Zipf(1.1) (user,item,pref) events over "
                        "1e7 items into depth=4 x width=2^20 sketch",
            "events_per_step_per_gpu": events_per_step, "depth": DEPTH, "width": WIDTH,
            "items": ITEMS, "zipf_s": ZIPF_S, "sketch_seed": SKETCH_SEED, "event_seed": SEED,
            "l2": "inputs_exceed_l2 (12 GB of events per step per GPU; the 32 MiB counter array is L2-resident state)",
            "parallelism": f"replica sketches x{n_gpus} + all-reduce(int64 sum)" if n_gpus > 1 else "single GPU"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import mahout_b200 as mb
    from mahout_b200 import _native as N
    from mahout_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    else:
        torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    peaks = _peaks()
    # host buffers of this rank live on the GPU's own NUMA node (matters for the e2e H2D path at N = 8)
    from mahout_b200.sketch import bind_host_thread_to_gpu
    orig_affinity = os.sched_getaffinity(0)
    numa_bound = bind_host_thread_to_gpu(local) if world > 1 else False

    ctx = mb.Context(local)
    # one non-default stream carries everything: the library's kernels, NCCL and the timing events
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    n = int(args.events)
    cdf = synth.zipf_cdf(ITEMS, ZIPF_S)
    cdf_dev = torch.from_numpy(cdf).to(dev)
    # resident batch: each rank owns events [rank*n, (rank+1)*n) of the stream
    _, item, pref = synth.events_device(ctx, SEED, rank * n, n, USERS, cdf_dev, None, want_user=False)
    bank = mb.SketchBank(1, WIDTH, DEPTH, SKETCH_SEED, 1, ctx)
    cptr, cells = bank.counters_ptr()
    from mahout_b200.sketch import _as_tensor
    counters = _as_tensor(cptr, cells, local)
    global_sketch = torch.empty_like(counters) if world > 1 else None

    def step():
        bank.update(None, item, pref)
        if world > 1:
            global_sketch.copy_(counters)
            dist.all_reduce(global_sketch, op=dist.ReduceOp.SUM)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
    bank.check()
    barrier()
    ctx.set_profiling(True)
    ctx.reset_profile()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(_physical_gpu_index(local))
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    k_ms, k_n = ctx.kernel_time(N.K_UPDATE)
    ctx.set_profiling(False)
    launches = ctx.launch_count() - launches0
    bank.check()
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * n * args.steps / (ms * 1e-3)

    # ---- end-to-end through the C ABI with HOST buffers (H2D inside, sketch read back) ----------
    e2e_n = int(min(n, args.e2e_events))
    hk = torch.empty(e2e_n, dtype=torch.int64).pin_memory()
    hp = torch.empty(e2e_n, dtype=torch.float32).pin_memory()
    hk.copy_(item[:e2e_n])
    hp.copy_(pref[:e2e_n])
    hout = torch.empty(DEPTH * WIDTH, dtype=torch.float64).pin_memory()
    hk_np, hp_np = hk.numpy(), hp.numpy()
    ebank = mb.SketchBank(1, WIDTH, DEPTH, SKETCH_SEED, 1, ctx)

    def e2e_step():
        N.check(N.lib().mb200_bank_update(ebank.handle, None, C.c_void_p(hk_np.ctypes.data),
                                          C.c_void_p(hp_np.ctypes.data), e2e_n, N.MEM_HOST), ctx.handle)
        N.check(N.lib().mb200_bank_read(ebank.handle, 0, 1, C.c_void_p(hout.data_ptr()), N.MEM_HOST),
                ctx.handle)

    # the narrow wire format of the same events (mb200_bank_update_u8): u32 key + one byte of quanta = 5 B/event
    # over PCIe instead of 12, and the sketch read back as int32 quanta (16 MiB instead of 32)
    hk32 = torch.empty(e2e_n, dtype=torch.int32).pin_memory()
    hq8 = torch.empty(e2e_n, dtype=torch.uint8).pin_memory()
    hk32.copy_(item[:e2e_n].to(torch.int32))
    hq8.copy_((pref[:e2e_n] * 2).to(torch.uint8))
    hout32 = torch.empty(DEPTH * WIDTH, dtype=torch.int32).pin_memory()
    hk32_np, hq8_np = hk32.numpy(), hq8.numpy()

    def e2e_step_narrow():
        N.check(N.lib().mb200_bank_update_u8(ebank.handle, None, C.c_void_p(hk32_np.ctypes.data),
                                             C.c_void_p(hq8_np.ctypes.data), e2e_n, N.MEM_HOST), ctx.handle)
        N.check(N.lib().mb200_bank_read_i32(ebank.handle, 0, 1, C.c_void_p(hout32.data_ptr()), N.MEM_HOST),
                ctx.handle)

    e2e_steps = max(2, min(args.steps, 5))

    def time_e2e(fn):
        for _ in range(2):
            fn()
        reps = []
        for _ in range(3):                      # the host side of a shared box is noisy: best of 3 repetitions
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                fn()
            barrier()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            reps.append(dt)
        return reps

    e2e_reps = time_e2e(e2e_step)
    e2e_s = min(e2e_reps)
    ebank.clear()
    narrow_reps = time_e2e(e2e_step_narrow)
    narrow_s = min(narrow_reps)
    # both formats feed the same counters
    ebank.clear()
    e2e_step_narrow()
    narrow_q = hout32.clone()
    ebank.clear()
    e2e_step()
    narrow_equal = bool(torch.equal(narrow_q.to(torch.float64) * 0.5, hout))
    # what the link itself delivers for the same bytes (explains the e2e number; not part of it)
    dkey = torch.empty(e2e_n, dtype=torch.int64, device=dev)
    dkey.copy_(hk, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    dkey.copy_(hk, non_blocking=True)
    torch.cuda.synchronize(dev)
    h2d_gbps = 8 * e2e_n / (time.perf_counter() - t0) / 1e9
    del dkey
    e2e_value = world * e2e_n * e2e_steps / e2e_s
    narrow_value = world * e2e_n * e2e_steps / narrow_s
    red_peak = synth.red64_peak(ctx, 22, 1 << 30)           # measured L2 RED.ADD.64 rate into a 32 MiB array

    if numa_bound:
        os.sched_setaffinity(0, orig_affinity)        # the CPU baseline below uses every core again
    # ---- parity + cpu_baseline on rank 0 ---------------------------------------------------------
    cpu = None
    parity = None
    if rank == 0:
        import oracle as orc
        threads = _host_threads()
        cal = 1 << 22
        rate, _, _ = _cpu_update_rate(item[:cal].cpu().numpy(), pref[:cal].cpu().numpy(), threads)
        sample = int(min(max(rate * (12.0 if world == 1 else 2.0), 1 << 25), 1 << 28, n))
        cpu_rate, cpu_dt, cpu_bank = _cpu_update_rate(item[:sample].cpu().numpy(),
                                                      pref[:sample].cpu().numpy(), threads)
        pbank = mb.SketchBank(1, WIDTH, DEPTH, SKETCH_SEED, 1, ctx)
        pbank.update(None, item[:sample], pref[:sample])
        got = pbank.read()
        parity = {"sketch_bit_exact": bool(got.tobytes() == cpu_bank.tobytes()), "events_checked": sample}
        pbank.close()
        s1 = int(min(sample, max(1 << 22, rate / max(threads, 1) * 2.0)))
        cpu1_rate, cpu1_dt, _ = _cpu_update_rate(item[:s1].cpu().numpy(), pref[:s1].cpu().numpy(), 1)
        cpu = {"value": cpu_rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"first {sample} events of rank 0's stream, {cpu_dt:.1f} s; oracle/ C port "
                         "(the Java reference cannot run: no JVM in the image)",
               # the reference is single-threaded per sketch (and serial under LocalJobRunner): SURVEY.md 8d
               "single_thread": {"value": cpu1_rate, "unit": UNIT, "cores": 1,
                                 "sample": f"first {s1} events, {cpu1_dt:.1f} s"}}

    dump = {} if args.dump_outputs and rank == 0 else None
    if dump is not None:
        if world > 1:
            q = global_sketch.view(DEPTH, WIDTH).to(torch.float64).cpu().numpy()
            dump["sketch"] = q * 2.0 ** -bank.frac_bits
        else:
            dump["sketch"] = bank.read()[0]
    # free the sketch-stage buffers before the cosine stage
    bank.close()
    ebank.close()
    del item, pref, hk, hp, counters
    torch.cuda.empty_cache()
    cosine = None
    if not args.no_cosine:
        cosine = run_cosine_stage(ctx, stream, world, rank, local, dev, peaks, args.steps, args.warmup, dump)
    if dump is not None:
        _write_dump(args.dump_outputs, dump)
    line = None
    if rank == 0:
        kern_s = (k_ms / max(k_n, 1)) * 1e-3
        model_gbps = ALGO_BYTES_PER_EVENT * n / kern_s / 1e9
        dram_gbps = K1_DRAM_BYTES_PER_EVENT * n / kern_s / 1e9
        reds = K1_REDS_PER_EVENT * n / kern_s
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64 fixed-point counters (== reference f64, exact)",
            "data": "synthetic", "config": _config(world, n),
            "clocks": clocks, "gpu_launches": int(launches),
            # headline e2e: the library's narrow wire format (u32 keys, one byte of quanta per event) from pinned host
            # memory + the sketch read back; the reference's own (long, float) layout is reported beside it
            "e2e": {"value": narrow_value, "unit": UNIT, "h2d_bytes_per_step": 5 * e2e_n,
                    "d2h_bytes_per_step": 4 * DEPTH * WIDTH,
                    "sample": f"{e2e_n} events/step from pinned host memory through mb200_bank_update_u8(MEM_HOST) "
                              "(u32 key + u8 quanta = 5 B/event) + mb200_bank_read_i32 of the whole sketch; best of 3 "
                              f"repetitions of {e2e_steps} steps",
                    "repetitions_s": narrow_reps, "counters_equal_wide_format": narrow_equal,
                    "wide_format": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 12 * e2e_n,
                                    "d2h_bytes_per_step": 8 * DEPTH * WIDTH, "repetitions_s": e2e_reps,
                                    "sample": "the same events as int64 key + float32 preference (the reference's parsed "
                                              "types) through mb200_bank_update(MEM_HOST) + mb200_bank_read (doubles)"},
                    "pinned_h2d_GBps": h2d_gbps, "host_threads_bound_to_gpu_numa_node": numa_bound,
                    "bound": "PCIe: bytes per event over the host link"},
            # frac is PHYSICAL: DRAM bytes per event measured with ncu x events / kernel time, against the measured
            # copy bandwidth.  The 32 MiB sketch is L2-resident, so the algorithmic model of SURVEY.md 8d (every
            # counter RMW as 16 B of HBM traffic) describes traffic that never reaches DRAM; its figure is kept under
            # "model" and may exceed 1.  What binds the kernel is the L2 reduction path: "l2_atomic".
            "roofline": {"bound": "hbm", "kernel": "k_update_single_v2", "achieved": dram_gbps, "peak": peaks["hbm"],
                         "unit": "GB/s", "frac": dram_gbps / peaks["hbm"],
                         "traffic": K1_DRAM_BYTES_PER_EVENT * n, "peak_source": peaks["source"],
                         "kernel_ms_per_launch": kern_s * 1e3, "launches_timed": int(k_n),
                         "dram_bytes_per_event_ncu": K1_DRAM_BYTES_PER_EVENT,
                         "model": {"algorithmic_bytes_per_event": ALGO_BYTES_PER_EVENT, "achieved": model_gbps,
                                   "frac": model_gbps / peaks["hbm"],
                                   "note": "12 B event + 4 x 16 B counter RMW as if every update went to HBM; the "
                                           "counters are L2-resident and ~3/4 of the events are absorbed in shared "
                                           "memory, so this is not a physical bound"},
                         "l2_atomic": {"peak_red64_per_s": red_peak, "reds_per_event_ncu": K1_REDS_PER_EVENT,
                                       "achieved_red64_per_s": reds, "frac": reds / red_peak,
                                       "peak_source": "mb200_bench_red64: RED.ADD.64 to uniformly random cells of a "
                                                      "32 MiB array, measured in this run"},
                         "atomic_updates_per_s": DEPTH * n / kern_s},
            "cpu_baseline": cpu, "parity": parity, "cosine": cosine,
        }
    # configs[3] / configs[4] run last, under a watchdog: if a stage hangs (a rank lost in a collective), the line
    # measured so far is still printed -- once -- and the processes leave
    printed = threading.Event()

    big = {}

    def emit(extra):
        if rank == 0 and not printed.is_set():
            printed.set()
            line.update(big)
            line.update(extra)
            print(json.dumps(line), flush=True)

    def bail_out():
        emit({"big_stages": f"watchdog: stopped after {args.big_timeout:.0f} s; the stages present in this line completed"})
        sys.stdout.flush()
        os._exit(0)

    dog = threading.Timer(args.big_timeout, bail_out)
    dog.daemon = True
    dog.start()
    run_big_stages(args, ctx, stream, world, rank, local, dev, peaks, big)
    dog.cancel()
    emit({})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()



# ------------------------------------------------------------------------------------------------
# cosine stage (BASELINE.json configs[2]): MovieLens-20M-shaped sketch build + all-pairs cosine top-50
# ------------------------------------------------------------------------------------------------


def _no_retries(fn):
    """a fused step that only succeeded through its second sweep (a pull-gather time-out: seconds) is a failed step as
    far as timing goes: the stage must report the other forms instead"""
    from mahout_b200 import similarity as sim

    def wrapped():
        r0 = sim.FUSED_RETRIES[0]
        out = fn()
        if sim.FUSED_RETRIES[0] != r0:
            raise RuntimeError("fused pull-gather: a peer block timed out (the result was recovered by a second sweep; "
                               "the timing of this form is void)")
        return out
    return wrapped


def _collective_steps(fn, n, dev, check_each):
    """n calls of a step that is collective across ranks (barriers inside).  A failure on one rank -- a shard that did
    not arrive through the copy engines, say -- must become a failure on all of them at the same point, or the others
    wait forever in the next collective: the ranks agree after every call (warm-up) or, so that the timed region holds
    nothing but the steps, once after the last call (a failed rank keeps calling: every call meets its peers)."""
    from mahout_b200 import similarity as sim
    out, first = None, None
    for _ in range(n):
        try:
            out = fn()
        except Exception as ex:
            first = first or ex
            out = None
        if check_each and not sim.all_ranks_ok(first is None, dev):
            raise first or RuntimeError("the step failed on another rank")
    if not check_each and not sim.all_ranks_ok(first is None, dev):
        raise first or RuntimeError("the step failed on another rank")
    return out


def _cpu_cosine_rows(bank_host, rows, k, threads):
    """oracle top-k of the given global rows, one oracle call per row spread over `threads` host threads
    (the oracle's own OpenMP loop runs over rows, so single-row calls are dealt out here)."""
    import oracle as orc
    from concurrent.futures import ThreadPoolExecutor
    orc.lib()

    def one(r):
        i1, s1, c1 = orc.bank_cosine_topk(bank_host, k, r0=r, r1=r + 1, nthreads=1)
        return i1[0], s1[0], c1[0]

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        res = list(ex.map(one, rows))
    dt = time.perf_counter() - t0
    return (np.array([r[0] for r in res]), np.array([r[1] for r in res]), np.array([r[2] for r in res]), dt)



def run_cosine_stage(ctx, stream, world, rank, local, dev, peaks, steps, warmup, dump=None):
    """One step = K2 normalise + all-gather of the 16-bit rows (N > 1) + K3 + K5 for this rank's block
    row of the N x N similarity matrix.  Returns the `cosine` object of the JSON line (rank 0); fills `dump`
    (rank 0, --dump-outputs) with the last step's top-k of DUMP_ROWS sampled rows per timed precision."""
    import torch
    import torch.distributed as dist
    import mahout_b200 as mb
    from mahout_b200 import _native as N
    from mahout_b200 import similarity as sim
    from mahout_b200 import synth
    from mahout_b200.sketch import cosine_topk_blocks, last_fallback_rows

    import bench_big as bb
    env = bb.Env(ctx, stream, world, rank, local, dev, peaks)
    plan = sim.ShardPlan(C3_ITEMS, world, rank)
    cdf = torch.from_numpy(synth.zipf_cdf(C3_ITEMS, ZIPF_S)).to(dev)
    perm = torch.from_numpy(synth.rank_permutation(C3_ITEMS, 3) - 1).to(dev)     # item rows 0..N-1
    # sketch build: every rank holds 1/G of the stream; the events travel to the owners of their items (route.cu)
    # and the owner groups them by item and updates its shard bank (group.cu)
    n_slice = C3_EVENTS // world
    bank = mb.SketchBank(plan.rows_per_shard, C3_WIDTH, C3_DEPTH, SKETCH_SEED, 1, ctx)
    build = bb.routed_build(env, plan, bank, C3_SEED, C3_EVENTS, C3_USERS, cdf, perm)
    for _ in range(2):                                  # steady state: workspaces and the router's columns exist
        bank.clear()
        b2 = bb.routed_build(env, plan, bank, C3_SEED, C3_EVENTS, C3_USERS, cdf, perm)
        if b2["route_ms"] + b2["k1_ms"] < build["route_ms"] + build["k1_ms"]:
            build = b2
    ctx.set_profiling(True)
    s_user, s_item, s_pref = synth.events_device(ctx, C3_SEED, rank * n_slice, n_slice, C3_USERS, cdf, perm)
    n_local = int(n_slice)

    ld = int(N.lib().mb200_row_ld(C3_WIDTH))
    vw = int(N.lib().mb200_valid_words(plan.rows_per_shard))
    a_rows = torch.empty((C3_DEPTH, plan.rows_per_shard, ld), dtype=torch.float16, device=dev)
    a_valid = torch.empty((C3_DEPTH, vw), dtype=torch.int32, device=dev)
    b_rows = torch.empty((world,) + tuple(a_rows.shape), dtype=torch.float16, device=dev) if world > 1 else None
    b_valid = torch.empty((world,) + tuple(a_valid.shape), dtype=torch.int32, device=dev) if world > 1 else None
    a_cnt = bank.counters_tensor()
    b_id = (world, 1) if world > 1 else (1, plan.rows_per_shard)
    out = {}

    dbg = os.environ.get("MB200_BENCH_DEBUG") is not None
    outs = {pr: (torch.empty((plan.rows_per_shard, C3_K), dtype=torch.int64, device=dev),
                 torch.empty((plan.rows_per_shard, C3_K), dtype=torch.float64, device=dev),
                 torch.empty((plan.rows_per_shard,), dtype=torch.int32, device=dev)) for pr in ("tensor", "certified", "rescored")}

    def step(precision, b_cnt=None):
        t_dbg = time.perf_counter()
        N.check(N.lib().mb200_bank_normalize(bank.handle, N.DTYPE_F16, C.c_void_p(a_rows.data_ptr()),
                                             C.c_void_p(a_valid.data_ptr())), ctx.handle)
        if dbg:
            print(f"[bench debug] {precision}: K2 call {1e3 * (time.perf_counter() - t_dbg):.2f} ms", file=sys.stderr)
        if world > 1:
            dist.all_gather_into_tensor(b_rows.view(-1, plan.rows_per_shard, ld), a_rows)
            dist.all_gather_into_tensor(b_valid.view(-1, vw), a_valid)
            br, bv = b_rows, b_valid
        else:
            br, bv = a_rows.unsqueeze(0), a_valid.unsqueeze(0)
        # outputs are allocated once: torch.empty inside the loop falls through to cudaMalloc on this non-default
        # stream, which costs milliseconds on a process that holds tens of GB (measured: 5 - 30 ms per step)
        return cosine_topk_blocks(ctx, a_rows, a_valid, br, bv, C3_DEPTH, C3_WIDTH, C3_K, a_id=(world, rank),
                                  b_id=b_id, dtype="f16", precision=precision, out=outs[precision],
                                  a_counters=a_cnt if precision != "tensor" else None, b_counters=b_cnt if precision != "tensor" else None)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        step("tensor")
    barrier()
    ctx.reset_profile()
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        idx, s, cnt = step("tensor")
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1) / steps
    k2_ms, k2_n = ctx.kernel_time(N.K_NORMALIZE)
    k3_ms, k3_n = ctx.kernel_time(N.K_COSINE)
    k5_ms, k5_n = ctx.kernel_time(N.K_RESCORE)
    launches = ctx.launch_count() - launches0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # pipelined variant (N > 1): chunked all-gather on a side stream overlapped with K3 pushes
    piped_ms, piped_equal = None, None
    if world > 1:
        be = sim.GpuShardBackend(ctx)
        be.bank = bank
        chunk_rows = (plan.rows_per_shard + C3_CHUNKS * 256 - 1) // (C3_CHUNKS * 256) * 256

        def step_piped():
            N.check(N.lib().mb200_bank_normalize(bank.handle, N.DTYPE_F16, C.c_void_p(a_rows.data_ptr()),
                                                 C.c_void_p(a_valid.data_ptr())), ctx.handle)
            return sim.pipelined_cosine(be, plan, a_rows, a_valid, C3_K, None, "f16", "tensor", None,
                                        chunk_rows, None)

        for _ in range(warmup):
            step_piped()
        barrier()
        e0.record(stream)
        for _ in range(steps):
            pidx, ps, pcnt = step_piped()
        e1.record(stream)
        barrier()
        piped_ms = e0.elapsed_time(e1) / steps
        t = torch.tensor([piped_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        piped_ms = float(t.item())
        piped_equal = bool(torch.equal(pidx, idx) and torch.equal(ps, s) and torch.equal(pcnt, cnt))
    # fused variant (N > 1): the shards are pulled over NVLink by the copy engines while one K3 launch
    # waits block by block on their arrival flags
    fused_ms, fused_equal, fused_err, fk3_ms, fk3_n, peers, cert_fallback = None, None, None, 0.0, 0, None, None
    if world > 1:
        try:
            peers = sim.PeerRows(ctx, plan, C3_DEPTH, C3_WIDTH)
            fout = (torch.empty_like(idx), torch.empty_like(s), torch.empty_like(cnt))

            def step_fused():
                N.check(N.lib().mb200_bank_normalize(bank.handle, N.DTYPE_F16, C.c_void_p(peers.rows.data_ptr()),
                                                     C.c_void_p(peers.valid.data_ptr())), ctx.handle)
                return sim.fused_gather_cosine(be, plan, peers, C3_K, None, "f16", "tensor", out=fout)

            _collective_steps(_no_retries(step_fused), warmup, dev, True)
            barrier()
            ctx.reset_profile()
            e0.record(stream)
            fidx, fs, fcnt = _collective_steps(_no_retries(step_fused), steps, dev, False)
            e1.record(stream)
            barrier()
            fused_ms = e0.elapsed_time(e1) / steps
            t = torch.tensor([fused_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            fused_ms = float(t.item())
            fused_equal = bool(torch.equal(fidx, idx) and torch.equal(fs, s) and torch.equal(fcnt, cnt))
            fk3_ms, fk3_n = ctx.kernel_time(N.K_COSINE)
        except Exception as ex:            # e.g. CUDA IPC not permitted on this box: the other forms still stand
            fused_ms, fused_equal, fused_err = None, None, repr(ex)[:200]
            peers = None
    # certified precision (exact top-k sets, tensor-core values): the north star's contract.  N = 1: local
    # counters; N > 1: fused pull-gather + the peers' banks mapped over NVLink (no counter gather)
    cert_ms, cidx, ccnt, cert_kernels = None, None, None, None
    try:
        if world == 1:
            cstep = lambda: step("certified", a_cnt)
        elif peers is not None:
            blocks = peers.map_counters(bank)

            def cstep():
                N.check(N.lib().mb200_bank_normalize(bank.handle, N.DTYPE_F16, C.c_void_p(peers.rows.data_ptr()),
                                                     C.c_void_p(peers.valid.data_ptr())), ctx.handle)
                return sim.fused_gather_cosine(be, plan, peers, C3_K, None, "f16", "certified", a_counters=a_cnt,
                                               counter_blocks=blocks, out=outs["certified"])
        else:
            cstep = None
        if cstep is not None:
            _collective_steps(_no_retries(cstep), warmup, dev, True)
            barrier()
            ctx.reset_profile()
            t_c0 = time.perf_counter()
            e0.record(stream)
            cidx, cs, ccnt = _collective_steps(_no_retries(cstep), steps, dev, False)
            e1.record(stream)
            barrier()
            cert_wall_ms = (time.perf_counter() - t_c0) * 1e3 / steps
            cert_ms = e0.elapsed_time(e1) / steps
            cert_kernels = {name: ctx.kernel_time(kid)[0] / steps for name, kid in
                            (("K2_normalize", N.K_NORMALIZE), ("K3_cosine_topk", N.K_COSINE), ("K5_merge_certify", N.K_RESCORE))}
            cert_kernels["host_wall_ms_per_step"] = cert_wall_ms
            if world > 1:
                t = torch.tensor([cert_ms], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                cert_ms = float(t.item())
            cert_fallback = last_fallback_rows(ctx)
    except Exception as ex:
        cert_ms, fused_err = None, (fused_err or "") + " certified: " + repr(ex)[:200]
    if world > 1 and peers is not None:
        peers.close()
    # exact (re-scored) variant, timed once
    b_cnt = a_cnt
    if world > 1:
        b_cnt = torch.empty((world,) + tuple(a_cnt.shape), dtype=a_cnt.dtype, device=dev)
        dist.all_gather_into_tensor(b_cnt.view(-1, C3_DEPTH, C3_WIDTH), a_cnt)
    step("rescored", b_cnt)                 # untimed: first-touch allocation of the re-score workspaces
    barrier()
    ctx.reset_profile()
    r_reps = max(1, min(steps, 3))
    e0.record(stream)
    for _ in range(r_reps):
        ridx, rs, rcnt = step("rescored", b_cnt)
    e1.record(stream)
    barrier()
    rescored_ms = e0.elapsed_time(e1) / r_reps
    if world > 1:
        t = torch.tensor([rescored_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        rescored_ms = float(t.item())
    r5_ms, r5_n = ctx.kernel_time(N.K_RESCORE)
    r5_ms /= max(r5_n, 1)
    fallback = last_fallback_rows(ctx)
    ctx.set_profiling(False)

    # ---- end to end: this rank's events start in pinned HOST memory, its rows' top-k ends in host memory;
    # bank allocation + zero fill, H2D staging, K1, K2, (all-gathers), K3, K5 and the D2H are all inside
    h_row, h_user, h_pref = (t.cpu().pin_memory() for t in (s_item, s_user, s_pref))
    del s_user, s_item, s_pref
    e2e_router = None
    if world > 1:
        probe = sim.EventRouter.__new__(sim.EventRouter)
        probe.ctx, probe.plan, probe.group = ctx, plan, None
        _, mat = sim.EventRouter.counts(probe, h_row.to(dev))
        e2e_router = sim.EventRouter(ctx, plan, int(mat.sum(axis=0).max()))

    def e2e_step(precision):
        eb = mb.SketchBank(plan.rows_per_shard, C3_WIDTH, C3_DEPTH, SKETCH_SEED, 1, ctx)
        try:
            if world == 1:
                eb.update(h_row.numpy(), h_user.numpy(), h_pref.numpy())
                return eb.cosine_topk(C3_K, None, True, "f16", precision)          # numpy (host) outputs
            # this rank's slice of the stream: H2D, routed to the owners over NVLink, grouped K1 on the owner
            d_ev = [t.to(dev, non_blocking=True) for t in (h_row, h_user, h_pref)]
            lrow, luser, lpref, _ = sim.route_events_device(ctx, plan, *d_ev, router=e2e_router)
            eb.update(lrow, luser, lpref)
            N.check(N.lib().mb200_bank_normalize(eb.handle, N.DTYPE_F16, C.c_void_p(a_rows.data_ptr()),
                                                 C.c_void_p(a_valid.data_ptr())), ctx.handle)
            dist.all_gather_into_tensor(b_rows.view(-1, plan.rows_per_shard, ld), a_rows)
            dist.all_gather_into_tensor(b_valid.view(-1, vw), a_valid)
            ec = eb.counters_tensor()
            if precision == "rescored":
                dist.all_gather_into_tensor(b_cnt.view(-1, C3_DEPTH, C3_WIDTH), ec)
            r = cosine_topk_blocks(ctx, a_rows, a_valid, b_rows, b_valid, C3_DEPTH, C3_WIDTH, C3_K,
                                   a_id=(world, rank), b_id=b_id, dtype="f16", precision=precision,
                                   a_counters=ec if precision == "rescored" else None,
                                   b_counters=b_cnt if precision == "rescored" else None)
            return tuple(t.cpu() for t in r)
        finally:
            eb.close()

    e2e = {}
    for precision in ("rescored", "tensor"):
        e2e_step(precision)
        best = None
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            e2e_step(precision)
            barrier()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            best = dt if best is None else min(best, dt)
        e2e[precision] = best

    if rank == 0:
        import oracle as orc
        pairs = float(C3_ITEMS) ** 2
        flops_rank = 2.0 * C3_DEPTH * plan.rows_per_shard * (plan.rows_per_shard * world) * ld
        k3_s = k3_ms / max(k3_n, 1) * 1e-3
        achieved = flops_rank / k3_s / 1e12
        # parity + CPU baseline on sampled rows of shard 0 (the oracle needs the whole bank)
        if world > 1:
            full = b_cnt.cpu().numpy()                                           # [G, E_loc, d, w] quanta
            bank_host = np.zeros((plan.rows_per_shard * world, C3_DEPTH, C3_WIDTH))
            for g in range(world):
                bank_host[g::world] = full[g] * 0.5
        else:
            bank_host = bank.read()
        threads = _host_threads()
        rows_chk = int(min(plan.rows_per_shard, threads * (24 if world == 1 else 4)))   # ~0.5 s per row and thread
        oi, osim, oc, cpu_s = _cpu_cosine_rows(bank_host, [l * world for l in range(rows_chk)], C3_K, threads)
        gi, gs, gc = ridx[:rows_chk].cpu().numpy(), rs[:rows_chk].cpu().numpy(), rcnt[:rows_chk].cpu().numpy()
        ti, ts, tc = idx[:rows_chk].cpu().numpy(), s[:rows_chk].cpu().numpy(), cnt[:rows_chk].cpu().numpy()
        exact_equal = bool((gi == oi).all() and (gc == oc).all() and gs.tobytes() == osim.tobytes())
        cert_sets = None
        if cidx is not None:
            ci_, cc_ = cidx[:rows_chk].cpu().numpy(), ccnt[:rows_chk].cpu().numpy()
            cert_sets = bool((cc_ == oc).all() and all(set(ci_[l, :cc_[l]].tolist()) == set(oi[l, :oc[l]].tolist())
                                                      for l in range(rows_chk)))
        # tensor precision: value of every returned pair vs the oracle's FP64 cosine of that pair
        max_rel, overlap, tot = 0.0, 0, 0
        for l in range(rows_chk):
            o = dict(zip(oi[l, :oc[l]].tolist(), osim[l, :oc[l]].tolist()))
            for c, v in zip(ti[l, :tc[l]].tolist(), ts[l, :tc[l]].tolist()):
                if c in o:
                    overlap += 1
                    max_rel = max(max_rel, abs(v - o[c]) / abs(o[c]))
            tot += int(oc[l])
        out = {
            "metric": "item_pair_cosine_sims_per_sec",
            # headline: certified precision (exact top-k sets, values <= 1e-3) when it ran, else tensor precision
            "value": pairs / ((cert_ms or min(ms, piped_ms or ms, fused_ms or ms)) * 1e-3),
            "unit": "pairs/s", "precision_of_value": "certified" if cert_ms else "tensor",
            "ms_per_step": cert_ms or min(ms, piped_ms or ms, fused_ms or ms),
            "ms_per_step_certified": cert_ms, "certified_fallback_rows": cert_fallback,
            "certified_kernels_ms_per_step": cert_kernels,
            "ms_per_step_tensor": min(ms, piped_ms or ms, fused_ms or ms), "ms_per_step_allgather_then_k3": ms,
            "ms_per_step_pipelined": piped_ms, "pipelined_equals_one_shot": piped_equal,
            "ms_per_step_fused_pull_gather": fused_ms, "fused_equals_one_shot": fused_equal,
            "fused_k3_ms_per_launch": (fk3_ms / max(fk3_n, 1)) if (world > 1 and fk3_n) else None,
            "fused_error": fused_err,
            "pipelined_chunk_rows": chunk_rows if world > 1 else None, "steps": steps, "warmup": warmup, "n_gpus": world, "scaling": "strong",
            "dtype": "f16 rows (x/||x|| * 2^12), f32 accumulate in TMEM; re-score in exact int64/f64",
            "config": {"workload": "configs[2]: MovieLens-20M-shaped synthetic (138493 users x 26744 items, 2e7 "
                                   "Zipf(1.1) events), sketch d=4 x W=4096, cosine top-50 per item",
                       "precision_timed": "certified (value), tensor (roofline, forms)", "items": C3_ITEMS,
                       "l2": "inputs_exceed_l2 (0.88 GB of FP16 rows, 3.5 GB of counters per step)", "depth": C3_DEPTH, "width": C3_WIDTH,
                       "k": C3_K, "parallelism": f"item-hash sharded x{world} + all-gather of f16 rows"
                       if world > 1 else "single GPU"},
            "kernels_ms_per_step": {"K2_normalize": k2_ms / max(k2_n, 1), "K3_cosine_topk": k3_ms / max(k3_n, 1),
                                    "K5_merge": k5_ms / max(k5_n, 1)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "k_cosine<256,1,true>", "achieved": achieved,
                         "peak": peaks["bf16"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16"],
                         "frac_of_burst_peak": achieved / peaks["bf16_burst"], "peak_source": peaks["source"],
                         "flops_per_launch": flops_rank, "kernel_ms_per_launch": k3_s * 1e3,
                         # ncu --set full of this kernel on this workload at 1 GPU
                         # (profiles/r1_k_cosine_v4_ncu.txt): dram read 64.33 GB + write 1.01 GB -- the A blocks
                         # are re-read for every B tile (DESIGN.md section 3, "Scheduling")
                         "traffic": 65.34e9 if world == 1 else None},
            "e2e": {"value": pairs / e2e["rescored"], "unit": "pairs/s", "ms_per_job": e2e["rescored"] * 1e3,
                    "h2d_bytes_per_step": 20 * n_local, "d2h_bytes_per_step": plan.rows_per_shard * (C3_K * 16 + 4),
                    "tensor_precision": {"value": pairs / e2e["tensor"], "ms_per_job": e2e["tensor"] * 1e3},
                    "sample": "whole job per rank: SketchBank(...) + update(host events, pinned) + cosine_topk -> host "
                              "arrays (API default precision = rescored, bit-equal to the reference); best of 3"},
            "rescored": {"ms_per_step": rescored_ms, "K5_merge_rescore_ms": r5_ms, "fallback_rows": int(fallback),
                         "pairs_per_s": pairs / (rescored_ms * 1e-3)},
            "sketch_build": dict(build, kernel="k_group_* + k_update_grouped (bank mode)",
                                 model_bytes_per_event=BANK_BYTES_PER_EVENT),
            "parity": {"rows_checked": rows_chk, "rescored_topk_and_sims_equal_oracle": exact_equal,
                       "certified_topk_sets_equal_oracle": cert_sets,
                       "tensor_max_rel_err": max_rel, "tensor_topk_overlap": overlap / max(tot, 1)},
            "cpu_baseline": {"value": rows_chk * C3_ITEMS / cpu_s, "unit": "pairs/s", "cores": threads, "kind": "port",
                             "sample": f"{rows_chk} rows x all {C3_ITEMS} columns, {cpu_s:.1f} s; oracle/ C port of "
                                       "DoubleCountMinSketch.cosine + top-k"},
        }
    if dump is not None:
        local_rows = np.arange(plan.local_count())
        pick = np.sort(np.random.default_rng(C3_SEED).choice(local_rows, min(DUMP_ROWS, local_rows.size), replace=False))
        dump["cosine_rows"] = plan.global_row(pick)
        sel = torch.from_numpy(pick).to(dev)
        results = {"tensor": (idx, s, cnt), "rescored": (ridx, rs, rcnt)}
        if cidx is not None:
            results["certified"] = (cidx, cs, ccnt)
        for precision, res in results.items():
            for part, t in zip(("idx", "sim", "cnt"), res):
                dump[f"cosine_{precision}_{part}"] = t[sel].cpu().numpy()
    if e2e_router is not None:
        e2e_router.close()
    bank.close()
    return out


def run_big_stages(args, ctx, stream, world, rank, local, dev, peaks, out):
    """BASELINE.json configs[3] and configs[4] (bench_big.py): at 8 GPUs by default, at other N when asked for with
    --big on (sizes then come from the --c4-* / --c5-* flags).  Fills `out` ({"config4": ..., "config5": ...}, rank 0)
    stage by stage, so that whatever is complete when the watchdog fires is still reported; a stage is skipped when
    the time already spent leaves no room for it (--big-budget)."""
    on = args.big == "on" or (args.big == "auto" and world == 8)
    if not on:
        return
    import torch
    import bench_big as bb
    env = bb.Env(ctx, stream, world, rank, local, dev, peaks)

    def room(name, need_s):
        used = env.elapsed()
        if used + need_s > args.big_budget:
            env.log(f"{name}: skipped ({used:.0f} s used of {args.big_budget:.0f} s, needs ~{need_s:.0f} s)")
            if rank == 0:
                out.setdefault("skipped_stages", []).append({"stage": name, "seconds_used": used, "seconds_needed": need_s})
            return False
        return True

    def guarded(name, fn):
        try:
            return fn()
        except Exception as ex:                      # a failed stage must not lose the rest of the line
            env.log(f"{name}: FAILED {ex!r}")
            torch.cuda.synchronize(dev)
            return {"name": name, "error": repr(ex)[:400]}

    c4 = "configs[3]: 1M-item all-pairs sketch cosine (width 4096), fused top-100 epilogue, item-hash sharded; " \
         "sketch rows built from config-3-style Zipf(1.1) events routed to their owners"
    if args.c4_items > 0:
        r = guarded("config4_d1", lambda: bb.big_cosine(env, "config4_d1", c4, int(args.c4_items), 5_000_000, args.c4_events, 1.1, 1,
                                                        4096, 100, "fused", int(args.c4_check_rows), 20240004))
        if rank == 0:
            out["config4"] = r
    if args.c5_events > 0 and room("config5a_skew_update", 15):
        r = guarded("config5a", lambda: bb.skew_update(env, args.c5_events, 10_000_000, 1.5, DEPTH, WIDTH,
                                                       max(1, min(args.steps, 3)), 1, 20240005))
        if rank == 0:
            out.setdefault("config5", {})["skew_update"] = r
    if args.c5_items > 0 and room("config5b_streamed_cosine", 150):
        r = guarded("config5b", lambda: bb.big_cosine(
            env, "config5b_streamed_cosine", "configs[4]b (scaled): 10M-item cosine top-100 at "
            f"{int(args.c5_items)} items, width 4096, depth 1, in the STREAMED form -- row chunks of every shard "
            "gathered into two staging buffers while K3 consumes them; the gathered operand never exists",
            int(args.c5_items), 5_000_000, args.c5_cos_events, 1.1, 1, 4096, 100, "pipelined", int(args.c5_check_rows),
            20240006, chunk_rows=int(args.c5_chunk_rows), warmup=0))
        if rank == 0:
            out.setdefault("config5", {})["streamed_cosine"] = r
            out["config5"]["scale_note"] = ("configs[4] asks for 1e10 events and 1e7 items: the update leg runs at full size; "
                                            "the cosine leg is scaled (2*N^2*W FLOP: 85 s at 1e7 items on 8 GPUs) -- at 1e7 x "
                                            "4096 the gathered FP16 operand would be 82 GB per depth row")
    if args.c4_d4 and args.c4_items > 0 and room("config4_d4", 90):
        r = guarded("config4_d4", lambda: bb.big_cosine(env, "config4_d4", c4, int(args.c4_items), 5_000_000, args.c4_events, 1.1, 4,
                                                        4096, 100, "fused", int(args.c4_check_rows_d4), 20240004))
        if rank == 0 and isinstance(out.get("config4"), dict):
            out["config4"]["depth4"] = r
    env.log("big stages done")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--events", type=float, default=1e9, help="events per step per GPU")
    ap.add_argument("--e2e-events", type=float, default=float(1 << 27))
    ap.add_argument("--no-cosine", action="store_true", help="skip the secondary cosine-stage measurement")
    ap.add_argument("--big", default="auto", choices=["auto", "on", "off"],
                    help="configs[3] / configs[4] stages (auto: at 8 GPUs)")
    ap.add_argument("--big-timeout", type=float, default=600.0, help="watchdog of the configs[3] / configs[4] stages")
    ap.add_argument("--big-budget", type=float, default=420.0, help="no new big stage starts once this many seconds of them are spent")
    ap.add_argument("--c4-items", type=float, default=1e6)
    ap.add_argument("--c4-events", type=float, default=2e9)
    ap.add_argument("--c4-check-rows", type=float, default=4096)
    ap.add_argument("--c4-check-rows-d4", type=float, default=128)
    ap.add_argument("--c4-d4", type=int, default=1, help="also run configs[3] at depth 4")
    ap.add_argument("--c5-events", type=float, default=1e10)
    ap.add_argument("--c5-items", type=float, default=4e6)
    ap.add_argument("--c5-cos-events", type=float, default=8e9)
    ap.add_argument("--c5-check-rows", type=float, default=512)
    ap.add_argument("--c5-chunk-rows", type=float, default=8192)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed steps' outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours (the reference arm times a calibrated prefix of the stream)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
