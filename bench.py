#!/usr/bin/env python
"""bench.py — placement decisions/sec on the BASELINE.json headline workload (1M models x 10k instances, C3).

One "step" = one pass of the hot path over one batch: a reaper-style sweep of B = n_models getNext decisions against one
snapshot epoch (SURVEY.md §8d).  Reported on one JSON line:
  value     decisions/s with the batch already resident in HBM (CUDA events around the scoring kernel, max over ranks)
  e2e       the same batch through mmp_place_batch with pinned HOST buffers (H2D + kernel + D2H inside the timed region)
  roofline  algorithmic bytes (1312 B/decision + 80 B/instance, SURVEY.md §8d) / measured kernel time vs the measured
            HBM copy peak in MEASURED_PEAKS.json
  cpu_baseline  the oracle (C++ restatement of the reference's Java path; the JVM cannot run here) on the host cores
`--impl reference` times only that CPU path.  N > 1 (torchrun): the registry is sharded by model across ranks (each rank
places its slice against a replicated instance table; no data-path collective), so total work is fixed: "strong".
`--dump-outputs DIR` writes what the last timed step computed as .npy files; the inputs are seeded, so two builds can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIG = os.environ.get("BENCH_CONFIG", "C3")  # C3 = the configuration BASELINE.json's metric is quoted on; C2 / C5 / C4: the others
_DEFAULT_SIZES = {"C2": (100_000, 1_000), "C3": (1_000_000, 10_000), "C5": (1_000_000, 10_000), "C4": (500_000, 2_500)}
N_MODELS = int(os.environ.get("BENCH_MODELS", _DEFAULT_SIZES.get(CONFIG, (1_000_000, 10_000))[0]))
N_INSTANCES = int(os.environ.get("BENCH_INSTANCES", _DEFAULT_SIZES.get(CONFIG, (1_000_000, 10_000))[1]))
SEED = {"C2": 2, "C3": 3, "C4": 4, "C5": 5}.get(CONFIG, 3)
METRIC = "placement decisions/sec at 1M models x 10k instances"
WORKLOADS = {"C2": "Zipf request rates, no type constraints", "C3": "mixed type constraints",
             "C5": "adversarial 95%-full capacity bin-packing, heavy type-constraint masks", "C4": "churn"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dump_dir, arrays: dict, rank: int = 0, world: int = 1):
    """--dump-outputs: every field of every structured array as <array>_<field>.npy in float64 (int64 values past 2**53
    round), so that two builds can be compared output for output on the same seeded inputs.  When all of it would exceed
    DUMP_LIMIT_BYTES, every array is cut to a fixed, seeded sample of its rows (<array>_index.npy holds the row numbers).
    With several ranks each writes its own slice under rank<r>/."""
    if not dump_dir:
        return
    if world > 1:
        dump_dir = os.path.join(dump_dir, f"rank{rank}")
    os.makedirs(dump_dir, exist_ok=True)
    full = sum(len(a) * len(a.dtype.names) * 8 for a in arrays.values())
    frac = 1.0 if full <= DUMP_LIMIT_BYTES else \
        DUMP_LIMIT_BYTES / sum(len(a) * (len(a.dtype.names) + 1) * 8 for a in arrays.values())
    for name, a in arrays.items():
        if frac < 1.0:
            idx = np.sort(np.random.default_rng(12345).choice(len(a), int(len(a) * frac), replace=False))
            np.save(os.path.join(dump_dir, f"{name}_index.npy"), idx.astype(np.float64))
            a = a[idx]
        for f in a.dtype.names:
            np.save(os.path.join(dump_dir, f"{name}_{f}.npy"), np.ascontiguousarray(a[f], dtype=np.float64))


def bytes_per_decision(row_words: int) -> int:
    """SURVEY.md §8d: exclusion-bitmap row + 24 B model row + 8 B result (1312 B at 10k instances, 1280 B padded row)."""
    return row_words * 4 + 24 + 8


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples = []
        self.stop_flag = threading.Event()
        self.proc = None
        self.t_mark = None  # samples taken before mark() (warm-up) are dropped
        self.stamps = []

    def mark(self):
        self.t_mark = time.perf_counter()

    def run(self):
        # NVML in-process (a query takes tens of microseconds: the timed region of this bench is a few milliseconds, which the
        # 100 ms period of `nvidia-smi -lms` cannot sample); nvidia-smi as the fall-back
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
            while not self.stop_flag.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                except Exception:
                    r = 0
                self.samples.append([str(sm), str(mx), "0"] + ["Active" if r & bit else "Not Active" for _, bit in names])
                self.stamps.append(time.perf_counter())
                time.sleep(0.001)
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            for line in self.proc.stdout:
                if self.stop_flag.is_set():
                    break
                parts = [p.strip() for p in line.split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
                    self.stamps.append(time.perf_counter())
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for p, ts in zip(list(self.samples), list(self.stamps)):
            if self.t_mark is not None and ts < self.t_mark:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy kernel)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def scoring_kernel() -> str:
    """The kernel mmp_place_batch_device launches for an untraced batch on an unsharded fleet: k_place_direct unless
    MMP_KERNEL selects the streaming kernel (lanes) or the cooperative tiles (tile)."""
    k = os.environ.get("MMP_KERNEL", "direct")
    return {"lanes": "k_place_lanes", "tile": "k_place"}.get(k, "k_place_direct")


def captured_traffic(batch: int):
    """dram__bytes_read + dram__bytes_write of one launch of the scoring kernel from the committed `ncu --set full` capture of
    this configuration (profiles/r02_ncu_<kernel>_<config>.json, written by tools/ncu_summary.py), scaled per decision when
    the capture was taken on another batch size (the traffic is proportional to the number of decisions)."""
    for name in (f"r02_ncu_{scoring_kernel()}_{CONFIG.lower()}.json",):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            nd = int(d.get("n_decisions") or 0)
            if nd > 0:
                return float(d["dram_bytes_per_launch"]) * batch / nd, f"profiles/{name.replace('.json', '.txt')}"
        except Exception:
            pass
    return None, None


def build_oracle(fl):
    """CPU baseline / checker only."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    return helpers, helpers.oracle_from_synth(fl)


def cpu_leg(fl, sd_all, budget_s: float, chunk: int, threads: int, dense: bool = False):
    """Time the oracle's getNext on chunks of the same workload for about budget_s seconds (dense: CPU mode (ii))."""
    helpers, oracle = build_oracle(fl)
    from modelmesh_b200.synth import SynthDecisions
    done, t_total, results = 0, 0.0, []
    n = len(sd_all.dec)
    pos = 0
    while t_total < budget_s and pos < n:
        hi = min(n, pos + chunk)
        sd = SynthDecisions(sd_all.dec[pos:hi], sd_all.fresh, sd_all.extra)
        od, off, idx = helpers.oracle_inputs_fast(fl, sd)
        od["decision_id"] = np.arange(pos, hi, dtype=np.uint64)
        t0 = time.perf_counter()
        res = oracle.get_next_batch(od, fl.type_names, off, idx, fl.now_ms, SEED, threads=threads, dense=dense)
        t_total += time.perf_counter() - t0
        results.append((pos, hi, res))
        done += hi - pos
        pos = hi
    return done, t_total, results


def run_reference(args, rank: int, world: int):
    """The reference's own CPU path (C++ restatement: no JVM in the image) on the host cores, on the SAME step as the repo's
    arm: one reaper-style sweep of N_MODELS getNext decisions per step, all host threads; CPU mode (ii) beside it."""
    if rank != 0:
        return
    if CONFIG == "C4":
        return run_reference_churn(args)
    from modelmesh_b200.synth import make_decisions, make_fleet
    fl = make_fleet(CONFIG, N_MODELS, N_INSTANCES, SEED)
    sd = make_decisions(fl, N_MODELS, SEED, sweep=True, plain=True)
    threads = host_threads()
    helpers, oracle = build_oracle(fl)
    od, off, idx = helpers.oracle_inputs_fast(fl, sd)
    times, dense_times = [], []
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = oracle.get_next_batch(od, fl.type_names, off, idx, fl.now_ms, SEED, threads=threads)
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            times.append(dt)
    dump_outputs(args.dump_outputs, {"decision": res[["target", "n_candidates"]]})
    for step in range(min(3, args.steps)):
        t0 = time.perf_counter()
        oracle.get_next_batch(od, fl.type_names, off, idx, fl.now_ms, SEED, threads=threads, dense=True)
        dense_times.append(time.perf_counter() - t0)
    tot = sum(times)
    value = N_MODELS * len(times) / tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * tot / len(times), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(world=max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "decisions/s", "cores": threads, "kind": "port",
                         "sample": f"the whole step: {N_MODELS} decisions x {len(times)} steps, C++ restatement of "
                                   f"CacheMissForwardingLB.getNext in its reference shape (ordered set walk); the Java reference cannot run: no JDK",
                         "dense": {"value": N_MODELS * len(dense_times) / sum(dense_times), "unit": "decisions/s", "cores": threads,
                                   "sample": f"{len(dense_times)} steps, CPU mode (ii) of BASELINE.md: entries through a rank-ordered array"}},
        "e2e": {"value": value, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=OUT, flush=True)


def workload_config(world: int):
    """The `config` object of the JSON line: a pure function of the configuration and the world size, so that the repo's arm
    and the --impl reference arm print the same one."""
    from modelmesh_b200.sharding import shard_range
    row_words = ((N_INSTANCES + 31) // 32 + 31) // 32 * 32
    lo, hi = shard_range(0, world, N_MODELS)
    gb = (hi - lo) * row_words * 4 / 1e9
    return {"workload": f"{CONFIG} {N_MODELS} models x {N_INSTANCES} instances, {WORKLOADS.get(CONFIG, '')}, one reaper-style sweep of "
                        f"{N_MODELS} getNext decisions per step",
            "batch": N_MODELS,
            "sharding": "registry sharded by model across ranks, instance table replicated" if world > 1 else "single GPU",
            "l2": ("inputs larger than L2 (exclusion bitmap %.2f GB per rank streamed every step)" % gb if gb > 0.2 else
                   "L2 flushed between timed steps (mmp_flush_l2): the %.1f MB bitmap would otherwise stay resident" % (gb * 1e3))}


CHURN_METRIC = "churn events/sec over a 500k-model fleet (placement + admission + LRU + eviction + republish + commit per 2 s window)"
CHURN_EVENTS = int(os.environ.get("BENCH_CHURN_EVENTS", 20_000))  # 10k events/s x 2 s


def _churn_oracle(w):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    from oracle import binding as ob
    fl = w.fleet
    o = helpers.oracle_from_synth(fl)
    models = np.zeros(fl.n_models, dtype=ob.SIM_MODEL)
    models["last_used"], models["type_idx"], models["size_units"] = fl.model_last_used, fl.model_type, fl.model_size
    sim = ob.OracleSim(o, models, fl.type_names, fl.edge_off, fl.edge_inst, fl.n_loaded, w.capacity, w.load_timeout_ms, fl.now_ms - 60_000)
    order = np.argsort(w.seed_instance, kind="stable")
    bounds = np.searchsorted(w.seed_instance[order], np.arange(fl.n_instances + 1))
    for i in range(fl.n_instances):
        sel = order[bounds[i]:bounds[i + 1]]
        if len(sel):
            sim.seed(i, w.seed_model[sel], w.seed_last_used[sel], w.seed_weight[sel], w.seed_load_ts[sel], fl.now_ms)
    return o, sim


def churn_config():
    return {"workload": f"C4 {N_MODELS} models x {N_INSTANCES} instances at 97 % fill, Poisson trace of {CHURN_EVENTS} events per 2 s window "
                        f"(70 % requests of loaded models (Zipf), 25 % of unloaded ones, 5 % removals), one window per step, commit every window",
            "batch": CHURN_EVENTS, "sharding": "single GPU",
            "l2": "L2 flushed between timed windows (mmp_flush_l2): the fleet's working set is smaller than L2"}


def run_reference_churn(args):
    from modelmesh_b200.synth import make_churn
    w = make_churn(N_MODELS, N_INSTANCES, SEED)
    fl = w.fleet
    o, sim = _churn_oracle(w)
    times = []
    for ep in range(args.warmup + args.steps):
        ev = w.events(ep, CHURN_EVENTS, SEED)
        now0 = fl.now_ms + ep * w.window_ms
        t0 = time.perf_counter()
        dec, evi, rows, _, _ = sim.step(ev, now0, now0 + w.window_ms, 400 + ep)
        if ep >= args.warmup:
            times.append(time.perf_counter() - t0)
    dump_outputs(args.dump_outputs, {"decision": dec, "eviction": evi, "instance": rows})
    value = CHURN_EVENTS * len(times) / sum(times)
    print(json.dumps({
        "impl": "reference", "metric": CHURN_METRIC, "value": value, "unit": "events/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * sum(times) / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": churn_config(),
        "cpu_baseline": {"value": value, "unit": "events/s", "cores": 1, "kind": "port",
                         "sample": f"{len(times)} windows of {CHURN_EVENTS} events, the oracle's closed loop (oracle/mm_sim.inc), one thread"},
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), file=OUT, flush=True)


def run_churn(args, rank: int, world: int, local_rank: int):
    """BASELINE.json configs[3]: the closed loop on one GPU, one republish window per step."""
    import torch
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        if rank != 0:  # the churn configuration is a single-GPU one: the other ranks wait
            dist.barrier()
            dist.destroy_process_group()
            return
    import ctypes as C
    from modelmesh_b200 import _lib
    from modelmesh_b200.fleet import Fleet
    from modelmesh_b200.synth import load_into_fleet, make_churn
    lib = _lib.load_product()
    w = make_churn(N_MODELS, N_INSTANCES, SEED)
    fl = w.fleet
    s = Fleet(fl.min_space_units, fl.min_churn_age_ms, fl.default_model_size_units, fl.n_instances, fl.n_models, device=local_rank, lib=lib)
    load_into_fleet(fl, s)
    s.churn_init(w.load_timeout_ms, fl.now_ms - 60_000, 512)
    s.churn_seed(w.seed_instance, w.seed_model, w.seed_last_used, w.seed_weight, w.seed_load_ts, fl.now_ms)
    check = not args.no_cpu
    if check:
        o, sim = _churn_oracle(w)
    sampler = ClockSampler(local_rank)
    launches0 = 0
    dev_ms, wall_ms, phases, mism, cpu_s = [], [], [], 0, []
    n_dec = n_evict = n_lru = n_pub = 0
    for ep in range(args.warmup + args.steps):
        if ep == 0:
            sampler.start()
            time.sleep(0.05)
        if ep == args.warmup:
            launches0 = s.kernel_launches()
            sampler.mark()
        ev = w.events(ep, CHURN_EVENTS, SEED)
        now0 = fl.now_ms + ep * w.window_ms
        s._ck(lib.mmp_flush_l2(s.h))
        t0 = time.perf_counter()
        dec, evi, rows, rep = s.churn_step(ev, now0, now0 + w.window_ms, 400 + ep)
        dt = time.perf_counter() - t0
        if check:  # every window against the oracle's closed loop: decisions, statuses, evictions, republished rows
            t1 = time.perf_counter()
            dec_o, evi_o, rows_o, npub_o, carry_o = sim.step(ev, now0, now0 + w.window_ms, 400 + ep)
            if ep >= args.warmup:
                cpu_s.append(time.perf_counter() - t1)
            keep = dec_o["status"] != 7
            bad = len(dec) != len(dec_o) or len(evi) != len(evi_o)
            if not bad:
                bad = any(not np.array_equal(dec[k], dec_o[k]) for k in ("event", "status", "self")) or \
                    any(not np.array_equal(dec[k][keep], dec_o[k][keep]) for k in ("model", "target", "n_candidates")) or \
                    any(not np.array_equal(evi[k], evi_o[k]) for k in ("instance", "model", "last_used", "weight", "order", "reload")) or \
                    any(not np.array_equal(rows[k], rows_o[k]) for k in ("lru_time", "used", "count", "capacity")) or rep.n_carry != carry_o
            mism += int(bad)
        if ep >= args.warmup:
            dev_ms.append(rep.ms_total); wall_ms.append(1000.0 * dt)
            phases.append([rep.ms_classify, rep.ms_place, rep.ms_route, rep.ms_apply, rep.ms_registry, rep.ms_commit])
            n_dec += len(dec); n_evict += len(evi); n_lru += rep.n_lru_events; n_pub += rep.n_published
    clocks = sampler.finish()
    launches = s.kernel_launches() - launches0
    dump_outputs(args.dump_outputs, {"decision": dec, "eviction": evi, "instance": rows})
    ph = np.asarray(phases)
    k = len(dev_ms)
    # standalone commits through the C ABI: a window's worth of numeric instance updates -> device path; one string change -> structural
    commit = {}
    rng = np.random.default_rng(1)
    rows2 = rows.copy()
    s.commit()  # (the closed loop left registry changes on the device: the first commit after it folds them into the host tables)
    for label, structural in (("device_path_ms", False), ("structural_path_ms", True)):
        ts, other = [], 0
        for rep_i in range(12 if not structural else 4):
            for i in rng.choice(fl.n_instances, size=min(fl.n_instances, 1200), replace=False):
                rows2[i]["rpm"] = int(rng.integers(0, 3000))
                s.instance_update(int(i), rows2[i])
            if structural:
                s.instance_upsert(0, rows2[0], fl.inst_ids[0] + ("x" * (rep_i % 2)), fl.inst_locs[0], fl.inst_zones[0], fl.inst_labels[0])
            t0 = time.perf_counter()
            s.commit()
            if s.commit_info()[0] == (1 if structural else 2):
                ts.append(1000.0 * (time.perf_counter() - t0))
            else:
                other += 1
        commit[label] = {"p50": float(np.percentile(ts, 50)) if ts else None, "p99": float(np.percentile(ts, 99)) if ts else None, "n": len(ts),
                         "took_the_other_path": other}
    peak, peak_src = measured_hbm_peak()
    copies = len(w.seed_model) / fl.n_instances
    # the LRU kernel's algorithmic bytes (SURVEY.md §8d): 16 B per resident copy scanned per eviction + 16 B per eviction emitted
    lru_bytes = (n_evict / k) * (copies * 16 + 16)
    apply_s = float(ph[:, 3].mean()) / 1000.0
    value = CHURN_EVENTS * k / (sum(dev_ms) / 1000.0)
    line = {
        "metric": CHURN_METRIC, "value": value, "unit": "events/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(dev_ms)), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic", "config": churn_config(),
        "e2e": {"value": CHURN_EVENTS * k / (sum(wall_ms) / 1000.0), "unit": "events/s", "h2d_bytes_per_step": int(CHURN_EVENTS * 24),
                "d2h_bytes_per_step": int((n_dec / k) * 72 + (n_evict / k) * 32 + fl.n_instances * 64), "ms_per_step": float(np.mean(wall_ms)),
                "entry_point": "mmp_churn_step (host buffers: events in, decisions / evictions / republished rows out)"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "k_lru_events", "achieved": lru_bytes / apply_s / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": lru_bytes / apply_s / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(lru_bytes), "kernel_ms_avg": 1000.0 * apply_s,
                     "note": "one warp per instance applies ITS events in order: a 2 s window holds ~8 events per instance, so the launch is "
                             "latency-bound by construction; the roofline figure is reported as SURVEY.md 8d defines it, not as a target"},
        "phases_ms": dict(zip(["classify", "place", "route", "apply_lru", "registry_republish", "commit"], [float(x) for x in ph.mean(axis=0)])),
        "window_commit_ms": {"p50": float(np.percentile(ph[:, 5], 50)), "p99": float(np.percentile(ph[:, 5], 99)),
                             "path": "device (re-rank by counting, tables, bitmap from device-resident edges), CUDA-event time inside the window"},
        "mmp_fleet_commit_ms": commit,
        "per_window": {"decisions": n_dec / k, "evictions": n_evict / k, "lru_events": n_lru / k, "records_republished": n_pub / k},
        "realtime_factor": 2000.0 / float(np.mean(wall_ms)),
        "cpu_baseline": ({"value": CHURN_EVENTS * len(cpu_s) / sum(cpu_s), "unit": "events/s", "cores": 1, "kind": "port",
                          "sample": f"the same {len(cpu_s)} windows through the oracle's closed loop (oracle/mm_sim.inc), one thread",
                          "parity_mismatching_windows": mism} if check else None),
        "clocks": clocks,
    }
    print(json.dumps(line), file=OUT, flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-instance-shards", action="store_true", help="N > 1: skip the instance-sharded leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if CONFIG == "C4":
        return run_churn(args, rank, world, local_rank)

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import ctypes as C
    from modelmesh_b200 import _lib
    from modelmesh_b200._lib import DECISION_IN, DECISION_OUT
    from modelmesh_b200.fleet import Fleet
    from modelmesh_b200.synth import SynthDecisions, load_into_fleet, make_decisions, make_fleet

    lib = _lib.load_product()  # raises if libmmplace.so is missing: no CPU fallback
    fl = make_fleet(CONFIG, N_MODELS, N_INSTANCES, SEED)
    sd_all = make_decisions(fl, N_MODELS, SEED, sweep=True, plain=True)
    # model-shard of this rank (whole registry when world == 1)
    from modelmesh_b200.sharding import shard_range
    lo, hi = shard_range(rank, world, N_MODELS)
    B = hi - lo
    solver = Fleet(fl.min_space_units, fl.min_churn_age_ms, fl.default_model_size_units, fl.n_instances, N_MODELS,
                   device=local_rank, lib=lib)
    load_into_fleet(fl, solver)
    solver._ck(lib.mmp_fleet_set_id_base(solver.h, lo))  # this rank's slice of the sweep keeps the sweep's decision numbering
    dec = np.ascontiguousarray(sd_all.dec[lo:hi])
    row_words = solver.row_words()

    # ---- device-resident timing (the `value`) ----
    d_in, d_out = C.c_void_p(), C.c_void_p()
    solver._ck(lib.mmp_device_alloc(solver.h, dec.nbytes, C.byref(d_in)))
    solver._ck(lib.mmp_device_alloc(solver.h, B * DECISION_OUT.itemsize, C.byref(d_out)))
    solver._ck(lib.mmp_device_upload(solver.h, d_in, dec.ctypes.data_as(C.c_void_p), dec.nbytes))
    kms = C.c_float()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # inputs smaller than L2 (C2: a 12.8 MB bitmap): write a buffer larger than L2 before every timed step
    flush = (lambda: solver._ck(lib.mmp_flush_l2(solver.h))) if B * row_words * 4 < 200e6 else (lambda: None)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.05)
    for _ in range(args.warmup):
        solver._ck(lib.mmp_place_batch_device(solver.h, d_in, B, d_out, fl.now_ms, SEED, C.byref(kms)))
    launches0 = solver.kernel_launches()
    barrier()
    kernel_ms = []
    sampler.mark()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush()
        solver._ck(lib.mmp_place_batch_device(solver.h, d_in, B, d_out, fl.now_ms, SEED, C.byref(kms)))
        kernel_ms.append(float(kms.value))
    barrier()
    wall_s = time.perf_counter() - t_wall0
    dev_ms = float(np.sum(kernel_ms))
    out_dev = np.zeros(B, dtype=DECISION_OUT)
    solver._ck(lib.mmp_device_download(solver.h, out_dev.ctypes.data_as(C.c_void_p), d_out, out_dev.nbytes))
    dump_outputs(args.dump_outputs, {"decision": out_dev}, rank, world)

    # ---- end to end through the C ABI with pinned host buffers ----
    e2e_ms = []
    e2e = None
    if not args.no_e2e:
        h_in, h_out = C.c_void_p(), C.c_void_p()
        solver._ck(lib.mmp_host_alloc(solver.h, dec.nbytes, C.byref(h_in)))
        solver._ck(lib.mmp_host_alloc(solver.h, B * DECISION_OUT.itemsize, C.byref(h_out)))
        C.memmove(h_in, dec.ctypes.data_as(C.c_void_p), dec.nbytes)
        for _ in range(args.warmup):
            solver._ck(lib.mmp_place_batch(solver.h, h_in, B, None, 0, None, 0, h_out, fl.now_ms, SEED))
        barrier()
        for _ in range(args.steps):
            flush()
            t0 = time.perf_counter()
            solver._ck(lib.mmp_place_batch(solver.h, h_in, B, None, 0, None, 0, h_out, fl.now_ms, SEED))
            e2e_ms.append(1000.0 * (time.perf_counter() - t0))
        barrier()
        out_e2e = np.frombuffer((C.c_char * (B * DECISION_OUT.itemsize)).from_address(h_out.value), dtype=DECISION_OUT).copy()
        assert np.array_equal(out_e2e, out_dev), "e2e and device-resident paths disagree"
    # ---- the same batch through the registry-sweep entry point (mmp_place_sweep: 4 B + 1 bit per decision to the device
    # instead of a 32-byte record; results back chunk by chunk), pinned host buffers, copies inside the timed region ----
    sweep_ms, e2e_sweep = [], None
    if not args.no_e2e:
        try:
            from modelmesh_b200._lib import DF_FAVOUR_SELF
            h_self, h_fav, h_out2 = C.c_void_p(), C.c_void_p(), C.c_void_p()
            fav_bits = np.packbits((dec["flags"] & DF_FAVOUR_SELF) != 0, bitorder="little")
            fav_bits = np.concatenate([fav_bits, np.zeros((-len(fav_bits)) % 4, dtype=np.uint8)])
            selfs = np.ascontiguousarray(dec["self"], dtype=np.int32)
            solver._ck(lib.mmp_host_alloc(solver.h, selfs.nbytes, C.byref(h_self)))
            solver._ck(lib.mmp_host_alloc(solver.h, max(4, fav_bits.nbytes), C.byref(h_fav)))
            solver._ck(lib.mmp_host_alloc(solver.h, B * DECISION_OUT.itemsize, C.byref(h_out2)))
            C.memmove(h_self, selfs.ctypes.data_as(C.c_void_p), selfs.nbytes)
            C.memmove(h_fav, fav_bits.ctypes.data_as(C.c_void_p), fav_bits.nbytes)
            for _ in range(args.warmup):
                solver._ck(lib.mmp_place_sweep(solver.h, lo, B, h_self, 1, h_fav, h_out2, fl.now_ms, SEED))
            barrier()
            for _ in range(args.steps):
                flush()
                t0 = time.perf_counter()
                solver._ck(lib.mmp_place_sweep(solver.h, lo, B, h_self, 1, h_fav, h_out2, fl.now_ms, SEED))
                sweep_ms.append(1000.0 * (time.perf_counter() - t0))
            barrier()
            out_sw = np.frombuffer((C.c_char * (B * DECISION_OUT.itemsize)).from_address(h_out2.value), dtype=DECISION_OUT).copy()
            if not np.array_equal(out_sw, out_dev):
                sweep_ms = []  # a result that differs is not a measurement
            else:
                e2e_sweep = {"h2d_bytes_per_step": int(N_MODELS * 4 + (N_MODELS + 7) // 8), "d2h_bytes_per_step": int(N_MODELS * DECISION_OUT.itemsize)}
        except Exception as ex:  # the headline e2e above does not depend on this leg
            print(f"[bench] sweep leg skipped: {ex}", file=sys.stderr)
            sweep_ms = []
    launches = solver.kernel_launches() - launches0
    clocks = sampler.finish() if rank == 0 else None

    # ---- B = 1 latency (p99 decision us): mmp_place_one round trips, three ways of launching the single decision ----
    lat = None
    if rank == 0:
        one = np.zeros(1, dtype=DECISION_OUT)
        lat = {}
        for mode, label in ((3, "resident_server"), (2, "cuda_graph"), (1, "small_kernel"), (0, "streaming_kernel")):
            solver._ck(lib.mmp_tune(solver.h, b"one_mode", mode))
            ts = []
            for i in range(300 + 2000):
                t0 = time.perf_counter()
                lib.mmp_place_one(solver.h, dec[i % B:i % B + 1].ctypes.data_as(C.c_void_p), None, None,
                                  one.ctypes.data_as(C.c_void_p), fl.now_ms, SEED)
                if i >= 300:
                    ts.append(1e6 * (time.perf_counter() - t0))
            lat[label] = {"p50_us": float(np.percentile(ts, 50)), "p99_us": float(np.percentile(ts, 99)), "n": len(ts)}
        solver._ck(lib.mmp_tune(solver.h, b"one_mode", 3))
        lat.update(lat["resident_server"])  # the default path: a request posted to the resident k_place_server
        lat["default_path"] = "resident_server"
        lat["note"] = ("host timer around mmp_place_one (launch + synchronise + 8-byte result through mapped memory); resident_server = a request "
                       "posted to k_place_server (a warp resident for a bounded time polling mapped memory: no launch per call, mmp_tune one_mode=3), cuda_graph = one "
                       "k_place_small node replayed, small_kernel = the same kernel as a stream launch, streaming_kernel = round 1's path")

    # ---- the batch scans on the same fleet (SURVEY.md §8d): ClusterStats (~50 B per instance), the reaper's registry sweep +
    # top-K (24 B per model), each with its CUDA-event time and GB/s against the measured HBM peak ----
    extra_kernels = None
    if rank == 0:
        try:
            peak_e, _ = measured_hbm_peak()
            ms = C.c_double()
            for _ in range(3):
                solver.stats()
            solver._ck(lib.mmp_last_timing(solver.h, b"stats", C.byref(ms)))
            stats_ms = float(ms.value)
            taken = np.zeros(N_MODELS, dtype=np.uint8)
            outm = np.zeros(N_MODELS, dtype=np.int32)
            part = -1 if fl.type_config is None else 0
            n_sel = 0
            for _ in range(3):
                taken[:] = 0
                solver._ck(lib.mmp_flush_l2(solver.h))
                n_sel = solver._ck(lib.mmp_reaper_select(solver.h, part, fl.now_ms, taken.ctypes.data_as(C.c_void_p),
                                                         outm.ctypes.data_as(C.c_void_p), len(outm)))
            solver._ck(lib.mmp_last_timing(solver.h, b"reaper", C.byref(ms)))
            reaper_ms = float(ms.value)
            live = solver.live_instances()
            extra_kernels = [
                {"kernel": "k_stats", "bytes": live * 52, "ms": stats_ms, "GB/s": live * 52 / (stats_ms / 1e3) / 1e9 if stats_ms > 0 else None,
                 "frac": live * 52 / (stats_ms / 1e3) / 1e9 / peak_e if stats_ms > 0 else None,
                 "note": "32 B row + 8 B capacity + 4 B partition + 8 B count/threads per instance; latency-bound at 10k instances"},
                {"kernel": "k_reaper_flag + cub select/sort/select (mmp_reaper_select)", "bytes": N_MODELS * 24, "ms": reaper_ms,
                 "GB/s": N_MODELS * 24 / (reaper_ms / 1e3) / 1e9 if reaper_ms > 0 else None,
                 "frac": N_MODELS * 24 / (reaper_ms / 1e3) / 1e9 / peak_e if reaper_ms > 0 else None, "selected": int(n_sel),
                 "note": "algorithmic bytes = 24 B per model (SURVEY.md 8d); the sort of the candidates is extra traffic on top"}]
        except Exception as ex:
            print(f"[bench] scan legs skipped: {ex}", file=sys.stderr)

    # ---- N > 1: the instance-sharded path of the north star (SURVEY.md §8e), measured in the same run.  Every rank holds
    # a column block of the bitmap for ALL models, resolves the whole batch over its rank range, and one
    # ncclAllReduce(min) over 64-bit min-loc keys combines the shards (inside mmp_place_batch_device). ----
    inst = None
    if world > 1 and not args.no_instance_shards:
        solver.close()  # free the registry shard's bitmap before building the column block
        sh = Fleet(fl.min_space_units, fl.min_churn_age_ms, fl.default_model_size_units, fl.n_instances, N_MODELS,
                   device=local_rank, shard_rank=rank, shard_count=world, lib=lib)
        load_into_fleet(fl, sh)
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(sh.shard_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, src=0)
        sh.shard_connect(bytes(uid.cpu().numpy().tobytes()))
        dec_all = np.ascontiguousarray(sd_all.dec)
        di, do = C.c_void_p(), C.c_void_p()
        sh._ck(lib.mmp_device_alloc(sh.h, dec_all.nbytes, C.byref(di)))
        sh._ck(lib.mmp_device_alloc(sh.h, N_MODELS * DECISION_OUT.itemsize, C.byref(do)))
        sh._ck(lib.mmp_device_upload(sh.h, di, dec_all.ctypes.data_as(C.c_void_p), dec_all.nbytes))
        def timed_leg():
            for _ in range(args.warmup):
                sh._ck(lib.mmp_place_batch_device(sh.h, di, N_MODELS, do, fl.now_ms, SEED, C.byref(kms)))
            barrier()
            ims = []
            for _ in range(args.steps):
                sh._ck(lib.mmp_place_batch_device(sh.h, di, N_MODELS, do, fl.now_ms, SEED, C.byref(kms)))
                ims.append(float(kms.value))
            barrier()
            out_sh = np.zeros(N_MODELS, dtype=DECISION_OUT)
            sh._ck(lib.mmp_device_download(sh.h, out_sh.ctypes.data_as(C.c_void_p), do, out_sh.nbytes))
            # every shard must hold the registry-sharded answers for its own model range
            agree = bool(np.array_equal(out_sh[lo:hi], out_dev))
            t = torch.tensor([float(np.sum(ims)), 0.0 if agree else 1.0], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0]), float(t[1]) == 0.0

        # (a) the collective path: every shard scores the whole batch over its rank range, one all-reduce(min)
        ms_coll, ok_coll = timed_leg()
        wlo, whi, wst = sh.shard_words()
        inst = {"value": N_MODELS * args.steps / (ms_coll / 1000.0), "unit": "decisions/s", "ms_per_step": ms_coll / args.steps,
                "scaling": "strong", "collective": "one ncclAllReduce(min, uint64) of %d min-loc keys per step (%.1f MB) + row-gather "
                "pass for open walks" % (N_MODELS, N_MODELS * 8 / 1e6), "open_decisions_per_step": sh.shard_open_decisions() // (args.steps + args.warmup),
                "rank0_row_words": [wlo, whi], "stored_row_bytes": wst * 4, "matches_registry_sharded": ok_coll}
        # (b) the peer-access path: the batch dealt across the shards, row words beyond the replicated front read from the
        # owning shard's HBM, results stored to every shard -- no NCCL call, no host synchronisation between the shards
        try:
            blobs = [None] * world
            dist.all_gather_object(blobs, sh.shard_ipc_export(N_MODELS))
            sh.shard_ipc_import(blobs)
            barrier()
            ms_peer, ok_peer = timed_leg()
            st = sh.shard_peer_stats()
            tk, tw = C.c_double(), C.c_double()
            lib.mmp_last_timing(sh.h, b"dealt_kernel", C.byref(tk)); lib.mmp_last_timing(sh.h, b"dealt_wait", C.byref(tw))
            tot = torch.tensor([float(st["remote_row_words"]) * 4.0, float(st["result_bytes_to_peers"])], dtype=torch.float64, device="cuda")
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
            n_dec = float(N_MODELS) * max(st["batches"], 1)
            inst["peer_access"] = {
                "value": N_MODELS * args.steps / (ms_peer / 1000.0), "unit": "decisions/s", "ms_per_step": ms_peer / args.steps, "scaling": "strong",
                "exchange": "k_place_dealt: decisions dealt by warp batch, peer loads of row words beyond the %d-word replicated front, "
                            "8-byte results stored to all %d shards, flag arrival + k_dealt_wait (no NCCL, no host sync)" % (16, world),
                "nvlink_bytes_per_decision": {"row_words_read": float(tot[0]) / n_dec, "results_written": float(tot[1]) / n_dec},
                "batches_on_peer_path": st["batches"], "matches_registry_sharded": ok_peer,
                "rank0_last_step_ms": {"k_place_dealt": tk.value, "k_dealt_wait": tw.value}}
        except Exception as ex:  # (the collective figure above stands on its own)
            print(f"[bench] peer-access leg skipped: {ex}", file=sys.stderr)
        sh.close()

    # ---- max over ranks ----
    stats = torch.tensor([dev_ms, float(np.sum(e2e_ms)) if e2e_ms else 0.0, float(np.sum(sweep_ms)) if sweep_ms else 0.0,
                          0.0 if sweep_ms else 1.0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max = float(stats[0]), float(stats[1])
    if e2e_sweep is not None and float(stats[3]) == 0.0:
        e2e_sweep.update({"value": N_MODELS * args.steps / (float(stats[2]) / 1000.0), "unit": "decisions/s",
                          "ms_per_step": float(stats[2]) / args.steps, "entry_point": "mmp_place_sweep"})
    else:
        e2e_sweep = None
    total_decisions = N_MODELS * args.steps
    value = total_decisions / (dev_ms_max / 1000.0)
    if e2e_ms:
        e2e = {"value": total_decisions / (e2e_ms_max / 1000.0), "unit": "decisions/s",
               "h2d_bytes_per_step": int(N_MODELS * DECISION_IN.itemsize), "d2h_bytes_per_step": int(N_MODELS * DECISION_OUT.itemsize),
               "ms_per_step": e2e_ms_max / args.steps}

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        alg_bytes = B * bytes_per_decision(row_words) + 80 * fl.n_instances
        k_avg_s = float(np.mean(kernel_ms)) / 1000.0
        achieved = alg_bytes / k_avg_s / 1e9
        traffic, traffic_src = captured_traffic(B)
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": peak_src, "kernel": scoring_kernel(),
                    "traffic_GBps": (traffic / k_avg_s / 1e9) if traffic else None,
                    "note": ("achieved = ALGORITHMIC bytes (whole bitmap row + model row + result per decision, SURVEY.md 8d) / kernel time. "
                             "k_place_direct reads only the row words a decision looks at, so its DRAM traffic (`traffic`, ncu) is far below "
                             "the algorithmic bytes and `frac` can exceed 1; traffic_GBps = traffic / kernel time is the physical HBM rate"),
                    "traffic_source": (traffic_src + " (ncu --set full, one launch; scaled per decision to this batch)") if traffic_src else None,
                    "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms_avg": 1000.0 * k_avg_s}
        cpu = None
        if not args.no_cpu:
            threads = host_threads()
            done, t_cpu, results = cpu_leg(fl, SynthDecisions(dec, sd_all.fresh, sd_all.extra), budget_s=12.0,
                                           chunk=min(B, 250_000), threads=threads)
            mism = 0
            for a, b_, res in results:
                mism += int(np.count_nonzero(res["target"] != out_dev["target"][a:b_]))
                mism += int(np.count_nonzero(res["n_candidates"] != out_dev["n_candidates"][a:b_]))
            single = None
            try:  # the same path on one thread, bounded sample (SURVEY.md §8d asks for both)
                d1, t1, _ = cpu_leg(fl, SynthDecisions(dec[:100_000], sd_all.fresh, sd_all.extra), budget_s=6.0, chunk=25_000, threads=1)
                single = {"value": d1 / t1, "unit": "decisions/s", "cores": 1, "sample": f"{d1} decisions"}
            except Exception as ex:
                print(f"[bench] single-thread cpu leg skipped: {ex}", file=sys.stderr)
            dense = None
            try:  # CPU mode (ii) of BASELINE.md §4: the same decisions, entries through a rank-ordered array
                d2, t2, _ = cpu_leg(fl, SynthDecisions(dec, sd_all.fresh, sd_all.extra), budget_s=5.0, chunk=min(B, 250_000), threads=threads, dense=True)
                dense = {"value": d2 / t2, "unit": "decisions/s", "cores": threads, "sample": f"{d2} decisions"}
            except Exception as ex:
                print(f"[bench] dense cpu leg skipped: {ex}", file=sys.stderr)
            cpu = {"value": done / t_cpu, "unit": "decisions/s", "cores": threads, "kind": "port", "single_thread": single, "dense": dense,
                   "sample": f"{done} decisions of the same sweep, {threads} threads, C++ restatement of the reference's "
                             f"sorted-set walk (CacheMissForwardingLB.getNext); the Java reference cannot run here",
                   "parity_mismatches_vs_gpu": mism}
        commit_fig = None
        if world == 1:
            try:  # mmp_fleet_commit after a publish window's worth of numeric instance updates (the device path), this fleet's size
                rng_c = np.random.default_rng(7)
                rows2 = fl.inst_rows.copy()
                ts_c, paths = [], []
                for _ in range(6):
                    for i in rng_c.choice(fl.n_instances, size=min(fl.n_instances, 1000), replace=False):
                        rows2[i]["rpm"] = int(rng_c.integers(0, 3000))
                        solver.instance_update(int(i), rows2[i])
                    t0 = time.perf_counter()
                    solver.commit()
                    ts_c.append(1000.0 * (time.perf_counter() - t0))
                    paths.append(int(solver.commit_info()[0]))
                commit_fig = {"p50_ms": float(np.percentile(ts_c[1:], 50)), "max_ms": float(np.max(ts_c[1:])), "n": len(ts_c) - 1,
                              "paths": paths, "note": "host clock around mmp_fleet_commit after 1 000 numeric instance updates; path 2 = rebuilt on the "
                              "device (re-rank by counting, rank tables, masks, bitmap from the device-resident edges), 1 = host"}
            except Exception as ex:
                print(f"[bench] commit leg skipped: {ex}", file=sys.stderr)
        line = {
            "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": workload_config(world),
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "latency_b1": lat, "wall_s_timed_region": wall_s, "extra": extra_kernels, "commit": commit_fig,
        }
        if e2e_sweep is not None and e2e is not None:
            # the workload is a registry sweep, so the call a host makes for it is mmp_place_sweep (INTEGRATION.md §3); the
            # same batch as 32-byte records through mmp_place_batch is kept beside it
            e2e["entry_point"] = "mmp_place_batch"
            line["e2e_records"] = e2e
            line["e2e"] = e2e_sweep
        if inst is not None:
            line["instance_sharded"] = inst
        print(json.dumps(line), file=OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _only_the_json_line_on_stdout():
    """Libraries print to the process's stdout behind Python's back (NCCL's version banner with NCCL_DEBUG=VERSION, ...): route
    file descriptor 1 to stderr for the whole run and keep the original for the one JSON line."""
    global OUT
    try:
        sys.stdout.flush()
        OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    except Exception:
        OUT = sys.stdout


OUT = sys.stdout

if __name__ == "__main__":
    sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (which may be read-only)
    _only_the_json_line_on_stdout()
    main()
