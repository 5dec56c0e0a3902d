#!/usr/bin/env python
"""bench.py — one JSON line per run (driver contract, hot-path tier).

A "step" is one pass of the hot path (PreFilter + pod x node fit/score + gang admit + queue
sort = one bs_evaluate) over one synthetic snapshot.

HEADLINE (every N): BASELINE.json configs[3]'s snapshot per GPU (100k pods / 10k nodes / 50k
PodGroups, 5 resource lanes) — the one the north-star target is quoted on; it fits one GPU.  Weak
scaling: every rank owns its own 100k pods / 50k groups, the node table is replicated, and the only
exchange is the all-gather of the admit bitmap, every step (engine peer-memory kernels; the same
through NCCL is timed beside it at N > 1).

  value         fit-evals/s, inputs resident in HBM, score matrix + fit bitmap materialised
  e2e           same metric through the C ABI with HOST (pinned) tables: H2D upload of the three
                tables + evaluate + D2H of every decision vector inside the timed region
  strong        N > 1: BASELINE configs[3] cut N ways and configs[4] (1M pods / 50k nodes / 9 lanes)
                group-sharded over the N GPUs as ONE problem, with an in-run parity check of the
                merged admit bitmap against the CPU oracle on a reduced snapshot
  roofline      gang_fit kernel, algorithmic bytes / its CUDA-event time vs measured HBM peak
  cpu_baseline  the CPU oracle (port of the reference algorithm) on the host cores, bounded sample

Timing: W warm-up steps, then a barrier + synchronize, then the timed steps with one CUDA event
per step on the engine's stream, then the exchange stream joined, a final event, barrier +
synchronize.  With --steps K the timed region runs exactly K steps.  Without it, it runs 200 steps
or --min-time seconds of device time (default 1 s), whichever is MORE (a 30 ms region cannot be
timed across 8 ranks); giving both makes --min-time a floor on top of K.  `steps` in the line is
what ran, `steps_requested` what was asked.  MAX over ranks.  Clocks are sampled through NVML
inside the process (no nvidia-smi subprocess between the barrier and the first step).

--dump-outputs DIR writes what the last timed step computed (rank 0) as DIR/<name>.npy, float64,
so that two builds can be compared output for output on the same seeded snapshot: see dump_outputs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "pod_x_node_fit_evals_per_sec"
UNIT = "fit-evals/s"
WORKLOAD_CFG = 4


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                d = json.load(f)
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(d.get("sm_max_mhz", 1965.0))
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0


def usable_threads() -> int:
    """Host threads this process can actually run: the smaller of the CPU affinity mask and the cgroup
    CPU quota (cpu.max quota/period) — a container on a 128-core box may own far fewer."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(math.ceil(int(txt[0]) / int(txt[1])))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(math.ceil(q / per))))
            break
        except Exception:
            continue
    return max(1, n)


class ClockSampler:
    """SM clock + throttle reasons of one GPU, sampled in-process through NVML every 50 ms (a thread: about 20 samples
    inside the >= 1 s timed region; NVML queries take driver locks, so no more often than that);
    `window(t0, t1)` summarises the samples taken inside a perf_counter interval.  Falls back to one
    nvidia-smi -lms subprocess (started long before the timed region) when NVML is unavailable."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake"}

    def __init__(self, torch_device_index: int):
        self.samples = []          # (t, sm_mhz, reasons_mask, power_w)
        self.sm_max = None
        self.stop_flag = False
        self.thread = None
        self.proc = None
        self.src = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                props = torch.cuda.get_device_properties(torch_device_index)
                uuid = getattr(props, "uuid", None)
                if uuid is not None:
                    h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                h = None
            if h is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = torch_device_index
                if vis:
                    try:
                        idx = int(vis.split(",")[torch_device_index])
                    except Exception:
                        pass
                h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv, self.h = pynvml, h
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.src = "nvml"
        except Exception:
            self.nv = None
            self.gpu = torch_device_index

    def _loop_nvml(self):
        nv, h = self.nv, self.h
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                rs = int(get_reasons(h))
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                self.samples.append((time.perf_counter(), mhz, rs, pw))
            except Exception:
                pass
            time.sleep(0.05)

    def _loop_smi(self):
        names = [0x8, 0x40, 0x20, 0x4]
        for ln in self.proc.stdout:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                mhz, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            self.sm_max = max(self.sm_max or 0.0, mx)
            rs = 0
            for bit, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    rs |= bit
            self.samples.append((time.perf_counter(), mhz, rs, None))

    def start(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._loop_nvml, daemon=True)
            self.thread.start()
            return
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.src = "nvidia-smi"
            self.thread = threading.Thread(target=self._loop_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def window(self, t0: float, t1: float):
        sel = [s for s in self.samples if t0 <= s[0] <= t1]
        if not sel:   # a region shorter than the sampling period: the two samples around it
            before = [s for s in self.samples if s[0] < t0][-1:]
            after = [s for s in self.samples if s[0] > t1][:1]
            sel = before + after
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "samples": 0, "reasons": ["no clock samples"],
                    "source": self.src}
        mask = 0
        for s in sel:
            mask |= s[2]
        pw = [s[3] for s in sel if s[3] is not None]
        return {"sm_mhz": float(np.median([s[1] for s in sel])), "sm_max_mhz": self.sm_max, "samples": len(sel),
                "reasons": sorted(v for k, v in self.REASONS.items() if mask & k),
                "power_w_max": max(pw) if pw else None, "source": self.src}

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()


def table_bytes(snap):
    n = 0
    for t in (snap.nodes, snap.pods, snap.groups):
        for f in t.__dataclass_fields__:
            if getattr(t, f) is not None:
                n += getattr(t, f).nbytes
    return n


def gang_fit_alg_bytes(P, N, G, L, n_fit_classes=64, narrow_lanes=0):
    """Algorithmic bytes of ONE gang_fit launch (DESIGN.md 'gang_fit roofline'):
    reads: residual table 8·L·N (int32 lanes count 4), requests 8·L·P, per-pod class 4·P, class-fit bits;
    writes: score matrix 8·P·N, fit bitmap P·N/8, per-pod results 16·P."""
    W = (N + 31) // 32
    reads = (8 * L - 4 * narrow_lanes) * N + 8 * L * P + 4 * P + 4 * W * n_fit_classes
    writes = 8 * P * N + 4 * P * W + 16 * P
    return reads + writes


def workload_config(scale: float):
    """The `config` object BOTH arms print (identical keys and values: the driver compares them)."""
    sc = lambda x: max(1, int(round(x * scale)))
    P, N, G = sc(100000), sc(10000), sc(50000)
    return {"workload": "cfg4: 100k pods / 10k nodes, 50k groups, priority-sorted queue "
                        "(BASELINE.json configs[3] snapshot per GPU)",
            "pods_per_gpu": P, "nodes": N, "groups_per_gpu": G, "lanes": 5,
            "outputs": "score matrix int64 PxN + fit bitmap + decisions",
            "l2": "each step streams an %.1f GB score matrix (>> 126 MB L2): working set larger than L2, "
                  "no explicit flush" % (8.0 * P * N / 1e9),
            "scale": scale}


def cpu_round_time(oracle, S, snap, n_pods, threads, faithful=True):
    sub = snap if n_pods >= snap.pods.n else S.Snapshot(snap.nodes, snap.pods.take(np.arange(n_pods)), snap.groups)
    t0 = time.perf_counter()
    oracle.round(sub, want_bitmap=True, want_score=False, faithful=faithful, threads=threads)
    return time.perf_counter() - t0


def cpu_sample(oracle, S, snap, seconds, threads, faithful=True):
    """Times the CPU oracle (reference algorithm, per-pod PreFilter as in core.go) on a bounded
    pod sample of the same snapshot: whole node and group tables, first n pods."""
    n = min(snap.pods.n, 64 * max(1, threads))
    dt = cpu_round_time(oracle, S, snap, n, threads, faithful)
    n2 = int(min(snap.pods.n, max(n, n * seconds / max(dt, 1e-4))))
    dt = cpu_round_time(oracle, S, snap, n2, threads, faithful)
    return n2 * snap.nodes.n / dt, n2, dt


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port; the Go binary cannot be built
    here) on the host cores.  B2 = every usable host thread over the FULL snapshot per step whenever
    the whole run fits ~4 minutes (it does for the driver's --steps 20 --warmup 5), B1 = one thread on
    a bounded sample (BASELINE.md §3's single-thread definition), reported beside it."""
    if rank != 0:
        return
    from oracle import oracle
    S = importlib.import_module("batch-scheduler_b200.snapshot")
    snap = S.config(WORKLOAD_CFG, args.scale)
    threads = usable_threads()
    steps = args.steps if args.steps is not None else 5
    warm = args.warmup if args.warmup is not None else 1
    v, _, _ = cpu_sample(oracle, S, snap, seconds=2.0, threads=threads)
    budget_s = 240.0
    full_s = snap.pods.n * snap.nodes.n / v
    n_step = snap.pods.n if full_s * (steps + warm) <= budget_s else \
        int(min(snap.pods.n, max(64, v * budget_s / (steps + warm) / snap.nodes.n)))
    sub = snap if n_step == snap.pods.n else S.Snapshot(snap.nodes, snap.pods.take(np.arange(n_step)), snap.groups)
    for _ in range(warm):
        oracle.round(sub, want_bitmap=True, want_score=False, faithful=True, threads=threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.round(sub, want_bitmap=True, want_score=False, faithful=True, threads=threads)
    dt = time.perf_counter() - t0
    value = steps * n_step * snap.nodes.n / dt
    v1, n1, dt1 = cpu_sample(oracle, S, snap, seconds=6.0, threads=1)
    what = ("per-pod PreFilter re-runs findMaxPG + the ordered node scan (core.go:120,140,161), fit bitmap written, "
            "full queue sort")
    sample = (f"{'all' if n_step == snap.pods.n else 'first'} {n_step} pods of the {snap.pods.n}-pod snapshot against all "
              f"{snap.nodes.n} nodes and {snap.groups.n} groups per step; {what}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(args.scale),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "label": "B2: every usable host thread (min of CPU affinity and cgroup quota)"},
        "cpu_baseline_1thread": {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                                 "sample": f"first {n1} pods x all {snap.nodes.n} nodes, {dt1:.1f} s; {what}",
                                 "label": "B1: single thread (BASELINE.md §3)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "sample_pods_per_step": n_step,
        "note": "reference = C restatement of pkg/scheduler/core/core.go (oracle/); the Go reference needs "
                "k8s.io/kubernetes v1.17.5 + ~130 modules and a Go toolchain, neither present",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class Harness:
    """One rank's view: torch.distributed plumbing + the timed-region protocol."""

    def __init__(self, args, rank, local_rank, world):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        self.dev = f"cuda:{local_rank}"

    def full_sync(self, *engs):
        for e in engs:
            e.sync()
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def timed(self, eng, step, steps_req, warmup, min_time_s, join=None, sampler=None):
        """W warm-up steps; barrier; K timed steps (K = max(steps_req, what min_time_s needs), the same on
        every rank) with an event per step on the engine stream; `join` (exchange stream) before the last
        event; barrier.  Returns total ms (max over ranks), steps, per-step ms of this rank, clock window."""
        torch = self.torch
        ext = torch.cuda.ExternalStream(eng.stream(), device=self.local_rank)
        for _ in range(warmup):
            step()
        self.full_sync(eng)
        # pilot: how long is a step?  (same count on every rank: max over ranks)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(ext)
        for _ in range(3):
            step()
        if join:
            join()
        p1.record(ext)
        self.full_sync(eng)
        est_ms = self.max_over_ranks(p0.elapsed_time(p1) / 3.0)
        steps = int(max(steps_req, math.ceil(min_time_s * 1e3 / max(est_ms, 1e-3))))
        steps = int(self.max_over_ranks(steps))
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        end = torch.cuda.Event(enable_timing=True)
        self.full_sync(eng)                      # barrier + synchronize; nothing but the loop follows
        t0 = time.perf_counter()
        evs[0].record(ext)
        for i in range(steps):
            step()
            evs[i + 1].record(ext)
        if join:
            join()
        end.record(ext)
        self.full_sync(eng)
        t1 = time.perf_counter()
        total = evs[0].elapsed_time(end)
        per = np.array([evs[i].elapsed_time(evs[i + 1]) for i in range(steps)])
        clocks = sampler.window(t0, t1) if sampler is not None else None
        return self.max_over_ranks(total), steps, per, clocks

    def gather_objects(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out


def step_stats(per):
    return {"p50_ms": float(np.percentile(per, 50)), "p99_ms": float(np.percentile(per, 99)),
            "max_ms": float(per.max()), "mean_ms": float(per.mean())}


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_PODS = 256


def dump_outputs(eng, out_dir):
    """Writes the round the engine last evaluated as its caller receives it: every decision vector of bs_fetch in
    full, and the rows of a fixed, seeded sample of pods (`pod_sample`) of the P x N score matrix and of the fit
    bitmap (words), which are GB-sized at the headline size.  float64 holds every value exactly: scores are small
    integers or INT64_MIN ("no fit"), the rest are 32-bit integers."""
    res = eng.fetch()
    arrays = {f: getattr(res, f) for f in ("prefilter", "feasible_count", "best_node", "best_score", "admit",
                                           "admit_bitmap", "new_denied", "order", "rank")}
    arrays["max_group"] = np.array([res.max_group])
    arrays["max_finished"] = np.array([res.max_finished])
    rng = np.random.default_rng(0)
    pods = np.sort(rng.choice(eng.P, min(eng.P, DUMP_SAMPLE_PODS), replace=False))
    arrays["pod_sample"] = pods
    arrays["score_rows"] = np.concatenate([eng.score_rows(int(p), 1) for p in pods])
    arrays["fit_bitmap_rows"] = np.concatenate([eng.fit_rows(int(p), 1) for p in pods])
    total = sum(a.size * 8 for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total / 2**20:.0f} MB (limit 64 MB); use a smaller --scale")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def make_nccl_exchange(H, eng, capi):
    """all_gather_into_tensor over a torch view of the engine's admit-bitmap device buffer, enqueued on
    the engine's stream right behind the round."""
    torch, dist = H.torch, H.dist
    eng.evaluate_async(); eng.sync()
    ptr, nbytes = eng.device_buffer(capi.BUF_ADMIT_BITMAP)

    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<i4", "data": (ptr, False), "version": 2}
    bitmap_t = torch.as_tensor(h, device=H.dev)
    gathered = torch.empty(H.world * bitmap_t.numel(), dtype=torch.int32, device=H.dev)
    ext = torch.cuda.ExternalStream(eng.stream(), device=H.local_rank)

    def exchange():
        with torch.cuda.stream(ext):
            dist.all_gather_into_tensor(gathered, bitmap_t)
    return exchange, gathered


def peer_setup(H, eng, words):
    def _ag(b):
        out = [None] * H.world
        H.dist.all_gather_object(out, b)
        return out
    eng.peer_setup(H.rank, H.world, words, _ag)
    H.dist.barrier()


def strong_leg(H, pkg, cfg, scale, steps_req, warmup, min_time_s, score=True):
    """ONE snapshot (BASELINE configs[cfg-1]) group-sharded over the ranks: first-pod capture resolved
    globally, contiguous group ranges balanced by pod count, node and group tables replicated, admit
    bitmap all-gathered every step by the engine's peer-memory exchange."""
    S = pkg.snapshot
    full = S.config(cfg, scale).resolve_groups()
    local = full.shard_groups(H.rank, H.world)
    P, N, G, L = local.pods.n, full.nodes.n, full.groups.n, full.lanes
    eng = pkg.Engine(L, H.local_rank, fit_bitmap=True, score=score)
    eng.upload(local)
    peer_setup(H, eng, (G + 31) // 32)
    total_ms, steps, per, _ = H.timed(eng, eng.evaluate_async, steps_req, warmup, min_time_s, join=eng.peer_join)
    pairs = H.sum_over_ranks(float(P) * N)
    # the same shard with no exchange and no peers: what the rank's own work takes
    H.dist.barrier()
    eng.peer_detach()
    H.dist.barrier()
    solo_ms, solo_steps, _, _ = H.timed(eng, eng.evaluate_async, max(5, min(steps_req, 20)), 2, 0.2)
    eng.close()
    ranks = H.gather_objects({"rank": H.rank, "pods": int(P), **step_stats(per)})
    out = {"config": {"workload": full.name, "pods": int(full.pods.n), "nodes": int(N), "groups": int(G), "lanes": int(L),
                      "sharding": f"{H.world}-way by contiguous group range, balanced by pod count; nodes + groups replicated",
                      "outputs": ("score matrix + " if score else "") + "fit bitmap + decisions", "scale": scale},
           "value": pairs * steps / (total_ms * 1e-3), "unit": UNIT, "ms_per_step": total_ms / steps, "steps": steps,
           "ms_per_step_no_exchange": solo_ms / solo_steps,
           "exchange_overhead_frac": (total_ms / steps) / (solo_ms / solo_steps) - 1.0,
           "per_rank": ranks}
    return out


def strong_parity(H, pkg, cfg, scale):
    """Outside any timed region: a reduced snapshot of the strong-scaling workload evaluated by the same
    sharded path (engine + peer-memory all-gather); rank 0 checks the merged gathered admit bitmap and
    its own decision vectors against the CPU oracle's UNSHARDED round."""
    S = pkg.snapshot
    full = S.config(cfg, scale).resolve_groups()
    local = full.shard_groups(H.rank, H.world)
    g0, g1 = local.meta["group_range"]
    G = full.groups.n
    eng = pkg.Engine(full.lanes, H.local_rank, fit_bitmap=False, score=False)
    eng.upload(local)
    peer_setup(H, eng, (G + 31) // 32)
    for _ in range(2):     # two rounds: both slot sets of the exchange are exercised
        eng.evaluate_async()
    eng.sync()
    words = eng.gathered_admit()
    res = eng.fetch()
    H.dist.barrier()
    eng.peer_detach()
    eng.close()
    ranges = H.gather_objects((int(g0), int(g1)))
    ok = None
    if H.rank == 0:
        from oracle import oracle
        ref = oracle.round(full, want_bitmap=False, threads=usable_threads())
        merged = np.zeros(G, bool)
        for r, (a0, a1) in enumerate(ranges):
            bits = np.unpackbits(words[r].view(np.uint8), bitorder="little")[:G].astype(bool)
            merged[a0:a1] = bits[a0:a1]
        idx = local.meta["pod_index"]
        ok = bool(np.array_equal(merged, ref.admit == S.ADMIT) and np.array_equal(res.admit[g0:g1], ref.admit[g0:g1])
                  and np.array_equal(res.prefilter, ref.prefilter[idx])
                  and np.array_equal(res.feasible_count, ref.feasible_count[idx])
                  and np.array_equal(res.best_node, ref.best_node[idx]) and res.max_group == ref.max_group)
    return {"parity_checked": ok, "snapshot": full.name + f" at scale {scale}", "pods": int(full.pods.n),
            "nodes": int(full.nodes.n), "groups": int(G),
            "what": "merged gathered admit bitmap == oracle admit, rank-0 admit/prefilter/feasible_count/best_node/"
                    "max_group == oracle's unsharded round"}


def sass_issue_roofline(pairs, ms, clock_mhz):
    """Decisions-only regime (SURVEY 8(d) R2): instruction-issue roofline.  Ops per (pod,node) pair are
    counted from the committed SASS of the decisions-only kernel (profiles/sass_ops_r2.json, written by
    profiles/tools/sass_count.py): peak = 148 SMs x 4 schedulers x 32 lanes x clock / issued ops per pair;
    the ALU-pipe bound uses the 64 lanes/clk/SM of the integer ALU pipe and the ALU ops per pair."""
    p = os.path.join(ROOT, "profiles", "sass_ops_r2.json")
    if not os.path.exists(p):
        return None
    try:
        ops = json.load(open(p))
        issue, alu = float(ops["issue_ops_per_pair"]), float(ops["alu_pipe_ops_per_pair"])
    except Exception:
        return None
    clk = clock_mhz * 1e6
    peak_issue = 148 * 128 * clk / issue
    peak_alu = 148 * 64 * clk / alu
    achieved = pairs / (ms * 1e-3)
    return {"bound": "int-issue", "achieved": achieved, "peak": peak_issue, "unit": UNIT, "frac": achieved / peak_issue,
            "issue_ops_per_pair": issue, "alu_pipe_ops_per_pair": alu, "alu_pipe_peak": peak_alu,
            "alu_pipe_frac": achieved / peak_alu, "clock_mhz": clock_mhz,
            "source": "ops counted from SASS: profiles/sass_ops_r2.json (kernel " + str(ops.get("kernel")) + ")"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debug only; marks the line)")
    ap.add_argument("--min-time", type=float, default=None,
                    help="the timed region lasts at least this many seconds of device time (more steps than --steps if "
                         "needed); default 1 s without --steps, none with it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-replay", action="store_true", help="skip the multi-round admission leg")
    ap.add_argument("--no-strong", action="store_true", help="N>1: skip the strong-scaling legs")
    ap.add_argument("--no-objects", action="store_true", help="skip the e2e legs that start from API objects")
    ap.add_argument("--exchange", default="both", choices=["p2p", "nccl", "both"],
                    help="N>1: admit-bitmap all-gather by the engine's peer-memory kernels (headline), by NCCL, or both")
    args = ap.parse_args()
    if args.min_time is None:
        args.min_time = 0.0 if args.steps is not None else 1.0

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    steps_req = args.steps if args.steps is not None else 200
    warmup = max(args.warmup if args.warmup is not None else 3, 3)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    H = Harness(args, rank, local_rank, world)
    sampler = ClockSampler(local_rank)
    sampler.start()               # long before any timed region; in-process, no subprocess per step

    pkg = importlib.import_module("batch-scheduler_b200")
    S = pkg.snapshot
    capi = pkg.capi

    snap = S.config(WORKLOAD_CFG, args.scale, shard=rank)
    P, N, G, L = snap.pods.n, snap.nodes.n, snap.groups.n, snap.lanes

    # pinned host copies of the three tables (the e2e leg uploads from these every step)
    def pin_table(t):
        for f in t.__dataclass_fields__:
            a = getattr(t, f)
            if a is None:
                continue
            h = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype)) if a.dtype != np.uint32 and a.dtype != np.uint64
                            else (torch.int32 if a.dtype == np.uint32 else torch.int64), pin_memory=True)
            v = h.numpy().view(a.dtype)
            v[...] = a
            setattr(t, f, v)
            t.__dict__.setdefault("_pins", []).append(h)
    for t in (snap.nodes, snap.pods, snap.groups):
        pin_table(t)

    eng = pkg.Engine(L, local_rank, fit_bitmap=True, score=True)
    eng.upload(snap)

    # ---- headline: device-resident weak-scaling leg ---------------------------------------------
    use_p2p = world > 1 and args.exchange in ("p2p", "both")
    exch_nccl = None
    legs = {}
    if world > 1 and args.exchange in ("nccl", "both"):
        exch_nccl, _gathered = make_nccl_exchange(H, eng, capi)

        def step_nccl():
            eng.evaluate_async()
            exch_nccl()
        tot, st, per, clk = H.timed(eng, step_nccl, steps_req, warmup, args.min_time, sampler=sampler)
        legs["nccl"] = {"ms_total": tot, "steps": st, "per": per, "clocks": clk}
    if use_p2p:
        peer_setup(H, eng, (G + 31) // 32)
    if world == 1 or use_p2p:
        launches0 = eng.launch_count()
        tot, st, per, clk = H.timed(eng, eng.evaluate_async, steps_req, warmup, args.min_time,
                                    join=eng.peer_join if use_p2p else None, sampler=sampler)
        legs["p2p" if use_p2p else "single"] = {"ms_total": tot, "steps": st, "per": per, "clocks": clk}
        launches_per_step = (eng.launch_count() - launches0) / float(st + warmup + 3)
    else:
        launches_per_step = None
    head_key = "p2p" if use_p2p else ("single" if world == 1 else "nccl")
    head = legs[head_key]
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    total_pairs = H.sum_over_ranks(float(P) * N)
    total_groups = H.sum_over_ranks(float(G))
    value = total_pairs * head["steps"] / (head["ms_total"] * 1e-3)
    admit_rate = total_groups * head["steps"] / (head["ms_total"] * 1e-3)
    per_rank = H.gather_objects({"rank": rank, **step_stats(head["per"])})
    exchange_lines = None
    if world > 1:
        exchange_lines = {}
        for k, lg in legs.items():
            allr = H.gather_objects(step_stats(lg["per"]))
            exchange_lines[k] = {"value": total_pairs * lg["steps"] / (lg["ms_total"] * 1e-3), "unit": UNIT,
                                 "ms_per_step": lg["ms_total"] / lg["steps"], "steps": lg["steps"],
                                 "p50_ms_max_rank": max(r["p50_ms"] for r in allr),
                                 "p99_ms_max_rank": max(r["p99_ms"] for r in allr)}
    if launches_per_step is None:
        l0 = eng.launch_count(); eng.evaluate_async(); eng.sync(); launches_per_step = eng.launch_count() - l0

    # ---- per-kernel CUDA-event times (same process, same data, per-step sync) -------------
    eng.set_profiling(True)
    kms = {k: [] for k in capi.KERNEL_NAMES}
    for _ in range(max(5, min(steps_req, 30))):
        eng.evaluate_async()
        eng.sync()
        for k, (ms, n) in eng.kernel_ms().items():
            kms[k].append(ms)
    eng.set_profiling(False)
    kavg = {k: float(np.mean(v)) for k, v in kms.items()}
    fit_ms = kavg["gang_fit"]
    peak, peak_src, sm_max_mhz = load_peaks()
    shape = eng.fit_shape() if hasattr(eng, "fit_shape") else None
    narrow = (shape["LN"] + shape["LS"]) if shape else 0
    alg = gang_fit_alg_bytes(P, N, G, L, 64, narrow)
    achieved = alg / (fit_ms * 1e-3) / 1e9 if fit_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get(f"cfg{WORKLOAD_CFG}_gang_fit_dram_bytes")
            traffic_src = "static: profiles/ncu_traffic.json (" + str(tj.get("source")) + "), not measured in this run"
        except Exception:
            traffic = None

    # ---- decisions-only regime (SURVEY 8(d) R2): same round, no P x N matrix leaves the SMs ------
    fused = None
    if world == 1:
        eng2 = pkg.Engine(L, local_rank, fit_bitmap=False, score=False)
        eng2.upload(snap)
        ftot, fst, fper, fclk = H.timed(eng2, eng2.evaluate_async, max(10, min(steps_req, 50)), 3, min(args.min_time, 0.3),
                                        sampler=sampler)
        eng2.set_profiling(True)
        fk = []
        for _ in range(10):
            eng2.evaluate_async(); eng2.sync()
            fk.append(eng2.kernel_ms()["gang_fit"][0])
        eng2.set_profiling(False)
        fms = ftot / fst
        clk_mhz = (fclk or {}).get("sm_mhz") or sm_max_mhz
        fused = {"ms_per_step": fms, "value": float(P) * N / (fms * 1e-3), "unit": UNIT, "steps": fst,
                 "gang_fit_ms": float(np.mean(fk)),
                 "what": "same round with out_flags=0: prefilter/admit/order/feasible-count/best-node only; "
                         "the tables are L2-resident, so the bound is instruction issue, not HBM",
                 "roofline": sass_issue_roofline(float(P) * N, float(np.mean(fk)), clk_mhz)}
        eng2.close()

    # ---- multi-round admission (SURVEY 8(f) row 4): the whole queue through bs_replay, once ----
    replay = None
    if world == 1 and not args.no_replay:
        order = eng.evaluate().order.copy()
        eng.replay(order, after_state=False)            # warm-up (allocations, first touch)
        eng.set_profiling(True)
        t0 = time.perf_counter()
        out = eng.replay(order, after_state=False)
        wall = time.perf_counter() - t0
        rms = eng.kernel_ms()["replay"][0]
        eng.set_profiling(False)
        replay = {"pods": int(P), "ms": wall * 1e3, "kernel_ms": rms, "pods_per_s": P / wall,
                  "assumed": int((out["node"] >= 0).sum()), "gangs_ready": int(out["ready"].sum()),
                  "what": "bs_replay: every pod of the queue (device sort order) through PreFilter -> first fitting node "
                          "-> assume -> Permit against mutable state; host queue in, verdicts out"}
        if rank == 0 and not args.no_cpu_baseline:
            from oracle import oracle
            sub = S.config(WORKLOAD_CFG, scale=min(args.scale, 0.3))
            engs = pkg.Engine(L, local_rank, fit_bitmap=False, score=False)
            engs.upload(sub)
            so = engs.evaluate().order.copy()
            engs.replay(so, after_state=False)
            t0 = time.perf_counter(); g = engs.replay(so, after_state=False); tg = time.perf_counter() - t0
            engs.close()
            t0 = time.perf_counter(); pf, node, rdy, _ = oracle.replay(sub, so); tc = time.perf_counter() - t0
            same = bool((pf == g["prefilter"]).all() and (node == g["node"]).all() and (rdy == g["ready"]).all())
            replay["cpu_port_sample"] = {"pods": int(sub.pods.n), "nodes": int(sub.nodes.n), "cpu_ms": tc * 1e3,
                                         "gpu_ms": tg * 1e3, "identical": same, "cores": 1,
                                         "what": "oracle bso_replay (sequential by nature) on the same reduced snapshot"}

    # ---- e2e leg: host tables -> C ABI -> host decisions, every step ------------------------
    res = None
    for _ in range(2):
        eng.upload(snap)
        res = eng.evaluate(view=True)
    H.full_sync(eng)
    t0 = time.perf_counter()
    e2e_steps = max(3, min(steps_req, 30))   # wall clock with host passes in it: enough steps to ride out jitter
    br = {"upload_nodes": 0.0, "upload_groups": 0.0, "upload_pods": 0.0, "evaluate_fetch": 0.0}
    for _ in range(e2e_steps):
        ta = time.perf_counter(); eng.upload_nodes(snap.nodes)
        tb = time.perf_counter(); eng.upload_groups(snap.groups)
        tc = time.perf_counter(); eng.upload_pods(snap.pods)
        td = time.perf_counter(); res = eng.evaluate(view=True)   # bs_evaluate_view: one D2H into the pinned arena, read in place
        te_ = time.perf_counter()
        br["upload_nodes"] += tb - ta; br["upload_groups"] += tc - tb; br["upload_pods"] += td - tc
        br["evaluate_fetch"] += te_ - td
        if world > 1 and not use_p2p and exch_nccl:
            exch_nccl()
            torch.cuda.synchronize()
    H.full_sync(eng)
    e2e_dt = H.max_over_ranks(time.perf_counter() - t0)
    e2e_value = total_pairs * e2e_steps / e2e_dt
    h2d = table_bytes(snap)
    d2h = sum(getattr(res, f).nbytes for f in ("prefilter", "feasible_count", "best_node", "best_score", "admit",
                                               "admit_bitmap", "new_denied", "order", "rank"))
    # ---- delta e2e: what a scheduling cycle looks like once the tables are resident — 1 % of the node rows and
    # 1 % of the group rows changed on the host (bs_update_nodes / bs_update_groups: H2D of the changed rows +
    # device scatter), evaluate, one D2H of every decision vector
    e2e_delta = None
    if world == 1:
        rng = np.random.default_rng(7)
        nn, ng = max(1, N // 100), max(1, G // 100)
        ni = np.sort(rng.choice(N, nn, replace=False)).astype(np.uint32)
        gi = np.sort(rng.choice(G, ng, replace=False)).astype(np.uint32)
        nrows = S.NodeTable(snap.nodes.alloc[:, ni], snap.nodes.requested[:, ni], snap.nodes.pod_count[ni],
                            snap.nodes.alloc_present[ni], snap.nodes.req_present[ni], snap.nodes.label_mask[ni],
                            snap.nodes.taint_mask[ni], snap.nodes.flags[ni])
        grows = S.GroupTable(snap.groups.min_member[gi], snap.groups.scheduled[gi], snap.groups.matched[gi],
                             snap.groups.flags[gi], snap.groups.min_res[:, gi], snap.groups.min_res_present[gi],
                             snap.groups.rep_sel[gi], snap.groups.rep_tol[gi], snap.groups.creation_ns[gi],
                             snap.groups.name_rank[gi])
        for _ in range(3):
            eng.update_nodes(ni, nrows); eng.update_groups(gi, grows); res = eng.evaluate(view=True)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            eng.update_nodes(ni, nrows); eng.update_groups(gi, grows); res = eng.evaluate(view=True)
        dd = time.perf_counter() - t0
        e2e_delta = {"ms_per_step": dd / e2e_steps * 1e3, "value": float(P) * N * e2e_steps / dd, "unit": UNIT,
                     "steps": e2e_steps, "changed_nodes": int(nn), "changed_groups": int(ng),
                     "h2d_bytes_per_step": int(sum(getattr(nrows, f).nbytes for f in nrows.__dataclass_fields__) + ni.nbytes +
                                               sum(getattr(grows, f).nbytes for f in grows.__dataclass_fields__
                                                   if getattr(grows, f) is not None) + gi.nbytes),
                     "d2h_bytes_per_step": int(d2h),
                     "what": "bs_update_nodes + bs_update_groups (1 % of the rows each) + bs_evaluate_view (one D2H of every "
                             "decision vector into the engine's pinned arena, read in place), wall clock"}
    if use_p2p:
        dist.barrier()
        eng.peer_detach()
    eng.close()

    # ---- e2e from API objects (packer included) + delta rounds: the C++ plugin mirror ----------
    objects = None
    pb = os.path.join(ROOT, "profiles", "tools", "plugin_bench")
    if rank == 0 and world == 1 and not args.no_objects and os.path.exists(pb):
        try:
            env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "batch-scheduler_b200") + ":" +
                       os.environ.get("LD_LIBRARY_PATH", ""))
            outp = subprocess.run([pb, str(args.scale), str(local_rank)], capture_output=True, text=True, timeout=300, env=env)
            objects = json.loads(outp.stdout.strip().splitlines()[-1])
            objects["value"] = float(P) * N / (objects["full_round_ms"] * 1e-3)
            objects["delta_value"] = float(P) * N / (objects["delta_round_ms"] * 1e-3)
            objects["unit"] = UNIT
        except Exception as ex:   # the leg is additional evidence, never the headline
            objects = {"error": repr(ex)[:200]}

    # ---- strong scaling: ONE snapshot sharded over the ranks (BASELINE configs[3] and [4]) ------
    strong = None
    if world > 1 and not args.no_strong:
        strong = {}
        s4 = strong_leg(H, pkg, 4, args.scale, steps_req, 3, min(args.min_time, 0.5))
        strong["cfg4"] = s4
        # cfg5: 1M pods x 50k nodes; a rank's int64 score shard is (1M / world) x 50k x 8 B
        shard_gb = 1e6 * args.scale / world * 50000 * args.scale * 8 / 1e9
        free_gb = torch.cuda.mem_get_info()[0] / 1e9
        with_score = shard_gb < 0.85 * free_gb
        s5 = strong_leg(H, pkg, 5, args.scale, max(5, min(steps_req, 20)), 2, min(args.min_time, 0.5), score=with_score)
        if not with_score:
            s5["note"] = f"score shard {shard_gb:.0f} GB does not fit {free_gb:.0f} GB free: fit bitmap + decisions only"
        strong["cfg5"] = s5
        strong["parity"] = strong_parity(H, pkg, 5, 0.02 * args.scale)
        strong["parity_checked"] = strong["parity"]["parity_checked"]

    # ---- CPU baseline (rank 0, N=1 only) ----------------------------------------------------
    cpu = None
    cpu1 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        threads = usable_threads()
        what = "per-pod PreFilter as in core.go (findMaxPG + ordered node scan per pod), OpenMP over pods"
        v, n_pods, dt = cpu_sample(oracle, S, snap, seconds=12.0, threads=threads)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"first {n_pods} pods x all {N} nodes / {G} groups of the same snapshot, {dt:.1f} s, {what}"}
        v1, n1, dt1 = cpu_sample(oracle, S, snap, seconds=5.0, threads=1)
        cpu1 = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"first {n1} pods x all {N} nodes, {dt1:.1f} s, one thread (BASELINE.md §3 B1)"}

    sampler.stop()
    if rank == 0:
        cfg = workload_config(args.scale)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": head["steps"],
            "steps_requested": steps_req, "warmup": warmup, "ms_per_step": head["ms_total"] / head["steps"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": cfg,
            "sharding": ("groups/pods per rank, node table replicated, admit bitmap all-gathered every step by "
                         + ("the engine's peer-memory kernels over NVLink (CUDA IPC): a push kernel closes the round, the wait "
                            "runs on a side stream one round deep" if use_p2p else "one NCCL all-gather")) if world > 1 else "single GPU",
            "timing": {"min_time_s": args.min_time, "per_rank": per_rank,
                       "what": "CUDA events on the engine stream, one per step; barrier + synchronize on both sides; max over ranks"},
            "exchange": exchange_lines,
            "admit_decisions_per_s": admit_rate,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "ms_per_step": e2e_dt / e2e_steps * 1e3,
                    "breakdown_ms": {k: v / e2e_steps * 1e3 for k, v in br.items()},
                    "what": "bs_upload_nodes/groups/pods from pinned host tables + bs_evaluate_view (one D2H of all decision "
                            "vectors into the engine's pinned arena, read in place) per step, wall clock"},
            "e2e_delta": e2e_delta,
            "e2e_objects": objects,
            "gpu_launches": int(round(launches_per_step * head["steps"])),
            "gpu_launches_per_step": launches_per_step,
            "kernel_ms": kavg,
            "decisions_only": fused,
            "replay": replay,
            "strong": strong,
            "roofline": {"bound": "hbm", "kernel": "gang_fit_kernel" + (str(shape) if shape else ""), "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": traffic,
                         "traffic_source": traffic_src, "peak_source": peak_src, "alg_bytes_per_launch": int(alg),
                         "kernel_ms": fit_ms},
            "cpu_baseline": cpu,
            "cpu_baseline_1thread": cpu1,
            "clocks": head["clocks"],
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
