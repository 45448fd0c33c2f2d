#!/usr/bin/env python
"""bench.py — kube-batch allocate-cycle throughput on B200 (driver contract, see DESIGN.md §measurement).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
  python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm (oracle port, mode A)

A "step" is ONE allocate cycle (allocate.go:43-194) over the BASELINE config-3 session: 50k pending tasks /
5k PodGroups / 5k nodes, default tiers [priority,gang][drf,predicates,proportion,nodeorder].
  value  = logical (task,node) pairs evaluated per second = sum over processed tasks of N / device time,
           snapshot already resident in HBM (kb_session_load done once), timed with CUDA events on the
           engine's stream, L2 flushed between steps.
  e2e    = same metric through the public C-ABI call sequence with HOST buffers:
           kb_session_load (host flatten + H2D) + kb_allocate (cycle + decisions D2H) per step, wall clock.
One JSON line on stdout (rank 0).  --dump-outputs DIR also writes the decisions of the last timed step as .npy files, so that
two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "scheduling-cycle throughput: tasks x nodes evaluated/sec"
UNIT = "task-node pairs/s"
ALGO_BYTES_PER_PAIR = 128          # SURVEY.md §8d: predicate+score-relevant node record at R=3, W=2


def workload_desc(name, snap, conf):
    return {
        "workload": f"{name}: {snap.T} pending tasks / {snap.meta.get('pending_jobs', snap.J)} PodGroups / {snap.N} nodes, "
                    f"tiers [{conf.describe()}] (BASELINE.json configs[2])",
        "tasks": int(snap.T), "nodes": int(snap.N), "jobs": int(snap.J), "queues": int(snap.Q),
        "seed": snap.meta.get("seed"), "l2": "256 MiB memset between steps (L2 flush)",
    }


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.samples = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def parity_verdict(workload, eng, res, replica=0):
    """'ok' iff this rank's decisions + node / job state equal the committed oracle digests (tests/golden/cycle_hashes.json;
    `replica` > 0: the digest of that rank's own cluster, synth.make(workload, replica))."""
    from kube_batch_b200 import digest
    hp = os.path.join(ROOT, "tests", "golden", "cycle_hashes.json")
    g = json.load(open(hp)).get(workload + (f"#{replica}" if replica else "")) if os.path.exists(hp) else None
    if g is None:
        return "no committed digest for this workload"
    ns, osr = eng.node_state(), eng.order_state()
    if digest.decisions_digest(res.decisions) != g["decisions"]:
        return "decisions differ from the oracle digest"
    if digest.state_digest(ns["idle"], ns["releasing"], osr["job_ready"], osr["job_share"]) != g["state"]:
        return "node/job state differs from the oracle digest"
    return "ok"


DECISION_FIELDS = ("node", "kind", "dispatched", "step", "dispatch_step")


def dump_outputs(out_dir, res):
    """The decision table one kb_allocate hands its caller, one DIR/decisions_<field>.npy per field.  float64 holds every
    int32 / uint32 value exactly; the largest workload (c5, 1M tasks) comes to 40 MB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for f in DECISION_FIELDS:
        np.save(os.path.join(out_dir, f"decisions_{f}.npy"), res.decisions[f].astype(np.float64))


def cpu_sample(snap, conf, mode, threads, seconds, warm_tasks=0):
    """One bounded sample of the CPU restatement.  warm_tasks > 0: the first warm_tasks task sweeps run with cached aggregates
    (not timed), then the timed sample starts in `mode` — the reference's cost per pair grows with the number of allocated pods
    (plugins/util/util.go:62-85 walks all of them per pair), so samples at several points of the cycle are needed."""
    from oracle import kbo
    o = kbo.allocate(snap, conf, mode=mode, threads=threads, max_seconds=seconds, warm_tasks=warm_tasks)
    r = o.result
    timed = int(r.timed_tasks) if warm_tasks else int(r.tasks_processed)
    return {"pairs_per_s": timed * snap.N / max(r.seconds, 1e-9), "seconds": r.seconds, "tasks": timed,
            "truncated": bool(r.truncated), "jobs_ready": int(r.jobs_ready), "at_task": int(warm_tasks)}


def stratified_reference(snap, conf, threads, seconds_each, total_tasks):
    """Mode A sampled at 0 / 25 / 50 / 75 % of the cycle's task sweeps (SURVEY 8d) and the full-cycle estimate: each quarter of
    the sweeps costs what its sample says."""
    from oracle import kbo
    samples = [cpu_sample(snap, conf, kbo.KBO_MODE_FAITHFUL, threads, seconds_each, warm_tasks=int(total_tasks * f)) for f in (0.0, 0.25, 0.5, 0.75)]
    rates = [max(s["pairs_per_s"], 1e-9) for s in samples]
    est_seconds = sum((total_tasks / 4.0) * snap.N / r for r in rates)
    return samples, total_tasks * snap.N / est_seconds, est_seconds


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank, world):
    """The reference's own algorithm on the host cores: oracle mode A (faithful cost pattern), 16 sweep workers
    like workqueue.ParallelizeUntil(ctx, 16, ...) capped at the core count; each step is a bounded sample."""
    if rank != 0:
        return
    from kube_batch_b200 import synth
    from oracle import kbo
    snap, conf = synth.make(args.workload)
    cores = host_cores()
    threads = min(16, cores)
    per_step = args.ref_seconds
    # the cycle's task sweeps (needed to place the samples): one fast pass with cached aggregates
    full_b = cpu_sample(snap, conf, kbo.KBO_MODE_OPTIMISED, threads, 0.0)
    total_tasks = full_b["tasks"]
    vals = []
    for i in range(args.warmup + args.steps):
        samples, est_rate, est_seconds = stratified_reference(snap, conf, threads, per_step / 4.0, total_tasks)
        if i >= args.warmup:
            vals.append((samples, est_rate, est_seconds))
    value = sum(v[1] for v in vals) / max(1, len(vals))                 # full-cycle estimate (labelled as such in `sample`)
    secs = sum(sum(s["seconds"] for s in v[0]) for v in vals)
    last = vals[-1]
    opt = full_b
    sample = (f"mode A = the reference's per-pair cost pattern (NodeInfo rebuilt per pair, every allocated pod scanned per pair, conservative "
              f"constants), {threads} sweep workers, STRATIFIED: {per_step / 4.0:.1f} s samples starting at 0 / 25 / 50 / 75 % of the cycle's "
              f"{total_tasks} task sweeps -> " + ", ".join(f"{s['pairs_per_s']:.3g} pairs/s @{s['at_task']}" for s in last[0]) +
              f"; value = ESTIMATE of the full cycle from those rates ({last[2]:.0f} s per cycle); mode B (cached aggregates, same decisions, "
              f"whole cycle really executed in {opt['seconds']:.1f} s) shown as value_mode_b")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, len(vals)), "higher_is_better": True,
        # same label as our arm at this N (N > 1: one cluster per GPU there); the CPU rate itself does not depend on N
        "scaling": "weak" if (world > 1 and args.sessions == "independent") else "strong",
        "vs_baseline": None, "dtype": "f64/i64 (CPU)", "data": "synthetic", "config": workload_desc(args.workload, snap, conf),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "value_mode_b": opt["pairs_per_s"], "host_cores": cores, "samples": last[0], "estimated_cycle_seconds": last[2]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference is pure Go and no Go toolchain exists here: this is the C++ restatement (oracle/), not libkbgpu",
    }
    print(json.dumps(line), flush=True)


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    from kube_batch_b200 import engine, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    uid = None
    # NCCL prints its version banner on the C-level stdout: keep stdout clean for the ONE JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        uid_t = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid_t.copy_(torch.frombuffer(bytearray(engine.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid_t, 0)
        uid = bytes(uid_t.cpu().numpy().tobytes())

    # N > 1 (DESIGN.md 6): the cycle is one serial replay, so a second GPU cannot shorten it; what N GPUs buy is N SESSIONS
    # at once.  Default: rank r schedules its OWN cluster of the workload's shape (synth.make(workload, replica=r)) — N
    # independent sessions, no collective, "weak" scaling; every rank's outcome is checked against the committed oracle digest
    # of its cluster.  --sessions replicated: every rank runs the SAME session (the engine's world_size > 1 default), "strong".
    independent = world > 1 and args.sessions == "independent"
    replica = rank if independent else 0
    snap, conf = synth.make(args.workload, replica=replica)
    if independent:
        eng = engine.Engine(device=local_rank)          # a single-GPU engine per rank: the ranks share nothing
    else:
        eng = engine.Engine(device=local_rank, rank=rank, world_size=world, nccl_unique_id=uid)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input steps: value ----
    eng.load(snap, conf)
    for _ in range(args.warmup):
        eng.allocate()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    dev_ms = 0.0
    last = None
    launches = 0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()                      # L2 flush, outside the event-timed cycle
        torch.cuda.synchronize()
        last = eng.allocate()
        dev_ms += last.stats.gpu_ms
        launches += last.stats.kernel_launches
    barrier()
    t_wall1 = time.perf_counter()
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    if dist is not None:
        t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    st = last.stats
    pairs = int(st.pairs_logical)

    # ---- parity of the timed cycle's outcome, on EVERY rank, against the committed oracle digests (outside the timed region) ----
    parity = parity_verdict(args.workload, eng, last, replica)
    if dist is not None:
        t = torch.tensor([1 if parity == "ok" else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 0 and parity == "ok":
            parity = "mismatch on another rank"
    pairs_all, groups_all = pairs, int(st.jobs_ready)
    if independent:            # units ALL ranks processed / max-over-ranks time
        t = torch.tensor([pairs, int(st.jobs_ready)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        pairs_all, groups_all = int(t[0].item()), int(t[1].item())
    value = pairs_all * args.steps / (dev_ms * 1e-3)
    groups_per_s = groups_all * args.steps / (dev_ms * 1e-3)

    # ---- end to end through the C ABI with host buffers: e2e ----
    e2e_steps = max(1, min(args.steps, 5))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.load(snap, conf)               # host flatten + H2D of the whole snapshot
        r = eng.allocate()                 # cycle + decisions D2H
    barrier()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_pairs = int(r.stats.pairs_logical)
    if independent:
        t = torch.tensor([e2e_pairs], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        e2e_pairs = int(t.item())
    e2e_value = e2e_pairs * e2e_steps / e2e_s

    if rank != 0:
        eng.close()
        if dist is not None:
            dist.destroy_process_group()
        if parity != "ok" and args.workload in ("c2", "c3", "c4"):
            raise SystemExit(f"bench.py rank {rank}: parity check failed: {parity}")
        return
    workload = workload_desc(args.workload, snap, conf)
    workload["parallelism"] = ("single GPU" if world == 1 else
                               f"{world} independent sessions, one cluster of this shape per GPU (seeds +1000 per rank), no collective" if independent else
                               f"one session replicated on {world} GPUs (every rank runs the whole cycle), no collective")

    # ---- roofline of the dominant kernel: algorithmic bytes of its scans / device time ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak = 6650.0; peak_src = "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
    scans = int(st.pairs_scanned) // max(1, snap.N)
    ach = int(st.pairs_scanned) * ALGO_BYTES_PER_PAIR / (st.gpu_ms * 1e-3) / 1e9 * world
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        traffic = tj.get("cycle_kernel_dram_bytes_per_launch") if bool(getattr(st, "pipeline", 0)) else tj.get("visit_kernel_dram_bytes_per_launch")
    pipe = bool(getattr(st, "pipeline", 0))
    if pipe:
        # persistent pipeline: ONE cycle_kernel launch per cycle; its scanner CTAs evaluate `pairs_scanned` (class, node) pairs
        # (one pass over the resident node tiles per scan request)
        kern, n_launch, bytes_per_launch = "cycle_kernel", 1, int(st.pairs_scanned) * ALGO_BYTES_PER_PAIR
    else:
        kern, n_launch, bytes_per_launch = "visit_kernel", int(st.kernel_launches), int(snap.N) * ALGO_BYTES_PER_PAIR
    roofline = {
        "bound": "hbm", "achieved": ach, "peak": peak * world, "unit": "GB/s", "frac": ach / (peak * world), "traffic": traffic,
        "kernel": kern, "launches_per_step": n_launch, "scans_per_step": scans,
        "algorithmic_bytes_per_launch": bytes_per_launch,
        "avg_launch_us": 1e3 * st.gpu_ms / max(1, n_launch), "peak_source": peak_src,
        # SURVEY 8d counts the reference's (task, node) pairs: 128 B each.  The engine scans one CLASS per visit instead of every
        # task, so `achieved` (pairs really scanned) is the honest kernel figure and this one is the algorithm-level equivalent
        "achieved_logical_pairs": int(st.pairs_logical) * ALGO_BYTES_PER_PAIR / (st.gpu_ms * 1e-3) / 1e9 * world,
        "frac_logical_pairs": int(st.pairs_logical) * ALGO_BYTES_PER_PAIR / (st.gpu_ms * 1e-3) / 1e9 / peak,
        "note": "pairs the scans really evaluated x 128 B / device time of the cycle; the node table stays resident in shared memory "
                "(pipeline) or L2 (per-launch kernels): the cycle is bound by the latency of the sequential replay, not by bandwidth",
    }

    # ---- the same K1+K2+K3 arithmetic as ONE launch over the full task x node matrix (kb_best_nodes): the
    #      speculative, non-sequential face of the path; shows what the kernel does when it is not latency-bound ----
    matrix = None
    if world == 1:
        eng.load(snap, conf)
        tms = []
        for _ in range(5):
            eng.best_nodes(0, snap.T)
            tms.append(eng.last_kernel_ms())
        mms = sorted(tms)[len(tms) // 2]
        mp = snap.T * snap.N
        matrix = {"kernel": "best_nodes_kernel", "pairs": mp, "ms": mms, "pairs_per_s": mp / (mms * 1e-3),
                  "achieved": mp * ALGO_BYTES_PER_PAIR / (mms * 1e-3) / 1e9, "unit": "GB/s", "peak": peak,
                  "frac": mp * ALGO_BYTES_PER_PAIR / (mms * 1e-3) / 1e9 / peak,
                  "note": "every (task,node) pair of the snapshot evaluated against the initial state in one launch; node tiles are staged "
                          "once per CTA by TMA and reused from shared memory, so the algorithmic-byte rate may exceed the HBM peak: "
                          "the kernel is instruction-bound, not bandwidth-bound"}

    # ---- CPU baseline on this box's host cores (bounded samples) ----
    from oracle import kbo
    cores = host_cores()
    threads = min(16, cores)
    b = cpu_sample(snap, conf, kbo.KBO_MODE_OPTIMISED, threads, args.cpu_seconds)
    samples, est_rate, est_seconds = stratified_reference(snap, conf, threads, args.cpu_seconds / 4.0, int(st.tasks_processed))
    cpu_baseline = {
        "value": est_rate, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": f"mode A (reference cost pattern), stratified: {args.cpu_seconds / 4.0:.1f} s samples starting at 0 / 25 / 50 / 75 % of the "
                  f"cycle's {int(st.tasks_processed)} task sweeps: " + ", ".join(f"{s['pairs_per_s']:.3g} pairs/s @{s['at_task']}" for s in samples) +
                  f"; value = full-cycle ESTIMATE from those rates ({est_seconds:.0f} s per cycle); "
                  f"mode B (cached aggregates): {b['tasks']} task sweeps in {b['seconds']:.1f} s"
                  f"{'' if b['truncated'] else ' = the whole cycle, really executed'}",
        "value_mode_b": b["pairs_per_s"], "host_cores": cores, "samples": samples, "estimated_cycle_seconds": est_seconds,
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak" if independent else "strong", "vs_baseline": None,
        "dtype": "f64 compares + i64 scores + u64 bitmasks", "data": "synthetic",
        "config": workload,
        "podgroups_placed_per_s": groups_per_s,
        "parity": parity,
        "pairs_scanned_per_s": int(st.pairs_scanned) / (st.gpu_ms * 1e-3),
        "pairs_scanned_per_step": int(st.pairs_scanned),
        "tasks_processed": int(st.tasks_processed), "tasks_allocated": int(st.tasks_allocated), "podgroups_ready": int(st.jobs_ready),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(r.stats.h2d_bytes), "d2h_bytes_per_step": int(r.stats.d2h_bytes),
                "ms_per_step": 1e3 * e2e_s / e2e_steps, "steps": e2e_steps,
                "what": "kb_session_load (host flatten + H2D) + kb_allocate (cycle + decisions D2H), wall clock"},
        "gpu_launches": launches,
        "sessions": ("independent" if independent else "replicated") if world > 1 else "one",
        "exchange": {0: "none (single GPU)", 1: "ncclAllGather per scan", 2: "fused peer-memory exchange (NVLink stores + flags) inside visit_kernel",
                     3: "none: every rank runs the whole cycle on the full (replicated) node table"}.get(int(st.exchange_mode), "?"),
        "engine_mode": "persistent pipeline (cycle_kernel)" if pipe else "per-visit launches (visit_kernel)",
        "visit_chains_per_step": int(st.scans), "scan_requests_per_step": int(getattr(st, "pipe_requests", 0)),
        "roofline": roofline, "roofline_matrix_kernel": matrix, "cpu_baseline": cpu_baseline, "clocks": clocks,
        "wall_ms_per_step_incl_flush": 1e3 * (t_wall1 - t_wall0) / args.steps,
        "lib": eng.L.kb_version().decode(),
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    eng.close()
    if dist is not None:
        dist.destroy_process_group()
    if parity != "ok" and args.workload in ("c2", "c3", "c4"):
        raise SystemExit(f"bench.py: parity check failed: {parity}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--sessions", default="independent", choices=["independent", "replicated"],
                    help="N > 1: one cluster per GPU (weak scaling, default) or the same session on every GPU (strong)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="wall-time bound of each cpu_baseline sample")
    ap.add_argument("--ref-seconds", type=float, default=6.0, help="wall-time bound of one --impl reference step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the decisions of the last timed step (rank 0) as DIR/decisions_<field>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm runs bounded samples, not whole cycles")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("bench.py: --gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
