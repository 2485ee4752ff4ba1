#!/usr/bin/env python3
"""bench.py — admission decisions/sec of the batched scheduling-cycle evaluator.

    python bench.py --gpus N --steps K --warmup W [--config 2] [--impl reference] [--dump-outputs DIR]

One "step" = one scheduling cycle (tree pass -> nominate [+ target search] -> group ->
order -> admit) over one synthetic snapshot of a BASELINE.json configuration.  Default
workload = cfg3, the configuration the north star's target is quoted on (1M pending x 10k
ClusterQueues, flat cohorts, DRF fair sharing): one reference cycle = the 10k queue heads.
cfg2 / cfg4 evaluate every pending workload as an entry (the batched evaluator).
`value` = decisions/sec with the snapshot already resident in HBM (device time from
CUDA events on the library's launching stream, L2 flushed between steps); `e2e` =
the same metric through the reference-facing C-ABI call kb_run_cycle with host
buffers (host -> device copies, kernels, device -> host copies all inside the timed
region).  N > 1: each rank evaluates its own snapshot shard (root cohorts are
independent, so there is no data-path collective) — weak scaling.

--impl reference times the CPU restatement of the reference's cycle (oracle/, the
Go toolchain is absent so the Go scheduler itself cannot run here) on the host cores.

--dump-outputs DIR writes the tables the last timed step handed its caller (rank 0's) as
DIR/<name>.npy; tables without rows are left out.  Inputs are seeded, so two builds, or the two --impl arms, run with the same
arguments can be compared table by table.
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

METRIC = "admission decisions/sec per scheduling cycle"
UNIT = "decisions/s"
WORKLOADS = {
    1: "cfg1: 100 pending x 10 CQ x 2 flavors x 3 resources",
    2: "cfg2: 100k pending x 1k ClusterQueues x 8 flavors x 4 resources, StrictFIFO, no borrowing",
    3: "cfg3: 1M pending x 10k ClusterQueues, BestEffortFIFO + flat cohorts + DRF fair sharing",
    4: "cfg4: 1M pending x 10k ClusterQueues, depth-4 hierarchical cohorts + within-cohort/reclaim preemption, 200k admitted",
    5: "cfg5: topology-aware placement, 100k nodes (10 blocks x 100 racks x 100 hosts), 10k podset requests per cycle (one head per ClusterQueue)",
}


# cfg3 runs the fair-sharing iterator, which holds one entry per ClusterQueue
# (fair_sharing_iterator.go:52-54): its step is one reference cycle over the Q heads.
HEADS = {1: "all", 2: "all", 3: "one_per_cq", 4: "one_per_cq", 5: "one_per_cq"}
DUMP_LIMIT = 64 << 20


def cycle_tables(out) -> dict:
    """The result tables of one scheduling cycle (abi.CycleOut), target lists cut to their used length."""
    t = {f: getattr(out, f) for f in ("decision", "mode", "borrow", "commit_rank", "ps_flavor", "ps_res_mode", "ps_tried_idx",
                                      "ps_count", "tgt_start", "node_usage")}
    t["tgt_adm"], t["tgt_reason"] = out.tgt_adm[:out.n_targets], out.tgt_reason[:out.n_targets]
    return t


def tas_tables(out, n_req: int) -> dict:
    """The result tables of one kb_tas_find (tas.TasOut), cut to the requests and assignments actually written."""
    n = int(out.asg_start[-1])
    return {"status": out.status[:n_req], "asg_start": out.asg_start, "asg_leaf": out.asg_leaf[:n], "asg_count": out.asg_count[:n]}


def dump_outputs(path: str, tables: dict) -> None:
    """Writes every table as <path>/<name>.npy: integers of up to 16 bits as float32, wider ones as float64 (exact up
    to 2^53, checked).  A table without rows is left out: the target lists of a cycle that preempts nothing are
    empty, and tgt_start already says so."""
    conv = {}
    for name, a in tables.items():
        a = np.asarray(a)
        if a.size == 0:
            continue
        f = a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64)
        if not np.array_equal(f.astype(a.dtype), a):
            raise ValueError(f"--dump-outputs: {name} is not exact in {f.dtype}")
        conv[name] = f
    total = sum(f.nbytes for f in conv.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, f in conv.items():
        np.save(os.path.join(path, name + ".npy"), f)


def algorithmic_bytes(snap) -> dict:
    """Algorithmic bytes per launch of each kernel (DESIGN.md (d)).

    nominate is SURVEY.md §8(d): B = W_eval*(P*R*8 + 24) + W_eval*out_B + (Q+C)*FR*32 + (Q+C)*16.
    tree: nominal/borrow/lend limits + CQ usage in, SubtreeQuota/usage/available/potentialAvailable out.
    rank: the 32-byte iterator key of every entry in, its rank out.
    admit: per entry the assignment rows (flavor 1 B + request 8 B per podset x resource) and 16 B of
           mode/borrow/targets, the root's quota tables (usage, SubtreeQuota, lendingLimit, borrowingLimit)
           in, usage back out, 5 B of decision + rank out.
    """
    W = snap.n_heads
    P = snap.n_podset / max(1, snap.n_wl)
    R, FR, N = snap.n_resource, snap.n_fr, snap.n_nodes
    nrg = snap.n_rg / max(1, snap.n_cq)
    wl_in = W * (P * R * 8 + 24)
    wl_out = W * (8 + P * nrg)
    nodes = N * FR * 32 + N * 16
    A = snap.n_adm
    AU = len(snap.arrays["adm_use_fr"])
    return {"k_nominate": wl_in + wl_out + nodes, "k_nominate_search_fair": wl_in + wl_out + nodes,
            # ranking of the admitted workloads: cq, priority, reservation time, uid, evicted in; sorted index, rank, per-CQ list out
            "k_rank_admitted": A * 37,
            # search tables: the four [node][FR] quota tables in, transposed usage + 32 B cell record + mask out; usage cells in, 32 B bucket records out
            "k_search_tables": N * FR * (32 + 44) + AU * (12 + 32),
            # target searches stream 32 B candidate records; the count is data dependent and reported by the library
            # (kb_stats.search_records); this entry is the per-entry floor used when the counter is absent
            "k_search_cells": wl_in + nodes, "k_nominate_walk": wl_in + wl_out + nodes,
            "k_fair_prep": N * FR * 16 + N * R * 16, "k_drain": W * 64, "k_tas": 0,
            # fused per-root cycle: nominal / limits / ClusterQueue usage in, usage out, entries in, assignments + decisions out
            "k_cycle_flat": N * FR * 40 + N * 16 + wl_in + wl_out + W * 5,
            "k_tree": N * FR * 64 + N * 16, "k_lone": N * FR * 64,
            "k_rank": W * 36, "k_scatter": W * 72, "k_scan_roots": N * 8,
            "k_admit": W * (P * R * 9 + 16) + N * FR * 40 + W * 5,
            "total": wl_in + wl_out + nodes}


def measured_traffic(config: int, kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return t[f"cfg{config}"][kernel]
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self._stop_evt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append((float(out[0]), float(out[1])))
                for n, v in zip(names, out[2:]):
                    if v.strip().lower() == "active":
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": sorted(self.reasons)}


def go_toolchain():
    """The reference is 100 % Go: with a Go toolchain on the box its own Scheduler.schedule() harness
    (scheduler_test.go:8139-8209) could serve as the reference arm.  Probe and report; without it the arm is the C++
    restatement (kind "port")."""
    import shutil
    exe = shutil.which("go")
    if not exe:
        return None
    try:
        return subprocess.run([exe, "version"], capture_output=True, text=True, timeout=10).stdout.strip() or exe
    except Exception:  # noqa: BLE001
        return exe


def cpu_baseline(snap, budget_s: float = 12.0):
    """Oracle (kind 'port') on one host core over repeated passes of the same snapshot."""
    import oracle
    oracle.run_cycle(snap)  # warm
    n, t0 = 0, time.perf_counter()
    while True:
        oracle.run_cycle(snap)
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= 200:
            break
    return {"value": n * snap.n_heads / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n} full passes of the same snapshot ({snap.n_heads} decisions each) in {dt:.1f} s, 1 thread "
                      f"(the reference cycle is single-goroutine, scheduler.go:468)",
            "go_toolchain_on_box": go_toolchain()}


def pin_to_gpu_numa(local_rank: int):
    """Bind this rank to the CPUs local to its GPU (sysfs local_cpulist of the PCI function) BEFORE any pinned host
    memory is allocated: first-touch then places the page-locked snapshot on the GPU's NUMA node, so the per-cycle
    DMA does not cross the inter-socket link.  Returns what was done for the bench line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        node = open(base + "/numa_node").read().strip()
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": int(node), "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001 — sysfs layout differs between boxes; running unpinned is only slower
        return {"numa_node": None, "error": type(e).__name__}
    return {"numa_node": None}


def drain_line(ev, config: int, cpu: bool):
    """Drain mode (SURVEY.md §8d): kb_run_drain over the WHOLE pending set of the configuration (every pending
    workload sits in its ClusterQueue's queue on the device), next to the host definition of the drain iterating the
    oracle.  decisions = entries evaluated over all cycles until a cycle admits nothing."""
    from kueue_b200 import abi, native, synth
    snap = native.pin_snapshot(synth.make_snapshot(config))  # heads ignored: whole queues
    out = abi.DrainOut(snap, max_cycles=1000, trace=False)
    ev.run_drain(snap, out)  # warm (allocations, first-touch)
    t0 = time.perf_counter()
    ev.run_drain(snap, out)
    wall = time.perf_counter() - t0
    line = {"pending": snap.n_wl, "cycles": out.n_cycles, "decisions": out.n_decisions, "admitted": out.n_admitted,
            "device_ms": out.gpu_ms, "decisions_per_s_device": out.n_decisions / (out.gpu_ms / 1e3) if out.gpu_ms else None,
            "e2e_ms": wall * 1e3, "decisions_per_s_e2e": out.n_decisions / wall,
            "e2e_includes": "upload of the whole snapshot from pinned host memory, per-ClusterQueue queue sort, all cycles, result download"}
    if cpu:
        import oracle
        from kueue_b200.drain import drain
        t0 = time.perf_counter()
        ref = drain(snap, oracle.run_cycle, max_cycles=1000)
        dt = time.perf_counter() - t0
        line["cpu"] = {"decisions_per_s": ref.n_decisions / dt, "cycles": ref.cycles, "decisions": ref.n_decisions, "admitted": ref.n_admitted,
                       "kind": "port", "cores": 1, "sample": f"kueue_b200/drain.py iterating the oracle: {ref.cycles} cycles in {dt:.1f} s"}
    return line


def run_tas(args, rank, world, local_rank):
    """cfg5: one step = kb_tas_find over the cycle's podset requests (FindTopologyAssignmentsForFlavor per head)."""
    import torch
    import torch.distributed as dist
    from kueue_b200 import abi, native, tas
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # N > 1: every rank places the requests of its own cohorts' ClusterQueues on its own replica of the topology
    # tables (cfg5 "sharded by cohort"): weak scaling, no data-path collective
    topo = tas.synth_topology(10, 100, 100)
    nreq = 10_000
    reqs = tas.synth_requests(topo, nreq, seed=7 + rank, shapes=16)
    cap = int(reqs.count.sum()) + 16
    ev = native.Evaluator(local_rank)
    ev.set_profile(True)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(3, args.warmup)):
        ev.tas_find(topo, reqs, cap)
    sampler = ClockSampler(local_rank); sampler.start()
    barrier()
    dev_ms, kms, launches = 0.0, np.zeros(20), 0
    for _ in range(args.steps):
        flush.zero_(); torch.cuda.synchronize()
        last = ev.tas_find(topo, reqs, cap)
        st = ev.stats()
        dev_ms += st.last_cycle_gpu_ms; kms += np.array(list(st.kernel_ms)); launches += st.kernel_launches
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tas_tables(last, nreq))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = ev.tas_find(topo, reqs, cap)
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([dev_ms, e2e_s, float(nreq)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, total = tmax[0].item(), tmax[1].item(), tsum[2].item()
    else:
        total = float(nreq)
    if rank == 0:
        NL, R = topo.n_leaves, len(topo.resources)
        ms = dev_ms / args.steps
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        names = abi.KERNEL_NAMES
        per = {names[i]: kms[i] / args.steps for i in range(20) if kms[i] > 0 and i != 14}
        kname = max(per, key=per.get)
        # algorithmic bytes: leaf pass = per distinct shape every leaf's capacity + usage rows (R x 16 B), masks (8 B) in, state + sliceState (8 B) out;
        # select = per request the (state, sliceState) of the domains of its level and of the children it descends into, 8 B each (lower bound: its level once)
        level_sizes = np.diff(topo.level_start)
        ab = {"k_tas_leaf": 16 * NL * (R * 16 + 16), "k_tas_reduce": 16 * int(level_sizes.sum()) * 16,
              "k_tas_select": float(sum(int(level_sizes[l]) for l in reqs.level) * 8 + nreq * 64)}
        kbytes = ab.get(kname, 0.0)
        top_ms = per[kname]
        achieved = kbytes / (top_ms / 1e3) / 1e9 if top_ms else 0.0
        h2d = int(topo.free.nbytes + topo.usage.nbytes + topo.cap_mask.nbytes * 2 + topo.parent.nbytes + reqs.pod_request.nbytes + reqs.count.nbytes * 8)
        d2h = int(nreq * 8 + out.asg_start[-1] * 8)
        line = {"metric": METRIC, "value": total / (ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": {"workload": WORKLOADS[5], "decisions_per_step_per_gpu": nreq, "request_shapes": 16,
                           "l2": "512 MiB flush buffer written between timed steps",
                           "timing": "CUDA events on the library stream around the kernels of kb_tas_find, summed over steps, max over ranks",
                           "placed": int((out.status == 0).sum()), "no_fit": int((out.status == 1).sum())},
                "clocks": clocks, "e2e": {"value": total * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": launches, "kernel_ms_per_step": per,
                "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                             "traffic": measured_traffic(5, kname), "algorithmic_bytes_per_launch": kbytes, "kernel_ms": top_ms,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"}}
        if world == 1 and not args.no_cpu_baseline:
            import oracle
            sample = tas.synth_requests(topo, 400, seed=7, shapes=16)
            oracle.tas_find(topo, sample)
            t0 = time.perf_counter(); n = 0
            while time.perf_counter() - t0 < 10:
                oracle.tas_find(topo, sample); n += 1
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": n * 400 / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"{n} passes over the first 400 requests of the same distribution on the same topology in {dt:.1f} s, 1 thread"}
        print(json.dumps(line))
    ev.close()
    if world > 1:
        dist.destroy_process_group()


def run_reference(args, rank, world):
    from kueue_b200 import synth
    if rank != 0:
        return
    import oracle
    if args.config == 5:
        from kueue_b200 import tas
        topo = tas.synth_topology(10, 100, 100)
        sample = tas.synth_requests(topo, 400, seed=7, shapes=16)
        for _ in range(args.warmup):
            oracle.tas_find(topo, sample)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            last = oracle.tas_find(topo, sample)
        dt = time.perf_counter() - t0
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, tas_tables(last, 400))
        val = args.steps * 400 / dt
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                          "config": {"workload": WORKLOADS[5], "sample": "every step places the first 400 requests of the cycle's distribution on the same 100k-node topology"},
                          "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port", "sample": f"{args.steps} passes of 400 requests"},
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    snap = synth.make_snapshot(args.config, heads=HEADS[args.config])
    if HEADS[args.config] == "one_per_cq":
        snap = synth.compact_to_heads(snap)
    for _ in range(args.warmup):
        oracle.run_cycle(snap)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = oracle.run_cycle(snap)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cycle_tables(last))
    val = args.steps * snap.n_heads / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.config],
                       "heads": "all pending workloads (batched evaluator)" if HEADS[args.config] == "all" else "one head per ClusterQueue (reference cycle)",
                       "decisions_per_step_per_gpu": snap.n_heads,
                       "sample": "every step is one full pass of the N=1 snapshot on rank 0's host cores"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": f"{args.steps} full passes ({snap.n_heads} decisions each); C++ restatement of "
                                       "pkg/scheduler, 1 thread like the reference's cycle",
                             "go_toolchain_on_box": go_toolchain()},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-drain", action="store_true")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"])
    ap.add_argument("--l2", default="rotate", choices=["rotate", "flush"],
                    help="how inputs are kept out of L2 between timed steps: rotate = device-resident copies of the snapshot "
                         "whose total exceeds L2, used round-robin; flush = a 512 MiB buffer is written before every step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the tables the last timed step returned (rank 0's) as DIR/<name>.npy, "
                         f"float32 / float64, at most {DUMP_LIMIT >> 20} MiB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.config == 5:
        return run_tas(args, rank, world, local_rank)

    import torch
    import torch.distributed as dist
    from kueue_b200 import abi, native, synth
    torch.cuda.set_device(local_rank)
    numa = pin_to_gpu_numa(local_rank) if world > 1 else {"numa_node": None}
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # Root cohorts are independent coupling domains (resource_node.go:106-108), so ranks take disjoint sets of roots
    # (kueue_b200.shard) and there is no collective on the data path; the decisions are gathered and merged on rank 0.
    #   weak scaling (default): the cluster grows with the number of GPUs (world x the config's ClusterQueues and
    #     pending workloads);
    #   strong scaling (--scaling strong, the default of cfg4): the configuration's own snapshot is split by root —
    #     cfg4 has 10 root cohorts, so 8 GPUs hold at most 2 roots each (5x is the ceiling of this partition).
    scaling = args.scaling or ("strong" if args.config == 4 else "weak")
    shard_map, glob_heads = None, None  # noqa: F841
    my_heads = None  # global entry positions of this rank's entries
    if world > 1 and scaling == "strong":
        from kueue_b200 import shard as kshard
        glob = synth.make_snapshot(args.config, heads=HEADS[args.config])
        if HEADS[args.config] == "one_per_cq":
            glob = synth.compact_to_heads(glob)
        glob_heads = glob.n_heads
        snap, shard_map = kshard.shard(glob, rank, world)
        my_heads = np.asarray(shard_map.heads)
        del glob
    elif world > 1:
        # weak scaling: the cluster is `world` times the configuration — since root cohorts never interact, that is
        # the union of `world` independent copies of the configuration (different seeds), one per rank; the sharding
        # of ONE snapshot by root (shard -> device per shard -> merge == unsharded oracle) is covered by tests/
        snap = synth.make_snapshot(args.config, heads=HEADS[args.config], seed=1000 + rank)
        if HEADS[args.config] == "one_per_cq":
            snap = synth.compact_to_heads(snap)
        glob_heads = snap.n_heads * world
        my_heads = np.arange(snap.n_heads) + rank * snap.n_heads
    else:
        snap = synth.make_snapshot(args.config, heads=HEADS[args.config])
    if HEADS[args.config] == "one_per_cq":
        snap = synth.compact_to_heads(snap)  # the cycle only ever receives the heads (queues.Heads())
    ev = native.Evaluator(local_rank)
    snap = native.pin_snapshot(snap)            # host SoA buffers are page-locked (kb_alloc_pinned)
    out = native.pin_cycle_out(abi.CycleOut(snap, with_usage=False))  # decisions only: the host cache applies usage itself (cache.AssumeWorkload)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident-input throughput (value) ----
    # Inputs must not be L2-resident when a timed step starts.  Default (--l2 rotate): the snapshot is uploaded into
    # several evaluators (own device tables each, static ones included) whose total size exceeds L2 (126 MB), and the
    # steps walk them round-robin, so a step's tables were last touched more than an L2 ago; the kernels' code stays
    # where a scheduler that runs cycle after cycle has it.  --l2 flush: one copy, a 512 MiB buffer written before every
    # step (this also evicts the code; reported as value_l2_flush next to the headline).
    L2_BYTES = 126 << 20
    ev.upload(snap)
    copy_bytes = max(1, int(ev.stats().h2d_bytes))
    n_copies = 1 if args.l2 == "flush" else min(64, int(np.ceil(1.35 * L2_BYTES / copy_bytes)) + 1)
    evs = [ev]
    for _ in range(n_copies - 1):
        e2 = native.Evaluator(local_rank)
        e2.upload(snap)
        evs.append(e2)

    def timed_pass(steps, use_flush, profile):
        dev, lau, km = 0.0, 0, np.zeros(20)
        for k in range(steps):
            e = evs[k % len(evs)]
            if use_flush:
                flush.zero_(); torch.cuda.synchronize()
            e.set_profile(profile)
            e.cycle_resident()
            st_ = e.stats()
            dev += st_.last_cycle_gpu_ms; lau += st_.kernel_launches; km += np.array(list(st_.kernel_ms))
            if profile:
                e.set_profile(False)
        return dev, lau, km

    use_flush = args.l2 == "flush"
    timed_pass(max(3, args.warmup) * len(evs) if not use_flush else max(3, args.warmup), use_flush, False)
    sampler = ClockSampler(local_rank); sampler.start()
    barrier()
    t_wall0 = time.perf_counter()
    dev_ms, launches, _ = timed_pass(args.steps, use_flush, False)
    barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # the tables of the last timed step, as kb_download hands them to a caller of the resident path
        last = evs[(args.steps - 1) % len(evs)].download(snap, abi.CycleOut(snap))
        dump_outputs(args.dump_outputs, cycle_tables(last))
    # per-kernel split (roofline.kernel_ms): the same K steps once more with an event before every kernel; not part of
    # `value` (the extra event records sit between the kernels of the timed stream)
    _, _, kms = timed_pass(args.steps, use_flush, True)
    # the other methodology, for comparison
    alt_ms = None
    if not use_flush and world == 1:
        timed_pass(3, True, False)
        alt_ms = timed_pass(args.steps, True, False)[0] / args.steps
    for e2 in evs[1:]:
        e2.close()
    evs = [ev]

    # ---- end-to-end through the C-ABI with host buffers (e2e) ----
    # steady state of the controller: ClusterQueue / Cohort specs do not change between cycles, so the shim keeps
    # static_generation constant and only usage + entries + admitted workloads cross PCIe every cycle.
    snap.static_generation = 1
    # N > 1: the shards' decisions travel to every rank (one NCCL all-gather of H bytes per rank, padded to the largest
    # shard) and rank 0 scatters them to their global entry positions (shard.merge for the decision table).  Root
    # cohorts never interact, so a rank's next cycle does not wait for the merge: a write-back thread gathers and merges
    # the decisions of cycle k while cycle k+1 runs (the timed region ends when the last merge is done).
    merged = {"n": 0, "full": None}
    if world > 1:
        import queue
        sizes = [None] * world
        dist.all_gather_object(sizes, my_heads)
        all_maps = sizes
        hmax = max(len(m) for m in all_maps)
        contiguous = all(len(m) == hmax and m[0] == r * hmax and m[-1] == (r + 1) * hmax - 1 for r, m in enumerate(all_maps))
        side = torch.cuda.Stream()
        mine_host = torch.zeros(hmax, dtype=torch.uint8).pin_memory()
        mine_dev = torch.zeros(hmax, dtype=torch.uint8, device="cuda")
        all_dev = torch.empty(world * hmax, dtype=torch.uint8, device="cuda")
        all_host = torch.empty(world * hmax, dtype=torch.uint8).pin_memory()
        full = np.zeros(glob_heads, np.uint8)
        q = queue.Queue()

        def writer():
            torch.cuda.set_device(local_rank)
            while True:
                dec = q.get()
                if dec is None:
                    return
                with torch.cuda.stream(side):
                    mine_host[:len(dec)] = torch.from_numpy(dec)
                    mine_dev.copy_(mine_host, non_blocking=True)
                    dist.all_gather_into_tensor(all_dev, mine_dev)
                    if rank == 0:
                        all_host.copy_(all_dev, non_blocking=True)
                side.synchronize()
                if rank == 0:
                    host = all_host.numpy()
                    if contiguous:
                        full[:] = host
                    else:
                        for r in range(world):
                            full[all_maps[r]] = host[r * hmax:r * hmax + len(all_maps[r])]
                    merged["full"] = full
                merged["n"] += 1
                q.task_done()

    def e2e_steps(n):
        if world == 1:
            for _ in range(n):
                ev.run_cycle(snap, out)
            return
        th = threading.Thread(target=writer, daemon=True)
        th.start()
        for _ in range(n):
            ev.run_cycle(snap, out)
            q.put(np.array(out.decision, copy=True))
        q.put(None)
        th.join()

    e2e_steps(2)
    barrier()
    t0 = time.perf_counter()
    e2e_steps(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    st = ev.stats()
    h2d, d2h = int(st.h2d_bytes), int(st.d2h_bytes)

    # ---- the same with incremental usage (kb_snapshot.usage_delta_*, SURVEY f2): the usage table stays on the device and
    # every step carries only the rows of the ClusterQueues that admitted a workload in this cycle (the rows the cache
    # would have touched); their values are unchanged, so every step still evaluates the same snapshot.  Reported next to
    # `e2e` (which keeps moving the whole table), never instead of it.
    inc_line = None
    if world == 1 and args.config == 3:
        import copy
        admitted = np.flatnonzero(np.asarray(out.decision) == 5)  # KB_DEC_ASSUMED
        dirty = np.unique(np.asarray(snap.wl_cq)[np.asarray(snap.heads)[admitted]]).astype(np.int32)
        usage = np.asarray(snap.cq_usage).reshape(snap.n_cq, snap.n_fr)
        seed = copy.copy(snap); seed.arrays = dict(snap.arrays); seed._struct = None
        seed.flags = snap.flags | abi.F_USAGE_RESIDENT
        ev.run_cycle(seed, out)  # leaves the table resident (same static_generation)
        inc = abi.FlatSnapshot(n_cq=snap.n_cq, n_cohort=snap.n_cohort, n_flavor=snap.n_flavor, n_resource=snap.n_resource,
                               pods_resource=snap.pods_resource, flags=snap.flags, now_ns=snap.now_ns)
        inc.arrays = {k: v for k, v in snap.arrays.items() if k != "cq_usage"}
        inc.arrays["cq_usage"] = np.zeros(0, np.int64)
        inc.set("usage_delta_cq", dirty); inc.set("usage_delta_rows", usage[dirty])
        inc = native.pin_snapshot(inc); inc.static_generation = snap.static_generation
        for _ in range(2):
            ev.run_cycle(inc, out)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ev.run_cycle(inc, out)
        inc_s = time.perf_counter() - t0
        sti = ev.stats()
        inc_line = {"value": snap.n_heads * args.steps / inc_s, "unit": UNIT, "h2d_bytes_per_step": int(sti.h2d_bytes), "d2h_bytes_per_step": int(sti.d2h_bytes),
                    "usage_rows_per_step": int(len(dirty)), "of_rows": int(snap.n_cq),
                    "what": "kb_snapshot.usage_delta_*: rows of the ClusterQueues that admitted in this cycle; the rest of the usage table stays on the device"}

    t = torch.tensor([dev_ms, e2e_s, float(snap.n_heads)], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, total_dec = tmax[0].item(), tmax[1].item(), tsum[2].item()
    else:
        total_dec = float(snap.n_heads)
    if rank == 0:
        ms_per_step = dev_ms / args.steps
        value = total_dec / (ms_per_step / 1e3)
        e2e = total_dec * args.steps / e2e_s
        ab = algorithmic_bytes(snap)
        top = int(np.argmax(kms))
        top_ms = kms[top] / args.steps
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        kname = abi.KERNEL_NAMES[top]
        kbytes = ab.get(kname, ab["total"])
        ss = list(st.search_stat)
        if kname in ("k_search_cells", "k_nominate_walk"):
            # streamed 32 B candidate records of the last cycle (kb_stats.search_stat: [1] all records, [4] those of the
            # multi-column GetTargets searches of k_nominate_walk) on top of the per-entry floor; the quota columns a
            # search stages are shared by the searches of one bucket and are part of the floor's node tables
            multi = ss[4]
            kbytes = float((ss[1] - multi) * 32 + ab[kname]) if kname == "k_search_cells" else float(multi * 32 + ab[kname])
        achieved = kbytes / (top_ms / 1e3) / 1e9 if top_ms > 0 else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.config], "heads": "all pending workloads (batched evaluator)" if HEADS[args.config] == "all" else "one head per ClusterQueue (reference cycle)",
                       "decisions_per_step_per_gpu": snap.n_heads,
                       "l2": ("512 MiB flush buffer written between timed steps" if use_flush else
                              f"inputs larger than L2: {n_copies} device-resident copies of the snapshot ({copy_bytes / 1e6:.1f} MB each, static tables included), "
                              f"timed steps walk them round-robin; with a 512 MiB flush before every step instead (evicts the kernel code as well): "
                              + (f"{alt_ms:.4f} ms/step" if alt_ms else "n/a")),
                       "timing": "CUDA events on the library stream around the cycle's kernels, summed over steps, max over ranks; kernel_ms_per_step from a second pass of the same steps with an event before every kernel",
                       "wall_ms_per_step_incl_flush": wall_ms / args.steps,
                       "e2e_static_tables": "quota / policy / topology tables uploaded once (static_generation constant), "
                                            "usage + entries + admitted workloads copied every step",
                       "multi_gpu": None if world == 1 else {"partition": ("the configuration's root cohorts split over the ranks (kueue_b200.shard)" if scaling == "strong" else
                                                                           "one independent copy of the configuration (its own root cohorts) per rank") + ", no data-path collective",
                                                             "e2e_includes": "NCCL all-gather of the shards' decisions + merge on rank 0, pipelined one cycle behind by a write-back thread (shards never interact)",
                                                             "host_affinity": numa}},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches,
            "search_counters": ({"searches": ss[0], "records_classified": ss[1], "candidates_visited": ss[2], "workloads_removed": ss[3],
                                 "records_of_multi_column_searches": ss[4]} if kms[abi.KERNEL_NAMES.index("k_nominate_walk")] > 0 else None),
            "kernel_ms_per_step": {abi.KERNEL_NAMES[i]: kms[i] / args.steps for i in range(20) if kms[i] > 0},
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": measured_traffic(args.config, kname),
                         "algorithmic_bytes_per_launch": kbytes, "kernel_ms": top_ms,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"},
        }
        if inc_line:
            line["e2e_incremental"] = inc_line
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(snap)
        if world == 1 and args.config in (2, 3) and not args.no_drain:
            line["drain"] = drain_line(ev, args.config, cpu=not args.no_cpu_baseline)
        print(json.dumps(line))
    ev.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
