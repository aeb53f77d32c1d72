#!/usr/bin/env python
"""bench.py — gossip edge-updates/s of the hot path on BASELINE.json's 10 M-node workload.

One STEP = one complete dissemination study on the resident cluster: reset to the bootstrap state, schedule the host
operations (SURVEY §8d item 4: one leave-intent + one fail at tick 0), run gossip ticks until the cluster is quiescent
(serfsim_run_until_converged).  `value` = edge-updates of all ranks ÷ wall time of K whole steps between two
barrier + synchronize brackets (max over ranks), inputs resident in HBM.  `e2e` = the same K studies driven through the C ABI
with HOST buffers: the operation schedule goes host→device and the member-status, status-time and Lamport-clock vectors of
every tracked subject come back device→host into pinned buffers inside the timed region (serfsim_results_async: the copies of
study k overlap the ticks of study k+1, the region ends when the last copy has landed).

Every step is CHECKED: convergence tick, edge-updates, messages, changed records and the final state hash must equal the CPU
oracle's run of the same workload (made once, outside the timed regions, on hosts with enough cores).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
           --master-port 29500 bench.py --gpus 8 --steps 5 --warmup 3
    python bench.py --impl reference          # the CPU oracle (port of the reference path) on the host cores
    python bench.py --dump-outputs out/       # also write what the last timed step computed to out/*.npy (see dump_outputs)
"""
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

METRIC = "gossip edge-updates/sec @10M nodes"
UNIT = "edge-updates/s"
HBM_FALLBACK_GBS = 6650.0          # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def make_scenario(args, nodes=None):
    from serf_b200 import scenarios
    n = nodes or args.nodes
    if args.workload == "leave_fail":
        return scenarios.dissemination_storm(n, args.degree, args.fanout, slots=max(2, args.slots), seed=1, waves=args.waves, with_fail=True)
    return scenarios.dissemination_storm(n, args.degree, args.fanout, slots=args.slots, seed=1, waves=args.waves)


def scenario_name(args):
    slots = max(2, args.slots) if args.workload == "leave_fail" else args.slots
    return f"storm_{args.nodes}_d{args.degree}_f{args.fanout}_r{slots}_w{args.waves}" + ("_fail" if args.workload == "leave_fail" else ""), slots


def config_dict(args, name, slots):
    what = ("one tracked subject leaves and one crashes at tick 0 (SURVEY §8d item 4: leave-intent + fail; probe / suspicion timers / dead inside the run)"
            if args.workload == "leave_fail" else f"{slots} tracked subject(s) leave at tick 0")
    return {"workload": f"configs[3] shape: {args.nodes}-node random graph (out-degree {args.degree}), fanout={args.fanout}, {what}, run to quiescence",
            "scenario": name, "nodes": args.nodes, "degree": args.degree, "fanout": args.fanout, "slots": slots,
            "retransmit_mult": 4, "cache": "member records (%d MB) + CSR (%d MB) exceed the 126 MB L2; no flush needed"
            % (args.nodes * 32 * slots // 2**20, args.nodes * args.degree * 4 // 2**20)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe).  nvidia-smi needs ~1 s to start, so it is
    launched before the warm-up; samples are time-stamped and only those inside [mark_begin, mark_end] — the timed
    regions — are summarised (all samples under load if the window caught none)."""

    QUERY = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()

        def summarise(rows):
            sm, mx, reasons = [], [], set()
            for _, r in rows:
                try:
                    sm.append(float(r[1])); mx.append(float(r[2]))
                except (ValueError, IndexError):
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons
        inside = [x for x in self.rows if self.t0 is not None and self.t0 <= x[0] <= (self.t1 or 1e30)]
        window = "timed regions"
        if not inside:
            inside, window = self.rows, "warm-up + timed regions (no sample fell inside the timed window)"
        sm, mx, reasons = summarise(inside)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def b_edge(fanout, p_dirty):
    """ALGORITHMIC bytes per edge-update (SURVEY.md §8d): edge index + amortised source record +
    destination record read + destination write-back when the merge changed it."""
    return 4.0 + 32.0 / fanout + 32.0 + 32.0 * p_dirty


# ---- the CPU oracle (test infrastructure): the checker of every step and the timed CPU baseline ----------------------
_ALL_CPUS = None                                         # taken before the driver thread is bound to the GPU's NUMA node


def physical_cpus():
    """One logical CPU per physical core of the cores this process may use, alternating between packages (NUMA nodes) so
    that consecutive oracle workers — which own consecutive id ranges — land on alternating memory controllers."""
    if _ALL_CPUS is not None:
        return _ALL_CPUS
    allowed = sorted(os.sched_getaffinity(0))
    by_pkg = {}
    for c in allowed:
        try:
            core = int(open(f"/sys/devices/system/cpu/cpu{c}/topology/core_id").read())
            pkg = int(open(f"/sys/devices/system/cpu/cpu{c}/topology/physical_package_id").read())
        except (OSError, ValueError):
            core, pkg = c, 0
        by_pkg.setdefault(pkg, {}).setdefault(core, c)
    lists = [list(v.values()) for _, v in sorted(by_pkg.items())]
    out = []
    for i in range(max(len(x) for x in lists)):
        out += [x[i] for x in lists if i < len(x)]
    return out


_ORACLE_CACHE = {}


def oracle_handle(args, nodes):
    """The oracle on the workload at `nodes` nodes: one worker per physical core, pinned (unpinned workers over every
    hyperthread varied 5x between two boxes in round 1).  Built once and reused."""
    import ctypes
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import lib, oracle_sim
    if nodes not in _ORACLE_CACHE:
        cpus = physical_cpus()
        sc = make_scenario(args, nodes)
        o = oracle_sim(sc.n, sc.slots, **sc.cfg)
        L = lib()
        L.oracle_sim_set_threads.restype, L.oracle_sim_set_threads.argtypes = ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]
        L.oracle_sim_set_affinity.restype, L.oracle_sim_set_affinity.argtypes = ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_int]
        assert L.oracle_sim_set_threads(o._h, len(cpus)) == 0
        arr = (ctypes.c_int * len(cpus))(*cpus)
        assert L.oracle_sim_set_affinity(o._h, arr, len(cpus)) == 0
        o.set_topology(sc.row_ptr, sc.col); o.set_subjects(sc.subjects)
        _ORACLE_CACHE[nodes] = (sc, o, len(cpus))
    return _ORACLE_CACHE[nodes]


def oracle_run(args, nodes):
    """One reset + schedule + run to quiescence of the oracle; returns timing and the totals the GPU steps are checked against."""
    sc, o, cores = oracle_handle(args, nodes)
    t0 = time.perf_counter()
    o.reset(sc.cfg.get("seed", 1)); sc.schedule(o)
    ticks, ok = o.run_until_converged(sc.max_ticks)
    dt = time.perf_counter() - t0
    st = o.stats()
    return {"seconds": dt, "ticks": ticks, "ok": bool(ok), "edge_updates": st["edge_updates"], "messages": st["messages"], "changed": st["changed"],
            "packets": st["packets"], "state_hash": int(o.state_hash()), "cores": cores, "nodes": nodes}


def time_oracle(args, nodes, repeats=3):
    """CPU baseline: median of `repeats` oracle runs on a bounded sample of the workload."""
    runs = [oracle_run(args, nodes) for _ in range(repeats)]
    runs.sort(key=lambda r: r["seconds"])
    r = runs[len(runs) // 2]
    return {"value": r["edge_updates"] / r["seconds"], "unit": UNIT, "cores": r["cores"], "kind": "port",
            "sample": f"same scenario at {nodes} nodes ({nodes / args.nodes:.3g} of the workload), full run to quiescence ({r['ticks']} ticks, "
                      f"{r['edge_updates']} edge-updates), median of {repeats} runs ({r['seconds']:.2f} s; min {runs[0]['seconds']:.2f}, max {runs[-1]['seconds']:.2f}); "
                      f"one pinned worker per physical core", "seconds": r["seconds"], "ticks": r["ticks"]}


DUMP_BYTES = 64 << 20                                    # --dump-outputs: all files together stay below this
DUMP_SEED = 20240601                                     # fixed: the same node ids are sampled on every run


def dump_outputs(outdir, sc, g, read_back, ticks, ok, gather):
    """Write what the last timed step computed, as a caller of the path receives it, to outdir/<name>.npy (float64: every value is
    an integer below 2**53).  Per-node vectors come from the end-to-end read-back and are sampled at the same node ids on every run:
      node_ids                      the sampled node ids (ascending)
      member_status_slot<s>         MemberStatus of tracked subject s in each sampled node's view
      status_ltime_slot<s>          its status Lamport time
      lamport_time                  each sampled node's Lamport clock
      convergence                   [tick of quiescence, 1 if converged]
      stats                         serfsim_stats_t in field order (Stats._fields_)
      state_hash                    [high 32 bits, low 32 bits] of the final state hash
    Every rank takes part (stats, state hash and the gather are collective); rank 0 writes."""
    from serf_b200 import Stats
    per_node = 2 + 2 * sc.slots                          # node id, clock, status and status time per slot
    k = min(sc.n, 1 << 20, (DUMP_BYTES - (1 << 16)) // (8 * per_node))
    ids = np.sort(np.random.default_rng(DUMP_SEED).choice(sc.n, size=k, replace=False))
    mine = ids[(ids >= g.first) & (ids < g.first + g.count)]
    at = mine - g.first
    local = {"node_ids": mine, "lamport_time": read_back["clock"].numpy().view(np.uint32)[at]}
    for s in range(sc.slots):
        local[f"member_status_slot{s}"] = read_back["status"][s].numpy()[at]
        local[f"status_ltime_slot{s}"] = read_back["ltime"][s].numpy().view(np.uint32)[at]
    st, h = g.stats(), int(g.state_hash())
    parts = gather(local)
    if parts is None:
        return
    out = {name: np.concatenate([p[name] for p in parts]) for name in local}
    assert (out["node_ids"] == ids).all()
    out["convergence"] = np.array([ticks, int(ok)])
    out["stats"] = np.array([st[name] for name, _ in Stats._fields_])
    out["state_hash"] = np.array([h >> 32, h & 0xFFFFFFFF])
    os.makedirs(outdir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(outdir, name + ".npy"), a.astype(np.float64))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nodes = args.ref_nodes or min(args.nodes, 2_000_000)          # bounded sample: K + W oracle runs must end within minutes
    vals = []
    for i in range(args.warmup + args.steps):
        r = oracle_run(args, nodes)
        if i >= args.warmup:
            vals.append(r)
    total_eu = sum(r["edge_updates"] for r in vals)
    total_s = sum(r["seconds"] for r in vals)
    v = total_eu / total_s
    secs = sorted(r["seconds"] for r in vals)
    sample = (f"same scenario at {nodes} nodes ({nodes / args.nodes:.3g} of the workload), every step a full run to quiescence ({vals[-1]['ticks']} ticks, "
              f"{vals[-1]['edge_updates']} edge-updates; {secs[len(secs) // 2]:.2f} s median, {secs[0]:.2f}–{secs[-1]:.2f} s); one pinned worker per physical core")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total_s / max(1, len(vals)), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic", "config": config_dict(args, *scenario_name(args)),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": vals[-1]["cores"], "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nodes", type=int, default=10_000_000)
    ap.add_argument("--degree", type=int, default=16)
    ap.add_argument("--fanout", type=int, default=4)
    ap.add_argument("--slots", type=int, default=1)
    ap.add_argument("--waves", type=int, default=1)
    ap.add_argument("--workload", default="leave_fail", choices=["leave_fail", "leave"],
                    help="leave_fail: SURVEY §8d item 4 (one subject leaves, one crashes; 2 tracked subjects); leave: the round-1 workload (1 subject leaves)")
    ap.add_argument("--ref-nodes", type=int, default=0, help="size of the bounded CPU sample (0: 1 M nodes inside the b200 arm, 2 M in the reference arm)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="A/B: leave the driver thread where the OS scheduler puts it")
    ap.add_argument("--no-check", action="store_true", help="skip the full-size oracle run every step is checked against")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                                                          "(a fixed sample of the per-node results, at most 64 MB; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")
    if args.warmup < 3:
        args.warmup = 3

    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from serf_b200 import GossipSim

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    global _ALL_CPUS
    _ALL_CPUS = physical_cpus()                          # the oracle's workers keep the whole machine (they pin themselves, one per physical core)
    from serf_b200 import bind_thread_near_gpu
    near = None if args.no_numa_bind else bind_thread_near_gpu(local_rank)   # the driver thread and its pinned buffers: the GPU's own NUMA node
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sc = make_scenario(args)
    g = sc.build(lambda n, s, **kw: GossipSim(n, s, **kw), device=local_rank, rank=rank, world_size=world, trace=0)
    if world > 1:
        from serf_b200 import dist as sdist
        sdist.connect(g, dist, torch.device("cuda", local_rank))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- what every step must reproduce: the oracle's run of the same workload (rank 0, outside the timed regions) ----
    expect = None
    cores = len(physical_cpus())
    if not args.no_check and rank == 0 and (cores >= 16 or args.nodes <= 2_000_000):
        e = oracle_run(args, args.nodes)
        expect = {k: e[k] for k in ("ticks", "ok", "edge_updates", "messages", "changed", "packets", "state_hash")}
        expect["oracle_seconds"] = e["seconds"]
    if world > 1:
        box = [expect]
        dist.broadcast_object_list(box, src=0)
        expect = box[0]
    checked = {"steps": 0}

    def check_step(ticks, ok):
        """Convergence tick and totals of this step against the oracle (stats / state_hash are collective when sharded)."""
        if expect is None:
            return
        st = g.stats()
        got = {"ticks": int(ticks), "ok": bool(ok), "edge_updates": st["edge_updates"], "messages": st["messages"], "changed": st["changed"], "packets": st["packets"],
               "state_hash": int(g.state_hash())}
        bad = {k: (got[k], expect[k]) for k in got if got[k] != expect[k]}
        if bad:
            raise SystemExit(f"bench self-check FAILED on rank {rank}: (gpu, oracle) {bad}")
        checked["steps"] += 1

    # pinned host buffers for the results a caller reads back (the C ABI copies into caller-owned memory); two sets: the copies of
    # study k overlap the ticks of study k+1
    def pinned_set():
        return {"status": [torch.empty(g.count, dtype=torch.uint8).pin_memory() for _ in range(sc.slots)],
                "ltime": [torch.empty(g.count, dtype=torch.int32).pin_memory() for _ in range(sc.slots)],     # Lamport times cross PCIe as u32
                "clock": torch.empty(g.count, dtype=torch.int32).pin_memory()}
    pins = [pinned_set(), pinned_set()]

    def one_step(read_back=None):
        g.reset(1)
        sc.schedule(g)                                 # host→device: the operation schedule
        ticks, ok = g.run_until_converged(sc.max_ticks)
        ms, launches = g.last_step_device_ms()
        out_bytes = 0
        if read_back is not None:                      # device→host: the step's result vectors (asynchronous: see the module docstring)
            for s in range(sc.slots):
                out_bytes += g.results_async(s, status=read_back["status"][s].numpy(), status_ltime=read_back["ltime"][s].numpy().view(np.uint32),
                                             lamport=read_back["clock"].numpy().view(np.uint32) if s == 0 else None)
        return ticks, ok, ms, launches, out_bytes

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        t, ok, *_ = one_step()
        check_step(t, ok)
    time.sleep(1.2)                                      # let nvidia-smi come up before the timed regions (all ranks: steps are collective)
    for k in range(4):                                   # … and the read-back path: staging buffers, copy stream and events are created on first use,
        one_step(pins[k & 1])                            # all four ring entries once (device allocations inside the timed region cost up to 15 ms per step)
    g.results_wait()

    # ---- device-timed region: K steps ----
    sync_all()
    sampler.mark_begin()
    dev_ms, launches, ticks_list = 0.0, 0, []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ticks, ok, ms, nl, _ = one_step()
        dev_ms += ms; launches += nl; ticks_list.append((ticks, ok))
    sync_all()
    wall_dev = time.perf_counter() - t0
    st = g.stats()                                       # global sums (all ranks) of the LAST step
    eu_per_step, changed = st["edge_updates"], st["changed"]
    for (t, ok) in ticks_list:                           # every timed step converged where the oracle does; the last one is compared in full
        if expect is not None and (int(t), bool(ok)) != (expect["ticks"], expect["ok"]):
            raise SystemExit(f"bench self-check FAILED: a timed step converged at {(t, ok)}, oracle {(expect['ticks'], expect['ok'])}")
    check_step(*ticks_list[-1])

    # ---- end-to-end region: host buffers in, host buffers out ----
    sync_all()
    t0 = time.perf_counter()
    d2h = 0
    for k in range(args.steps):
        last_ticks, last_ok, _, _, ob = one_step(pins[k & 1])
        d2h = ob
    g.results_wait()                                     # the last copies have landed in host memory
    sync_all()
    wall_e2e = time.perf_counter() - t0
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    if expect is not None:                               # the vectors that came back are the converged ones: every other node sees the leaver as Left
        from serf_b200 import MemberStatus
        stv = pins[(args.steps - 1) & 1]["status"][0].numpy()
        lo, hi = g.first, g.first + g.count
        subj = int(sc.subjects[0])
        others = np.delete(stv, subj - lo) if lo <= subj < hi else stv
        if int((others != MemberStatus.LEFT).sum()) > 8:
            raise SystemExit("bench self-check FAILED: the status vector read back end to end is not the converged one")
    if args.dump_outputs:                                # the last end-to-end step: its read-back is what a caller receives
        def gather(local):
            if world == 1:
                return [local]
            parts = [None] * world
            dist.all_gather_object(parts, local)
            return parts if rank == 0 else None
        dump_outputs(args.dump_outputs, sc, g, pins[(args.steps - 1) & 1], last_ticks, last_ok, gather)

    t = torch.tensor([dev_ms, wall_e2e, wall_dev], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, wall_e2e, wall_dev = [float(x) for x in t.cpu()]

    if rank == 0:
        total_eu = eu_per_step * args.steps
        value = total_eu / wall_dev                    # K whole steps (reset + schedule + ticks), sync to sync
        p_dirty = changed / max(1, eu_per_step)
        be = b_edge(args.fanout, p_dirty)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"
        tick_launches = launches                       # kernels of the executed ticks (tick kernels ≥ 98 % of them; launches past the quiescent tick return at once and are not counted)
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", f"r2_traffic_{args.workload}.json")      # ncu capture of THIS workload with the shipped kernel
        if world == 1 and os.path.exists(tpath):
            tj = json.load(open(tpath))
            # DRAM bytes of ONE run of this workload (every tick_kernel launch of the capture) over the launches of one bench step: the same
            # denominator as algorithmic_bytes_per_launch (launches that return at once — gated ticks, the idle half of a dual launch — count in both)
            traffic = (tj.get("dram_bytes_read", 0.0) + tj.get("dram_bytes_write", 0.0)) / max(1.0, launches / args.steps)
            traffic_src = f"{os.path.relpath(tpath, ROOT)} (ncu dram__bytes_read.sum + dram__bytes_write.sum over all tick_kernel launches of one run, per launch of a bench step; {tj.get('source', '')})"
        # per-GPU: each GPU runs its own tick kernel over its shard; algorithmic bytes split evenly
        achieved = (total_eu / world) * be / (dev_ms * 1e-3) / 1e9
        h2d = len(sc.ops) * 12
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * wall_dev / args.steps, "kernel_ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u32", "data": "synthetic", "config": config_dict(args, sc.name, sc.slots),
                "ticks_to_convergence": ticks_list[-1][0], "edge_updates_per_step": eu_per_step, "p_dirty": p_dirty,
                "self_check": ({"against": "CPU oracle, same workload at full size", "steps_checked_in_full": checked["steps"], "timed_steps_convergence_checked": args.steps,
                                "fields": ["ticks", "ok", "packets", "edge_updates", "messages", "changed", "state_hash"], "oracle_seconds": expect["oracle_seconds"]}
                               if expect is not None else f"skipped ({'--no-check' if args.no_check else str(cores) + ' host cores'})"),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_src,
                             "algorithmic_bytes_per_launch": total_eu * be / world / max(1, tick_launches), "peak_source": peak_src, "kernel": "tick_kernel", "bytes_per_edge_update": be,
                             "launches": tick_launches, "avg_launch_us": 1e3 * dev_ms / max(1, tick_launches),
                             "note": "achieved = algorithmic bytes of the step / device time of the step (CUDA events on the launch stream around all its tick launches, idle timer-wait ticks included)"},
                "e2e": {"value": total_eu / wall_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": 1e3 * wall_e2e / args.steps},
                "gpu_launches": launches, "clocks": clocks,
                "host": {"driver_thread_cpus": (f"{len(near)} CPUs of the GPU's NUMA node" if near else "unbound")}}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = {k: v for k, v in time_oracle(args, args.ref_nodes or 1_000_000).items() if k not in ("seconds", "ticks")}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
