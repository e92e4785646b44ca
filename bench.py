#!/usr/bin/env python
"""bench.py — task x worker cost evaluations per second on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg1..cfg5]
                    [--dump-outputs DIR]

One *step* is one management pass (pm_match: cost-matrix build -> argmin ->
resolution sweep) over one synthetic swarm.  N=1 workload: BASELINE configs[2],
the configuration the north-star target is quoted on: 100k asks x 1M workers (the
800 GB int64 cost matrix is streamed through HBM in 8 GiB tiles, so every step's
working set is far larger than L2).  N>1: BASELINE configs[4]'s per-GPU shape —
1M asks x 1M workers per GPU, Zipf-priced workers, 10 % infeasible asks; exactly
configs[4] (1M x 8M) at N=8 — workers range-sharded, one process per GPU
(torchrun); the one data-path exchange per pass is a packed all-gather INSIDE the
library (pm_comm: NCCL resolved at run time); nothing in the step calls
torch.distributed.

Prints ONE JSON line (rank 0).  `value` is device-resident throughput; `e2e`
goes through the C ABI with host (pinned) tables: H2D of asks+workers and D2H of
the assignment inside the timed region.  `--impl reference` times the CPU
oracle (the reference's scheduler restated; the Rust reference cannot be built
here) on the box's host cores on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step computed, as DIR/<name>.npy
in float64 (every value exact), so that two builds can be compared output for
output on the same seeded inputs; see dump_outputs().
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

METRIC = "task_x_worker_cost_evaluations_per_sec"
UNIT = "evals/s"
DATA = "synthetic (splitmix64, seeds 0xB2000001 workers / 0xB2000002 asks / 0xB2000003 prices)"

WORKLOADS = {
    # name: (n_asks, n_workers_per_gpu, ask kind, description)
    "cfg1": (1_000, 10_000, "uniform1", "1k asks x 10k workers, uniform single-GPU asks"),
    "cfg2": (100_000, 100_000, "mixed", "100k asks x 100k workers, mixed {1,2,4,8}-GPU asks"),
    "cfg3": (100_000, 1_000_000, "mixed", "100k asks x 1M workers, mixed asks, log-uniform worker prices + ask price caps (auction columns)"),
    # multi-GPU shapes of BASELINE configs[3]/[4] (workers sharded; run with --gpus 4 / --gpus 8)
    "cfg4": (1_000_000, 250_000, "mixed", "1M asks x 250k workers per GPU (1M x 1M over 4 GPUs), mixed asks"),
    "cfg5": (1_000_000, 1_000_000, "skewed", "1M asks x 1M workers per GPU (1M x 8M over 8 GPUs), Zipf(1.1) worker prices, 10% infeasible asks"),
}
PRICES = {"cfg3": "loguniform", "cfg5": "zipf"}
DUMP_BYTES = 64_000_000         # --dump-outputs: bytes written at most, .npy headers included
DUMP_SEED = 0xB2000004          # positions kept when the outputs are larger than that


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Write each integer array as out_dir/<name>.npy in float64, which holds every u32 / i32 value exactly.  When the
    whole would exceed `budget`, every array longer than its share keeps the same seeded positions from run to run
    (the positions go to <name>_index.npy), so two runs on the same inputs stay comparable element for element."""
    arrays = dict(arrays)
    if sum(a.size for a in arrays.values()) * 8 + 128 * len(arrays) > budget:
        share = (budget - 2 * 128 * len(arrays)) // 8 // (2 * len(arrays))     # values + positions per array
        for name, a in list(arrays.items()):
            if a.size > share:
                idx = np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, share, replace=False))
                arrays[name], arrays[name + "_index"] = a[idx], idx
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a).astype(np.float64))


def split_best(best):
    """Packed cost<<32 | worker keys as two arrays: float64 holds each half exactly, but not the packed int64."""
    best = np.asarray(best, dtype=np.int64)
    return {"ask_best_cost": best >> 32, "ask_best_worker": best & 0xFFFFFFFF}


def host_cpus():
    """Cores this process may actually run on: the affinity mask, cut by the cgroup CPU quota when there is one."""
    aff = len(os.sched_getaffinity(0))
    quota = None
    for path, parse in (("/sys/fs/cgroup/cpu.max", lambda t: None if t.split()[0] == "max" else float(t.split()[0]) / float(t.split()[1])),):
        try:
            quota = parse(open(path).read())
        except Exception:
            pass
    if quota is None:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            quota = q / per if q > 0 else None
        except Exception:
            pass
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return {"threads": eff, "affinity": aff, "cgroup_quota_cpus": quota, "os_cpu_count": os.cpu_count()}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_tables(workload: str, n_gpus: int, n_models: int = 0):
    from protocol_b200 import synth

    T, Wg, kind, desc = WORKLOADS[workload]
    W = Wg * n_gpus
    # --models N: a permissionless pool's free-form model strings (node.rs:463-484) instead of the 16-entry catalogue;
    # more than 31 distinct ones puts a per-worker acceptance word in shared memory (BITS=1), more than the shared-memory
    # table holds leaves it in global memory (BITS=0)
    cat = synth.wide_model_catalogue(n_models) if n_models else None
    w = synth.make_workers(W, price=PRICES.get(workload), catalogue=cat)
    a = synth.make_asks(T, kind)
    bits, npat, nmod, words = synth.intern_tables(w, a)
    return w, a, (bits, npat, nmod, words), (T, W, Wg, desc)


def config_dict(args, desc, T, W, Wg, world):
    """The workload, identical in both arms (the driver compares them); arm-specific detail goes under `detail`."""
    return {"workload": f"{args.workload}: {desc}" + (f", {args.models} distinct worker model strings" if args.models else ""),
            "n_asks": T, "n_workers": W, "workers_per_gpu": Wg,
            "mode": "first_fit (try_form_new_groups)", "cost_tile_gib": args.tile_gib,
            "l2": "inputs larger than L2: each step streams the int64 cost matrix "
                  f"({T * Wg * 8 / 1e9:.0f} GB per GPU) through HBM in {args.tile_gib} GiB tiles",
            "parallelism": (f"worker-sharded x{world}, one packed all-gather per pass inside the library (pm_comm)"
                            if world > 1 else "single GPU"),
            "scaling_note": "N=1 runs BASELINE configs[2] (100k asks x 1M workers); N>1 runs configs[4]'s per-GPU shape "
                            "(1M asks x 1M workers per GPU; exactly configs[4] at N=8): evals/s is work-normalised, "
                            "per-GPU work is fixed for N>=2"}


# ----------------------------------------------------------------------------- reference arm
def run_reference(args):
    """CPU oracle on the host cores: all-pairs evaluation of a bounded sample, all threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pm_oracle as orc

    w, a, (bits, npat, nmod, words), (T, W, Wg, desc) = make_tables(args.workload, max(args.gpus, 1), args.models)
    cpus = host_cpus()
    cores = cpus["threads"]
    # bounded sample: a band of asks against every worker, ~2e9 pair evaluations per step at most
    sample_rows = max(1, min(T, int(2.0e9 // max(W, 1)), 20_000))
    t0 = (T - sample_rows) // 2

    def step():
        return orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, t0, t0 + sample_rows, 0, W,
                                   threads=cores, want_rows=True, want_cols=True)

    for _ in range(args.warmup):
        step()
    t_start = time.perf_counter()
    evals = 0
    for _ in range(args.steps):
        last = step()
        evals += last["evals"]
    dt = time.perf_counter() - t_start
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**split_best(last["row_best"]), "ask_count": last["row_count"],
                                         "worker_first_ask": last["col_first"]})
    value = evals / dt
    # the faithful loop (string/AoS, re-filter per group) on a small sample, single thread
    faithful = faithful_sample(orc, w, a)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 predicate -> int64 packed cost",
        "data": DATA,
        "config": config_dict(args, desc, T, W, Wg, max(args.gpus, 1)),
        "detail": {"path": "cpu (oracle/pm_oracle.cpp, SoA restatement, all pairs)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "host_cpus": cpus,
                         "sample": f"asks [{t0},{t0 + sample_rows}) x all {W} workers, all pairs, {cores} threads",
                         "faithful_single_thread": faithful},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference = C++ restatement of crates/orchestrator node_groups scheduler (Rust toolchain absent); "
                "Redis/JSON/HTTP time of the real orchestrator excluded",
    }
    print(json.dumps(line), file=RESULT_OUT, flush=True)


def faithful_sample(orc, w, a, n_nodes=4000, n_cfgs=400):
    """orc_form_groups (AoS + strings + per-group re-filter) on a prefix; evals/s of its own counter."""
    from protocol_b200 import abi

    nodes = []
    keep = []
    for i in range(min(n_nodes, len(w.a))):
        f = int(w.a["flags"][i])
        has = lambda b: bool(f & b)
        nodes.append(orc.make_node(
            address=f"0x{i:040x}", status=int(w.status[i]), p2p=has(abi.PM_W_P2P), specs=has(abi.PM_W_HAS_SPECS),
            gpu_count=int(w.a["gpu_count"][i]) if has(abi.PM_W_HAS_GPU_COUNT) else None,
            gpu_model=w.model_strings[int(w.a["model_id"][i])] if has(abi.PM_W_HAS_GPU_MODEL) else None,
            gpu_mem=int(w.a["gpu_mem_mb"][i]) if has(abi.PM_W_HAS_GPU_MEM) else None,
            cpu_cores=int(w.b["cpu_cores"][i]) if has(abi.PM_W_HAS_CPU_CORES) else None,
            ram=int(w.b["ram_mb"][i]) if has(abi.PM_W_HAS_RAM) else None,
            storage=int(w.b["storage_gb"][i]) if has(abi.PM_W_HAS_STORAGE) else None))
    reqs = [orc.Req(a.requirement_string(t)) for t in range(min(n_cfgs, len(a)))]
    keep.append(reqs)
    cfgs = [(f"cfg-{t}", int(a.asks["min_group_size"][t]), int(a.asks["max_group_size"][t]), reqs[t])
            for t in range(len(reqs))]
    t0 = time.perf_counter()
    g = orc.form_groups(nodes, cfgs, proximity=False)
    dt = time.perf_counter() - t0
    return {"evals_per_s": g.evals / dt if dt > 0 else None, "evals": g.evals, "seconds": dt,
            "sample": f"{len(nodes)} nodes x {len(cfgs)} configs, 1 thread"}


# ----------------------------------------------------------------------------- our arm
def result_digest(res) -> int:
    """64-bit digest of the assignment a pass produced (equal on every rank of a sharded pass)."""
    import zlib

    h = 0
    for arr in (res.group_ask, res.group_off, res.group_members, res.worker_ask):
        h = zlib.crc32(np.ascontiguousarray(arr).view(np.uint8), h)
    return (h << 32) | (int(res.n_groups) & 0xFFFFFFFF)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from protocol_b200 import abi
    from protocol_b200.engine import Comm, Engine, pinned_empty

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the matching engine has no CPU path")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        # torch.distributed is the launcher-side plumbing only: it hands the communicator id to every rank and does
        # the barrier + max-over-ranks of the timing.  The data-path exchange is inside pm_match (pm_comm).
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        box = [Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm = Comm(box[0], world, rank, local_rank)

    w, a, (bits, npat, nmod, words), (T, W, Wg, desc) = make_tables(args.workload, world, args.models)
    mode = abi.PM_MODE_FIRST_FIT | {"materialized": abi.PM_PATH_MATERIALIZED, "fused": abi.PM_PATH_FUSED,
                                    "fused-lean": abi.PM_PATH_FUSED | abi.PM_NO_ASK_STATS}[args.path]

    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        eng = Engine(device=local_rank, timing=True, cost_tile_bytes=args.tile_gib << 30, stream=stream.cuda_stream)
        eng.set_asks(a.asks, a.opts)
        eng.set_model_table(bits, npat, nmod, words)
        eng.set_workers(w.a, w.b)
        if comm is not None:
            eng.attach_comm(comm)   # this rank evaluates workers [rank * Wg, (rank + 1) * Wg)

        def step():
            eng.match(mode)         # N > 1: evaluate own share -> one packed all-gather -> resolution, all inside

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        for _ in range(args.warmup):
            step()
        ranks_agree = None
        if world > 1:   # untimed: every rank must hold the same assignment after the exchange
            mine = torch.tensor([result_digest(eng.fetch()) & 0x7FFFFFFFFFFFFFFF], dtype=torch.int64, device="cuda")
            every = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            ranks_agree = bool(all(int(x.item()) == int(mine.item()) for x in every))
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        acc = {"ms_build": 0.0, "ms_argmin": 0.0, "ms_fused": 0.0, "ms_resolve": 0.0, "ms_exchange": 0.0, "n_build_launches": 0,
               "n_argmin_launches": 0, "n_fused_launches": 0, "n_launches": 0, "cost_bytes_written": 0,
               "cost_bytes_read": 0, "evals": 0}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(args.steps):
            step()
            st = eng.stats()
            for k in acc:
                acc[k] += st[k]
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        clocks = sampler.stop() if rank == 0 else None
        if world > 1:
            tms = torch.tensor([ms], device="cuda")
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        evals_per_step = T * W
        value = evals_per_step * args.steps / (ms * 1e-3)
        last = eng.fetch()          # the last timed pass's result; every rank holds the same one
        groups_formed = int(last.n_groups)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {
                "worker_group": last.worker_group, "worker_ask": last.worker_ask, "group_ask": last.group_ask,
                "group_off": last.group_off, "group_members": last.group_members, **split_best(last.ask_best),
                "ask_count": last.ask_count})

        # ---- e2e: host tables in pinned memory -> H2D -> match -> D2H, all inside the timed region
        lo = rank * Wg if world > 1 else 0
        n_mine = Wg if world > 1 else W
        pa = pinned_empty(n_mine, abi.WORKER_A)
        pb = pinned_empty(n_mine, abi.WORKER_B)
        pa[:] = w.a[lo:lo + n_mine]
        pb[:] = w.b[lo:lo + n_mine]
        # caller-owned tables live in pinned host memory (pm_alloc_pinned), SURVEY 8b "ownership"
        p_asks = pinned_empty(len(a.asks), abi.ASK)
        p_opts = pinned_empty(len(a.opts), abi.GPU_OPT)
        p_asks[:] = a.asks
        p_opts[:] = a.opts
        h2d = n_mine * 32 + len(a.asks) * 32 + len(a.opts) * 32
        d2h = 0

        def e2e_step():
            nonlocal d2h
            eng.set_asks(p_asks, p_opts)
            # a rank re-uploads the rows it evaluates; the other shards' rows are only read by the replicated
            # resolution sweep and stay resident
            eng.upsert_workers(pa, pb, first=lo, sync=False)
            step()
            res = eng.fetch(copy=False)
            d2h = (res.worker_group.nbytes + res.worker_ask.nbytes + res.group_ask.nbytes + res.group_off.nbytes
                   + res.group_members.nbytes + res.ask_best.nbytes + res.ask_count.nbytes)
            return res

        e2e_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2e_steps = max(1, min(args.steps, 5))
        e0.record(stream)
        t_wall = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        e1.record(stream)
        barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t_wall) * 1e3)
        if world > 1:
            tms = torch.tensor([e2e_ms], device="cuda")
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            e2e_ms = float(tms.item())
        e2e_value = evals_per_step * e2e_steps / (e2e_ms * 1e-3)

        # ---- sub-records outside the headline (N = 1): the path the product's own management pass takes, and the
        # north-star extension mode on this workload's price columns
        extras = {}
        if world == 1 and not args.no_extras:
            extras["fused_lean"] = fused_lean_record(eng, abi, T, W, stream, torch)
            if args.workload in PRICES and args.path == "materialized":
                extras["auction"] = auction_record(eng, abi, T, W)

    if rank == 0:
        peak, peak_src = peaks()
        roof = None
        traffic = ncu_traffic()
        if args.path == "materialized" and acc["n_build_launches"]:
            b_gbs = acc["cost_bytes_written"] / (acc["ms_build"] * 1e-3) / 1e9
            r_gbs = acc["cost_bytes_read"] / (acc["ms_argmin"] * 1e-3) / 1e9
            BUILD = "pm_build_cost_fast"   # the fast-form build kernel (pm_build_cost is the generic / staged form)
            dom = BUILD if acc["ms_build"] >= acc["ms_argmin"] else "pm_argmin"
            ach = b_gbs if dom == BUILD else r_gbs
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "peak_source": peak_src,
                    "traffic": (traffic or {}).get(dom),
                    "algorithmic_bytes_per_eval": 8,
                    "algorithmic_bytes_per_launch": (acc["cost_bytes_written"] / acc["n_build_launches"]) if dom == BUILD
                    else (acc["cost_bytes_read"] / acc["n_argmin_launches"]),
                    "avg_launch_ms": (acc["ms_build"] / acc["n_build_launches"]) if dom == BUILD
                    else (acc["ms_argmin"] / acc["n_argmin_launches"]),
                    "other": {"kernel": "pm_argmin" if dom == BUILD else BUILD,
                              "achieved": r_gbs if dom == BUILD else b_gbs,
                              "frac": (r_gbs if dom == BUILD else b_gbs) / peak,
                              "avg_launch_ms": (acc["ms_argmin"] / acc["n_argmin_launches"]) if dom == BUILD
                              else (acc["ms_build"] / acc["n_build_launches"]),
                              "traffic": (traffic or {}).get("pm_argmin" if dom == BUILD else BUILD)}}
        elif acc["n_fused_launches"]:
            roof = {"bound": "hbm", "kernel": "pm_fused_eval", "achieved": None, "peak": peak, "unit": "GB/s",
                    "frac": None, "traffic": (traffic or {}).get("pm_fused_eval"),
                    "note": "fused path is integer-issue-bound; HBM is not its roof (SURVEY 8d)"}
        cpu = cpu_baseline(args, w, a, bits, words, T, W) if world == 1 and not args.no_cpu else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32 predicate -> int64 packed cost", "data": DATA,
            "config": config_dict(args, desc, T, W, Wg, world),
            "detail": {"path": args.path},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps},
            "gpu_launches": acc["n_launches"],
            "roofline": roof,
            "cpu_baseline": cpu,
            "clocks": clocks,
            "kernel_ms_per_step": {k: acc[k] / args.steps for k in ("ms_build", "ms_argmin", "ms_fused", "ms_exchange", "ms_resolve")},
            "groups_formed": groups_formed,
        }
        if ranks_agree is not None:
            line["ranks_agree"] = ranks_agree
        line.update(extras)
        print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.barrier()          # nobody tears its communicator down while another rank is still in a pass
    eng.close()
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def fused_lean_record(eng, abi, T, W, stream, torch, steps=5):
    """The pass pm_plugin_try_form_new_groups runs: evaluation + reduction on chip, no per-ask statistics."""
    mode = abi.PM_MODE_FIRST_FIT | abi.PM_PATH_FUSED | abi.PM_NO_ASK_STATS
    eng.match(mode)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        eng.match(mode)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    st = eng.stats()
    return {"evals_per_s": T * W / (ms * 1e-3), "ms_per_step": ms, "steps": steps, "ms_fused": st["ms_fused"],
            "ms_resolve": st["ms_resolve"], "groups_formed": int(eng.fetch().n_groups),
            "note": "same groups as the materialised pass; integer-issue-bound, ~20 MB of DRAM traffic per pass"}


def auction_record(eng, abi, T, W):
    """North-star extension (no reference counterpart, self-oracle): price-capped eps-auction on the same tables."""
    from protocol_b200 import synth

    caps = np.exp(np.log(20) + synth._unit(synth.SEED_EXT, T, 3) * np.log(100)).astype(np.uint32)   # log-uniform 20..2000
    eng.set_price_caps(caps)
    t0 = time.perf_counter()
    eng.match(abi.PM_MODE_AUCTION)
    dt = time.perf_counter() - t0
    st = eng.stats()
    res = eng.fetch()
    return {"seconds": dt, "rounds": st["n_rounds"], "evals": st["evals"], "asks_assigned": int(res.n_groups),
            "table_walks": st["n_tiles"], "pool_refills": st["n_build_launches"], "kernel_launches": st["n_launches"],
            "eps": "1 throughout (default; eps-scaling loses the T*eps bound under price caps, tests/test_oracle_auction.py)", "price_caps": "log-uniform 20..2000",
            "note": "rounds are not multiplied into the headline evals/s (SURVEY 8d)"}


def cpu_baseline(args, w, a, bits, words, T, W):
    from oracle import pm_oracle as orc

    cpus = host_cpus()
    cores = cpus["threads"]
    rows = max(1, min(T, int(1.5e9 // max(W, 1))))
    t0 = (T - rows) // 2
    orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, t0, t0 + min(rows, 64), 0, W, threads=cores)
    t_s = time.perf_counter()
    ev = orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, t0, t0 + rows, 0, W, threads=cores)["evals"]
    dt = time.perf_counter() - t_s
    return {"value": ev / dt, "unit": UNIT, "cores": cores, "kind": "port", "host_cpus": cpus,
            "sample": f"asks [{t0},{t0 + rows}) x all {W} workers = {ev:.3g} pair evaluations, {cores} threads, {dt:.1f} s",
            "faithful_single_thread": faithful_sample(orc, w, a)}


RESULT_OUT = sys.stdout


def main():
    # stdout carries exactly ONE line, the result: native libraries write banners to file descriptor 1 (NCCL prints its
    # version there when a communicator is created), so fd 1 is pointed at stderr and the line goes to a saved copy
    global RESULT_OUT
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: cfg3 (BASELINE configs[2]) on one GPU, cfg5's per-GPU shape on several")
    ap.add_argument("--path", default="materialized", choices=["materialized", "fused", "fused-lean"])
    ap.add_argument("--tile-gib", dest="tile_gib", type=int, default=8)
    ap.add_argument("--models", type=int, default=0,
                    help="distinct worker model strings (0: the 16-entry catalogue; > 31 selects the wide-catalogue kernel variants)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", dest="no_extras", action="store_true", help="skip the fused_lean / auction sub-records")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step returned as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload is None:
        args.workload = "cfg3" if args.gpus <= 1 else "cfg5"
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    except BaseException:
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        raise


if __name__ == "__main__":
    main()
