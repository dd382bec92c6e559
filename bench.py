#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: search nodes/sec (N-Queens all-solutions) and Sudoku
puzzles/sec, on 1/2/4/8 B200, next to the reference dequan timed on the host cores.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun ... bench.py --gpus N ...                      (N > 1, one rank per GPU, NCCL)

--dump-outputs DIR: what the last HBM-resident step of each workload returned, as DIR/<name>.npy (float32 / float64):
N-Queens {solutions, nodes} and first solution; for the batches, solution / node count / status of a fixed, seeded
sample of the instances (`*_index` holds their indices) and the batch totals {sat, unsat, budget, nodes}.  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.

One "step" = one complete solve of the workload through the C ABI; every timed loop runs K of them.  The workload is
the same at every N, so that the 1/2/4/8-GPU series is a strong-scaling series of ONE job: BASELINE config C5, 17-Queens all-solutions (95 815 104
solutions / 5 474 619 051 nodes, tests/golden/reference_large.json; about 15 ms on one B200), FC-surviving prefixes
dealt to the ranks by key, {solutions, nodes} summed with NCCL.  The line also carries `sudoku` (config C3, 1M puzzles,
sharded over the ranks) and, at N == 1, `extra.nqueens14_1gpu` (config C2) and `extra.colouring` (config C4), each
with value / e2e / roofline / cpu_baseline of its own.
`value`  : inputs/tables already resident in HBM (compiled model re-used), whole-job nodes/s.
`e2e`    : the same through the host-facing C-ABI calls with HOST buffers, every step: dq_compile of the flat
           model descriptor (CSP::FinalizeModel + Assignment::Reset), table upload, solve, result read-back, dq_free.
Every result of every step is checked against the reference's answers; a mismatch aborts the bench.
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
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# SURVEY.md §8d: forward-checking domain updates per node (A) -> algorithmic lane-ops/node = 5A+4 (queens), 2A+4 (!=,0)
QUEENS_A = {14: 79143794 / 19787662, 15: 498817896 / 121498513, 16: 3342155422 / 795563572, 17: 23537105544 / 5474619051}
# colouring, G(200, 4.2/199), k=3, 100 k-node budget: later neighbours of the assigned vertex, averaged over the nodes of
# the first 12 instances (3 000 013 updates / 1 100 407 nodes; DESIGN.md §4.4)
COLOURING_A = 2.726
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "dequan_ref")


def golden_queens():
    """(solutions, nodes) per board size from the runs of the unmodified reference under tests/golden/."""
    out = {}
    for name in ("reference.json", "reference_large.json"):
        with open(os.path.join(ROOT, "tests", "golden", name)) as f:
            for n, g in json.load(f)["nqueens"].items():
                out[int(n)] = (g["count"]["solutions"], g["count"]["nodes"])
    return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from profiles/r2_traffic.json (written by
    scripts/ncu_traffic.py out of an `ncu --set full` report, with the commit it was measured at); None if absent."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None, None
    e = json.load(open(p)).get(key)
    if not e:
        return None, None
    return int(e["dram_bytes_read"] + e["dram_bytes_write"]), f"profiles/r2_traffic.json[{key}]@{e.get('commit', '?')[:9]}"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        load = sm[len(sm) // 2:] if sm else []          # the busiest half of the samples = "under load"
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons}


def run_ref(args_list, timeout=900):
    out = subprocess.run([REF_BIN] + [str(a) for a in args_list], capture_output=True, text=True, timeout=timeout, check=True).stdout
    return [json.loads(line) for line in out.splitlines() if line.strip()]


def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
def cpu_baseline_queens():
    """Reference dequan on the host cores, bounded sample of the same workload."""
    thr = cpu_threads()
    if not os.path.exists(REF_BIN):
        return cpu_baseline_port_queens()
    t = time.time()
    o = run_ref(["nqueens", 17, "count", thr, 8, 3])[0]
    wall = time.time() - t
    return {"value": o["nodes"] / o["seconds"], "unit": "nodes/s", "cores": min(thr, 17), "kind": "reference",
            "sample": f"17-Queens subtree under prefix (8,3), one depth-3 subtree per thread ({o['nodes']} nodes, {wall:.1f}s)"}


def cpu_baseline_port_queens():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    from dequan_b200.model import nqueens
    n = 11
    t = time.time()
    o = oracle_lib.solve(nqueens(n), "count")
    dt = time.time() - t
    return {"value": o.nodes / dt, "unit": "nodes/s", "cores": 1, "kind": "port",
            "sample": f"{n}-Queens all-solutions with the C restatement (oracle/_ref absent)"}


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation, all host threads, same metric/config."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    thr = cpu_threads()
    n = 17
    cmd = ["nqueens", 17, "count", thr, 8, 3]
    times, nodes = [], 0
    kind = "reference" if os.path.exists(REF_BIN) else "port"
    for i in range(args.warmup + args.steps):
        if kind == "reference":
            o = run_ref(cmd)[0]
            dt, nd = o["seconds"], o["nodes"]
        else:
            b = cpu_baseline_port_queens()
            nd = 1
            dt = 1.0 / b["value"]
        if i >= args.warmup:
            times.append(dt)
            nodes += nd
    total = sum(times)
    val = nodes / total
    sample = "17-Queens subtree under prefix (8,3) split over the host threads (bounded sample of the 5.47e9-node tree)"
    line = {"impl": "reference", "metric": "search_nodes_per_sec", "value": val, "unit": "nodes/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(len(times), 1),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": workload_config(args.gpus, n),
            "cpu_baseline": {"value": val, "unit": "nodes/s", "cores": min(thr, n), "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def sample_rows(n, k):
    """At most k of the n instance indices of a batch, ascending, chosen with a fixed seed: --dump-outputs writes the
    per-instance outputs of these rows only, so that two runs with the same arguments dump the same rows."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def dump_outputs(path, outputs):
    """--dump-outputs: one float32 / float64 array per name as `path/<name>.npy`, at most 64 MB in all."""
    assert all(a.dtype in (np.float32, np.float64) for a in outputs.values())
    assert sum(a.nbytes for a in outputs.values()) <= 64_000_000
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), a)


def workload_config(n_gpus, n):
    return {"workload": f"nqueens{n}_count_all", "baseline_config": {17: "C5", 14: "C2"}.get(n, ""),
            "parallelism": "prefix split" + (f", keys dealt to {n_gpus} GPUs, NCCL sum" if n_gpus > 1 else ""),
            "l2": "flushed between steps"}


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default="auto")
    ap.add_argument("--sudoku-n", type=int, default=1_000_000)
    ap.add_argument("--givens", type=int, default=30)
    ap.add_argument("--colouring-n", type=int, default=32768)
    ap.add_argument("--no-sudoku", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of each workload computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from dequan_b200 import api, multi
    from dequan_b200.model import nqueens

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    api.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    QUEENS = golden_queens()

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure_queens(n, steps, warmup):
        """value / e2e legs of the N-Queens all-solutions workload; every step's result is checked."""
        want_sols, want_nodes = QUEENS[n]
        csp = nqueens(n)
        model = api.Model(csp)

        def solve_step(m):
            """-> (this rank's result, the whole job's result)"""
            loc = m.solve_tree("count", part_rank=rank, part_count=world, engine=args.engine)
            if world == 1:
                return loc, loc
            return loc, multi.reduce_tree(loc, m.nodes_upto, "count", n, device=dev)

        def timed_steps(step_fn, k, w):
            tot, kern, launches = 0.0, 0.0, 0
            for i in range(w + k):
                flush.fill_(i & 0xFF)
                sync_all()
                t0 = time.perf_counter()
                loc, res = step_fn()
                # (at N > 1 the step ends with the all_gather of the ranks' records and its read-back: every rank holds
                # the global answer here, so the step needs no second barrier; the MAX over ranks is taken below)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                sols, nodes = res.solutions, res.nodes
                assert (sols, nodes) == (want_sols, want_nodes), f"parity failure in bench step: {(sols, nodes)}"
                if i >= w:
                    tot += dt
                    kern += loc.kernel_ms
                    launches += loc.launches
            if world > 1:
                t = torch.tensor([tot, kern], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                tot, kern = float(t[0]), float(t[1])
            return tot, kern, launches, res

        tot, kern_ms, launches, last = timed_steps(lambda: solve_step(model), steps, warmup)
        # roofline leg: the search kernel's own duration from CUDA events on its stream (DQ_TREE_TIME_KERNELS; the steps
        # above replay the solve as one CUDA graph, whose inner events cannot be read back); this rank's own node count
        dom_ms, dom_nodes, dom_records = 0.0, 0, 0
        for i in range(steps):
            flush.fill_(i & 0xFF)
            sync_all()
            loc = model.solve_tree("count", part_rank=rank, part_count=world, engine=args.engine, time_kernels=True)
            assert (loc.solutions, loc.nodes) == (want_sols, want_nodes) or world > 1
            dom_ms += loc.search_kernel_ms
            dom_nodes, dom_records = loc.nodes - loc.frontier_nodes, loc.n_prefixes
        desc_keep = csp.desc()          # the host-side flat descriptor: the input buffers of the C-ABI call

        def e2e_step():
            m = api.Model(csp, desc_keep)   # dq_compile: FinalizeModel + Reset on the host, tables uploaded by the solve
            r = solve_step(m)
            m.close()
            return r
        e_tot, _, _, _ = timed_steps(e2e_step, steps, warmup)
        return {"n": n, "nodes": want_nodes, "steps": steps, "tot": tot, "kern_ms": kern_ms, "launches": launches, "e_tot": e_tot,
                "dom_ms": dom_ms, "dom_nodes": dom_nodes, "dom_records": dom_records, "table_bytes": model.table_bytes(),
                "engine": model.solve_tree("count", part_rank=rank, part_count=world, engine=args.engine).engine,
                "outputs": {f"nqueens{n}": np.array([last.solutions, last.nodes], dtype=np.float64),
                            f"nqueens{n}_first": np.array(last.first or [], dtype=np.float64)}}

    def queens_block(q, int_peak, hbm_peak, peak_src):
        n, steps = q["n"], q["steps"]
        return {"value": q["nodes"] * steps / q["tot"], "unit": "nodes/s", "ms_per_step": 1e3 * q["tot"] / steps,
                "kernel_ms_per_step": q["kern_ms"] / steps,
                "e2e": {"value": q["nodes"] * steps / q["e_tot"], "unit": "nodes/s", "h2d_bytes_per_step": q["table_bytes"] + 64,
                        "d2h_bytes_per_step": 64 + 4 * n + 8 * 64, "ms_per_step": 1e3 * q["e_tot"] / steps},
                "gpu_launches": q["launches"], "engine": q["engine"],
                "roofline": roofline_queens(n, world, q["dom_nodes"], q["dom_records"], q["dom_ms"] / steps, int_peak, hbm_peak, peak_src,
                                            q["table_bytes"])}

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n = 17
    Q = measure_queens(n, args.steps, args.warmup)
    Q14 = measure_queens(14, args.steps, args.warmup) if world == 1 and not args.no_extra else None
    sudoku = None
    if not args.no_sudoku:
        sudoku = sudoku_section(args, torch, api, dev, world, rank, dist, flush)      # still inside the clock-sampling window
    colouring = None
    if world == 1 and not args.no_extra:
        colouring = colouring_section(args, torch, api, dev, flush)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    clocks = sampler.stop()
    if args.dump_outputs:
        outputs = dict(Q["outputs"])
        for part in (Q14["outputs"] if Q14 else {}, sudoku.pop("_outputs") if sudoku else {},
                     colouring.pop("_outputs") if colouring else {}):
            outputs.update(part)
        dump_outputs(args.dump_outputs, outputs)
    int_peak, _ = api.measure_int_peak()
    hbm_peak, peak_src = peaks()
    qb = queens_block(Q, int_peak, hbm_peak, peak_src)
    line = {
        "metric": "search_nodes_per_sec", "value": qb["value"], "unit": "nodes/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": qb["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": workload_config(world, n),
        "clocks": clocks, "e2e": qb["e2e"], "gpu_launches": qb["gpu_launches"], "engine": qb["engine"],
        "kernel_ms_per_step": qb["kernel_ms_per_step"], "roofline": qb["roofline"],
    }
    if not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_queens()
    if sudoku is not None:
        line["sudoku"] = sudoku_rooflines(sudoku, hbm_peak, peak_src, int_peak)
    extra = {}
    if Q14 is not None:
        extra["nqueens14_1gpu"] = dict(config=workload_config(1, 14), steps=Q14["steps"], **queens_block(Q14, int_peak, hbm_peak, peak_src))
    if colouring is not None:
        extra["colouring"] = colouring_rooflines(colouring, int_peak, hbm_peak, peak_src)
    line["extra"] = extra
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def roofline_queens(n, world, lane_nodes, records, lane_ms, int_peak, hbm_peak, peak_src, table_bytes=0):
    """Roofline of the dominant kernel, k_queens_bucket_t (depth-bucketed subtree search).  It is integer-issue bound
    (SURVEY.md §8d): algorithmic work = (5A+4) lane-ops per node, A = forward-checking domain updates per node; the peak
    is the LOP3 rate measured in this run, i.e. the ALU pipe alone (16 lanes per clock and SM quarter) — the kernel also
    issues integer multiply-adds on the FMA pipe next to it.  nodes_per_launch is what THIS rank's launch searched."""
    ops_per_node = 5 * QUEENS_A[n] + 4
    achieved = lane_nodes * ops_per_node / (lane_ms * 1e-3) if lane_ms else 0.0
    traffic, src = ncu_traffic(f"k_queens_bucket/nqueens{n}") if world == 1 else (None, None)
    return {"bound": "int32-alu", "kernel": "k_queens_bucket_t", "achieved": achieved / 1e12, "peak": int_peak / 1e12,
            "unit": "Tlane-op/s per GPU", "frac": achieved / int_peak, "kernel_ms": lane_ms,
            "nodes_per_launch": lane_nodes, "ops_per_node": ops_per_node, "peak_source": "LOP3 microbenchmark, this run",
            # the job's true input is the model table (a few KB); what the kernel streams from HBM is the ENGINE'S OWN frontier:
            # one 16-byte record per depth-k subtree, written by the level kernels before it
            "traffic": traffic, "traffic_source": src, "algorithmic_bytes": table_bytes, "frontier_bytes": records * 16,
            "hbm": {"achieved": records * 16 / (lane_ms * 1e-3) / 1e9 if lane_ms else None, "peak": hbm_peak, "unit": "GB/s",
                    "peak_source": peak_src, "what": "frontier records read by the launch"}}


def sudoku_rooflines(out, hbm_peak, peak_src, int_peak):
    kpps, nps = out.pop("_kernel_pps"), out["nodes_per_sec"]
    traffic, src = ncu_traffic("sudoku_pipeline/1M_g30") if out.get("shard", out["n"]) == 1_000_000 else (None, None)
    out["roofline_int"] = {"bound": "int32-alu", "ops_per_node": 2 * 10 + 4, "achieved": nps * 24 / 1e12, "peak": int_peak / 1e12,
                           "unit": "Tlane-op/s", "frac": nps * 24 / int_peak}
    out["roofline"] = {"bound": "hbm", "achieved": kpps * 174 / 1e9, "peak": hbm_peak, "unit": "GB/s",
                       "frac": kpps * 174 / 1e9 / hbm_peak, "traffic": traffic, "traffic_source": src,
                       "algorithmic_bytes": 174 * out.get("shard", out["n"]), "peak_source": peak_src,
                       "note": "instance stream; the search is integer-issue bound (roofline_int)"}
    return out


def sudoku_section(args, torch, api, dev, world=1, rank=0, dist=None, flush=None):
    """BASELINE config C3: batch of synthetic 9x9 Sudoku (810 binary != arcs), first solution each.  With N GPUs the
    batch is cut into N contiguous shards, one per rank; the only collective is the final sum of {solved, nodes}."""
    from dequan_b200 import generators as G
    from dequan_b200 import multi
    from dequan_b200.model import sudoku_template
    n_total = args.sudoku_n
    lo, hi = multi.shard_range(n_total, rank, world)
    n = hi - lo
    cells = G.sudoku_batch(n, givens=args.givens, start=lo)
    tmpl = api.Model(sudoku_template())

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    # HBM-resident leg
    d_cells = torch.from_numpy(cells).to(dev)
    d_sol = torch.empty_like(d_cells)
    d_nodes = torch.empty(n, dtype=torch.int64, device=dev)
    d_status = torch.empty(n, dtype=torch.uint8, device=dev)
    steps, warm = args.steps, 3
    kern, tot, launches, total_nodes = 0.0, 0.0, 0, 0
    for i in range(warm + steps):
        if flush is not None:
            flush.fill_(i & 0xFF)               # a shard may fit the 126 MB L2: evict it between steps (untimed)
        sync_all()
        t0 = time.perf_counter()
        st = tmpl.solve_batch_cells_ptr(d_cells.data_ptr(), n, 81, d_sol.data_ptr(), d_nodes.data_ptr(), d_status.data_ptr(), device=True)
        torch.cuda.synchronize()                # (shards are independent: each rank's own time, MAX over ranks below)
        dt = time.perf_counter() - t0
        assert st.n_sat == n
        if i >= warm:
            tot += dt; kern += st.kernel_ms; launches += st.kernel_launches; total_nodes = st.total_nodes
    tot, kern = reduce_max(tot), reduce_max(kern)
    dumped = None
    if args.dump_outputs:           # the last HBM-resident step's outputs (at N > 1: this rank's shard)
        rows = sample_rows(n, 65536)
        idx = torch.from_numpy(rows).to(dev)
        dumped = {"sudoku_index": (lo + rows).astype(np.float64),
                  "sudoku_solution": d_sol[idx].cpu().numpy().astype(np.float32),
                  "sudoku_nodes": d_nodes[idx].cpu().numpy().astype(np.float64),
                  "sudoku_status": d_status[idx].cpu().numpy().astype(np.float32),
                  "sudoku_totals": np.array([st.n_sat, st.n_unsat, st.n_budget, st.total_nodes], dtype=np.float64)}
    # host-buffer leg (pinned), copies inside the timed region
    h_cells = torch.from_numpy(cells).pin_memory()
    h_sol = torch.empty((n, 81), dtype=torch.uint8).pin_memory()
    h_nodes = torch.empty(n, dtype=torch.int64).pin_memory()
    h_status = torch.empty(n, dtype=torch.uint8).pin_memory()
    e_tot = 0.0
    for i in range(warm + steps):
        if flush is not None:
            flush.fill_(i & 0xFF)
        sync_all()
        t0 = time.perf_counter()
        st = tmpl.solve_batch_cells_ptr(h_cells.data_ptr(), n, 81, h_sol.data_ptr(), h_nodes.data_ptr(), h_status.data_ptr())
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warm:
            e_tot += dt
    e_tot = reduce_max(e_tot)
    if world > 1:      # the one collective of a sharded batch: totals
        g = multi.reduce_batch(st.n_sat, st.n_unsat, st.n_budget, total_nodes, device=dev)
        assert g.n_sat == n_total
        total_nodes = g.nodes
    # checks: device and host legs agree; solutions are valid grids consistent with the givens
    sol = h_sol.numpy()
    assert (d_sol.cpu().numpy() == sol).all() and (d_nodes.cpu().numpy() == h_nodes.numpy()).all()
    g = sol.reshape(n, 9, 9)
    want = np.arange(1, 10)
    assert (np.sort(g, axis=2) == want).all() and (np.sort(g, axis=1) == want[:, None]).all()
    assert (sol[cells != 0] == cells[cells != 0]).all()
    if rank != 0:
        return None
    n_shard, n = n, n_total
    pps = n * steps / tot
    kpps = n * steps / (kern * 1e-3)
    out = {"metric": "sudoku_puzzles_per_sec", "value": pps, "unit": "puzzles/s", "n": n, "givens": args.givens, "n_gpus": world,
           "scaling": "strong", "shard": n_shard, "steps": steps, "ms_per_step": 1e3 * tot / steps, "kernel_ms_per_step": kern / steps,
           "nodes_per_puzzle": total_nodes / n, "nodes_per_sec": total_nodes * steps / (kern * 1e-3),
           "config": {"workload": f"sudoku_1M_g{args.givens}" if n == 1_000_000 else f"sudoku_{n}_g{args.givens}", "l2": "flushed between steps"},
           "e2e": {"value": n * steps / e_tot, "unit": "puzzles/s", "h2d_bytes_per_step": n * 81, "d2h_bytes_per_step": n * 90,
                   "ms_per_step": 1e3 * e_tot / steps},
           "gpu_launches": launches, "_kernel_pps": kpps}
    if dumped is not None:
        out["_outputs"] = dumped
    if not args.no_cpu and os.path.exists(REF_BIN):
        sample = min(n_shard, 16000)
        path = "/tmp/dq_bench_sudoku.txt"
        with open(path, "w") as f:
            f.write("\n".join(G.sudoku_lines(cells[:sample])) + "\n")
        thr = cpu_threads()
        o = run_ref(["sudoku", path, "boxes", thr, sample, "quiet"])[-1]
        # parity at scale against the unmodified reference: the node total of the sample must be the reference's
        assert int(h_nodes.numpy()[:sample].sum()) == int(o["nodes"]), ("sudoku node total differs from the reference",
                                                                      int(h_nodes.numpy()[:sample].sum()), o["nodes"])
        out["cpu_baseline"] = {"value": o["puzzles"] / o["wall_seconds"], "unit": "puzzles/s", "cores": thr, "kind": "reference",
                               "sample": f"first {sample} puzzles, one per thread, model build included",
                               "nodes_per_sec": o["nodes"] / o["wall_seconds"]}
    return out


def colouring_section(args, torch, api, dev, flush):
    """BASELINE config C4: batch of G(200, 4.2/199) 3-colouring instances near the phase transition (vertices in
    maximum-cardinality order), first solution under a 100 000-node budget each, tri-state result."""
    from dequan_b200 import generators as G
    n, nv, k, c, budget = args.colouring_n, 200, 3, 4.2, 100_000
    off, edges = G.colouring_batch(n, nv, c)
    steps, warm = args.steps, 3
    pad = (-2 * int(off[-1])) % 16
    d_edges = torch.from_numpy(np.concatenate([edges.reshape(-1), np.zeros(pad, dtype=np.uint8)])).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_col = torch.empty((n, nv), dtype=torch.uint8, device=dev)
    d_nodes = torch.empty(n, dtype=torch.int64, device=dev)
    d_status = torch.empty(n, dtype=torch.uint8, device=dev)
    tot = kern = search = 0.0
    launches = 0
    for i in range(warm + steps):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st = api.solve_batch_graphs_ptr(nv, k, off, d_off.data_ptr(), d_edges.data_ptr(), d_col.data_ptr(), d_nodes.data_ptr(),
                                        d_status.data_ptr(), node_budget=budget, device=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warm:
            tot += dt; kern += st.kernel_ms; search += st.search_kernel_ms; launches += st.kernel_launches
    total_nodes = st.total_nodes
    dumped = None
    if args.dump_outputs:           # the last HBM-resident step's outputs
        rows = sample_rows(n, 16384)
        idx = torch.from_numpy(rows).to(dev)
        dumped = {"colouring_index": rows.astype(np.float64),
                  "colouring_colours": d_col[idx].cpu().numpy().astype(np.float32),
                  "colouring_nodes": d_nodes[idx].cpu().numpy().astype(np.float64),
                  "colouring_status": d_status[idx].cpu().numpy().astype(np.float32),
                  "colouring_totals": np.array([st.n_sat, st.n_unsat, st.n_budget, st.total_nodes], dtype=np.float64)}
    h_edges = torch.from_numpy(edges.reshape(-1).copy()).pin_memory()
    h_col = torch.empty((n, nv), dtype=torch.uint8).pin_memory()
    h_nodes = torch.empty(n, dtype=torch.int64).pin_memory()
    h_status = torch.empty(n, dtype=torch.uint8).pin_memory()
    e_tot = 0.0
    for i in range(warm + steps):
        flush.fill_(i & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st2 = api.solve_batch_graphs_ptr(nv, k, off, 0, h_edges.data_ptr(), h_col.data_ptr(), h_nodes.data_ptr(), h_status.data_ptr(),
                                         node_budget=budget, device=False)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if i >= warm:
            e_tot += dt
    # checks: both legs agree; every returned colouring is proper
    col, status = h_col.numpy(), h_status.numpy()
    assert (d_col.cpu().numpy() == col).all() and (d_nodes.cpu().numpy() == h_nodes.numpy()).all() and (d_status.cpu().numpy() == status).all()
    for i in np.nonzero(status == 1)[0][:2000]:
        e = edges[off[i]:off[i + 1]]
        assert (col[i][e[:, 0]] != col[i][e[:, 1]]).all() and col[i].max() < k
    out = {"metric": "colouring_nodes_per_sec", "value": total_nodes * steps / tot, "unit": "nodes/s", "instances": n,
           "instances_per_sec": n * steps / tot, "node_budget": budget, "steps": steps, "ms_per_step": 1e3 * tot / steps,
           "kernel_ms_per_step": kern / steps, "search_kernel_ms": search / steps, "nodes": total_nodes,
           "sat": st.n_sat, "unsat": st.n_unsat, "budget": st.n_budget,
           "config": {"workload": f"colouring_g200_c{c}_k{k}_{n}", "baseline_config": "C4", "l2": "flushed between steps"},
           "e2e": {"value": total_nodes * steps / e_tot, "unit": "nodes/s", "instances_per_sec": n * steps / e_tot,
                   "h2d_bytes_per_step": int(st2.h2d_bytes), "d2h_bytes_per_step": int(st2.d2h_bytes), "ms_per_step": 1e3 * e_tot / steps},
           "gpu_launches": launches, "engine": "lane per instance (k_graphs_adjacency x2, k_graphs_lane)",
           "_bytes_in": int(2 * off[-1] + 8 * (n + 1))}
    if dumped is not None:
        out["_outputs"] = dumped
    if not args.no_cpu and os.path.exists(REF_BIN):
        sample = min(n, 256)
        path = "/tmp/dq_bench_graphs.txt"
        with open(path, "w") as f:
            f.write("\n".join(G.graph_lines(off[:sample + 1], edges, nv)) + "\n")
        thr = cpu_threads()
        o = run_ref(["color", path, k, budget, thr, "quiet"])[-1]
        # parity at scale against the unmodified reference: the node total of the sample must be the reference's
        assert int(h_nodes.numpy()[:sample].sum()) == int(o["nodes"]), ("colouring node total differs from the reference",
                                                                      int(h_nodes.numpy()[:sample].sum()), o["nodes"])
        out["cpu_baseline"] = {"value": o["nodes"] / o["wall_seconds"], "unit": "nodes/s", "cores": thr, "kind": "reference",
                               "sample": f"first {sample} instances, one per thread, model build included",
                               "instances_per_sec": sample / o["wall_seconds"]}
    return out


def colouring_rooflines(out, int_peak, hbm_peak, peak_src):
    ops = 2 * COLOURING_A + 4
    bytes_in = out.pop("_bytes_in")
    ms = out["search_kernel_ms"]
    achieved = out["nodes"] * ops / (ms * 1e-3)
    traffic, src = ncu_traffic(f"k_graphs_lane/{out['config']['workload']}")
    algo = bytes_in + out["instances"] * (200 + 9)
    out["roofline"] = {"bound": "int32-alu", "kernel": "k_graphs_lane", "achieved": achieved / 1e12, "peak": int_peak / 1e12,
                       "unit": "Tlane-op/s", "frac": achieved / int_peak, "kernel_ms": ms, "nodes_per_launch": out["nodes"],
                       "ops_per_node": ops, "peak_source": "LOP3 microbenchmark, this run", "traffic": traffic, "traffic_source": src,
                       "algorithmic_bytes": algo,
                       "hbm": {"achieved": algo / (out["kernel_ms_per_step"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "peak_source": peak_src}}
    return out


def _quiet_stdout():
    """The driver reads ONE JSON line from stdout: native libraries that print there (the NCCL version banner) are sent
    to stderr, and `print` keeps the real stdout."""
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real


if __name__ == "__main__":
    _quiet_stdout()
    main()
