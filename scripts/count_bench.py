"""The counting batches (dq_count_batch_cells / dq_count_batch_graphs) against the FIRST-mode batch on the same input:

  sudoku_L2 : 1 M synthetic Sudoku (30 givens), solution limit 2: the uniqueness check of a puzzle generator
  sudoku_L0 : the same batch, every solution
  colour_L0 : 32 768 3-colourings of G(200, 4.2/199), node budget 100 000, every solution

The FIRST-mode batch picks its engine (the 9x9 Sudoku lane pipeline, the colouring lane engine); the count always runs
on the generic warp engine.  Per workload: wall time of one call (it ends in a synchronise) for the count and for the
FIRST-mode batch, median of REPEATS after one warm-up of each, kernel_ms, and what the count found.  Where both found a
solution of an instance within the budget, the count's DFS-first solution must equal the FIRST-mode batch's.  Prints
one JSON line per workload, after one line naming the card and its power limit."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dequan_b200 import api  # noqa: E402
from dequan_b200 import generators as G  # noqa: E402
from dequan_b200.model import sudoku_template  # noqa: E402

REPEATS = 3


def timed(fn):
    fn()
    ts, r = [], None
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return r, sorted(ts)[REPEATS // 2], ts


def run(name, count_fn, first_fn, nv):
    c, tc, tc_all = timed(count_fn)
    f, tf, tf_all = timed(first_fn)
    both = (c.solutions >= 1) & (f.status == 1)
    assert (c.first[both, :nv] == f.solution[both, :nv]).all(), name
    hist = np.bincount(np.minimum(c.solutions, 3).astype(np.int64), minlength=4)
    row = {"workload": name, "instances": int(len(c.status)), "count_ms": round(tc * 1e3, 3), "first_ms": round(tf * 1e3, 3),
           "count_over_first": round(tc / tf, 2), "count_kernel_ms": round(c.kernel_ms, 3), "first_kernel_ms": round(f.kernel_ms, 3),
           "count_nodes": int(c.total_nodes), "first_nodes": int(f.total_nodes), "solutions": int(c.solutions.sum()),
           "instances_with_0_1_2_3plus_solutions": hist.tolist(), "count_budget": int(c.n_budget),
           "count_ms_all": [round(t * 1e3, 3) for t in tc_all], "first_ms_all": [round(t * 1e3, 3) for t in tf_all]}
    print(json.dumps(row), flush=True)
    return row


def main():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True, check=True).stdout.splitlines()[0]
    print(json.dumps({"card": card, "device": api.device_info()["name"]}), flush=True)
    m = api.Model(sudoku_template())
    cells = G.sudoku_batch(1_000_000, givens=30)
    run("sudoku_L2", lambda: m.count_batch_cells(cells, solution_limit=2), lambda: m.solve_batch_cells(cells), 81)
    run("sudoku_L0", lambda: m.count_batch_cells(cells, solution_limit=0), lambda: m.solve_batch_cells(cells), 81)
    off, edges = G.colouring_batch(32_768, 200, 4.2)
    run("colour_L0", lambda: api.count_batch_graphs(200, 3, off, edges, node_budget=100_000),
        lambda: api.solve_batch_graphs(200, 3, off, edges, node_budget=100_000), 200)


if __name__ == "__main__":
    main()
