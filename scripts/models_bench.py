"""dq_solve_models against a loop of dq_solve_tree over the same handles, on seeded workloads of many different small
models: what a caller holding generated levels, puzzles of different shapes or scheduling variants runs.

  (a) 10 000 drop-in-sized models: random models of 6-12 variables, N-Queens 6-10, small 3-colourings; FIRST mode
  (b) 1 000 3-colourings of G(n, c/(n-1)) with 20-30 vertices, c = 4.0 / 4.5; FIRST and COUNT_ALL
  (c) (a) plus four rows+columns Sudoku trees (1.3 M nodes each) that take the split search; FIRST mode

Per workload: wall time of one solve_models call (it ends in a synchronise) and of the loop, each after a warm-up of
both (the loop's warm-up also uploads every handle's tables, so the loop runs with every model cached, as the drop-in
header does on a repeated call), models/s, nodes/s, n_split and kernel_ms.  The batch's answers must equal the loop's,
model by model.  Prints one JSON line per workload and mode, after one line naming the card and its power limit."""
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from dequan_b200 import api  # noqa: E402
from dequan_b200 import generators as G  # noqa: E402
from dequan_b200.model import REFERENCE_SUDOKU, colouring, nqueens, sudoku  # noqa: E402
from randmodels import random_model  # noqa: E402

REPEATS = 3


def small_models(n, seed=20261021):
    rng = random.Random(seed)
    out = []
    for i in range(n):
        r = rng.random()
        if r < 0.8:
            nv = rng.randint(6, 12)
            out.append(random_model(seed + i, nv, rng.randint(nv // 2, 2 * nv), rng.randint(2, 7), "ne" if i % 5 == 0 else "all"))
        elif r < 0.9:
            out.append(nqueens(rng.randint(6, 10)))
        else:
            nv = rng.randint(8, 16)
            out.append(colouring(nv, 3, [tuple(e) for e in G.colouring_instance(nv, 3.0, seed, i)]))
    return out


def medium_colourings(n, seed=20261022):
    rng = random.Random(seed)
    out = []
    for i in range(n):
        nv = rng.randint(20, 30)
        out.append(colouring(nv, 3, [tuple(e) for e in G.colouring_instance(nv, 4.0 if i % 2 == 0 else 4.5, seed, i)]))
    return out


def run(name, csps, mode):
    models = [api.Model(c) for c in csps]
    batch = api.solve_models(models, mode)
    loop = [models[i].solve_tree(mode) for i in range(len(models))]
    for i, t in enumerate(loop):
        assert (batch.status[i], batch.solutions[i], batch.nodes[i], batch.first[i]) == (t.status, t.solutions, t.nodes, t.first), (name, mode, i)
    t_batch, t_loop = [], []
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        batch = api.solve_models(models, mode)
        t_batch.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for m in models:
            m.solve_tree(mode)
        t_loop.append(time.perf_counter() - t0)
    tb, tl = sorted(t_batch)[REPEATS // 2], sorted(t_loop)[REPEATS // 2]
    nodes = sum(batch.nodes)
    row = {"workload": name, "mode": mode, "models": len(models), "nodes": nodes, "n_split": batch.n_split,
           "batch_ms": round(tb * 1e3, 3), "loop_ms": round(tl * 1e3, 3), "speedup": round(tl / tb, 1),
           "batch_models_per_s": round(len(models) / tb), "loop_models_per_s": round(len(models) / tl),
           "batch_nodes_per_s": round(nodes / tb), "loop_nodes_per_s": round(nodes / tl),
           "kernel_ms": round(batch.kernel_ms, 3), "launches": batch.launches,
           "batch_ms_all": [round(t * 1e3, 3) for t in t_batch], "loop_ms_all": [round(t * 1e3, 3) for t in t_loop]}
    print(json.dumps(row), flush=True)
    for m in models:
        m.close()
    return row


def main():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True, check=True).stdout.splitlines()[0]
    print(json.dumps({"card": card, "device": api.device_info()["name"]}), flush=True)
    a = small_models(10_000)
    run("a", a, "first")
    b = medium_colourings(1_000)
    run("b", b, "first")
    run("b", b, "count")
    big = [sudoku(REFERENCE_SUDOKU, boxes=False, alldiff=True), sudoku(REFERENCE_SUDOKU, boxes=False, alldiff=False)] * 2
    run("c", a + big, "first")


if __name__ == "__main__":
    main()
