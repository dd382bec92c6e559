"""GPU: `bench.py --dump-outputs` writes what the timed path computed, and `--steps` sets every timed loop.  The
benchmark's inputs at these sizes are instances the unmodified reference has answered (tests/golden/reference_large.json:
17-Queens, the first 10 000 puzzles of the Sudoku batch, the first 64 G(200, 4.2/199) 3-colouring instances)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from dequan_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_dump_outputs(golden, golden_large, product_lib, tmp_path):
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                        "--sudoku-n", "10000", "--colouring-n", "64", "--no-cpu", "--dump-outputs", str(out)],
                       capture_output=True, text=True, check=True, timeout=900)
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == line["sudoku"]["steps"] == line["extra"]["colouring"]["steps"] == 2
    assert line["extra"]["nqueens14_1gpu"]["steps"] == 2
    got = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64_000_000

    for n, g in ((17, golden_large["nqueens"]["17"]["count"]), (14, golden["nqueens"]["14"]["count"])):
        assert got[f"nqueens{n}"].tolist() == [g["solutions"], g["nodes"]]
        assert got[f"nqueens{n}_first"].tolist() == g["first"]

    g = golden_large["sudoku10k"]
    assert got["sudoku_index"].tolist() == list(range(g["n"]))
    assert got["sudoku_nodes"].tolist() == g["nodes"] and (got["sudoku_status"] == 1).all()
    assert "".join(map(str, got["sudoku_solution"].astype(np.int64).reshape(-1).tolist())) == g["solutions"]
    assert got["sudoku_totals"].tolist() == [g["n"], 0, 0, sum(g["nodes"])]

    g = [c for c in golden_large["colouring200"] if (c["k"], c["c"]) == (3, 4.2)][0]
    assert got["colouring_index"].tolist() == list(range(g["count"]))
    assert [api.OUTCOME[int(s)] for s in got["colouring_status"]] == g["status"]
    assert got["colouring_nodes"].tolist() == g["nodes"]
    for colours, first in zip(got["colouring_colours"].astype(np.int64).tolist(), g["first"]):
        assert colours == (first if first is not None else [255] * g["n_vertices"])
    assert got["colouring_totals"].tolist() == [g["status"].count(s) for s in ("sat", "unsat", "budget")] + [sum(g["nodes"])]
