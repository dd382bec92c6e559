"""dq_solve_models / api.solve_models / b200::SolveAll: many independent models in one call.  Every batch below is one
call, and each model's status, solution count, node count and first solution must be what the reference (goldens),
the oracle and a single dq_solve_tree of the same handle report."""
import ctypes as C
import json
import os
import random
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from dequan_b200 import api
from dequan_b200.model import CSP, REFERENCE_SUDOKU, DomainType, Op, OpConstraint, nqueens, sudoku
from randmodels import dup_suite, model_suite, random_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _got(r, i):
    return (r.status[i], r.solutions[i], r.nodes[i], r.first[i])


def _tree(t):
    return (t.status, t.solutions, t.nodes, t.first)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["first", "count"])
def test_reference_goldens(product_lib, golden, mode):
    gs = golden["random_suite"]
    models = [api.Model(c) for c in model_suite(gs["n"], gs["seed0"])]
    r = api.solve_models(models, "count" if mode == "count" else "first")
    for i, want in enumerate(gs[mode]):
        assert _got(r, i) == (want["status"], want["solutions"], want["nodes"], want["first"]), (mode, i)
    g = json.load(open(os.path.join(GOLD, "reference_dups.json")))["duplicate_values"]
    models = [api.Model(c) for c in dup_suite(g["n"], g["seed0"])]
    r = api.solve_models(models, mode)
    for i, want in enumerate(g[mode]):
        assert _got(r, i) == (want["status"], want["solutions"], want["nodes"], want["first"]), (mode, i)


def _op_inequality():
    csp = CSP()                                            # test/main-test.cpp:187-233
    v = [csp.AddIntVar(0, 10), csp.AddIntVar(0, 10), csp.AddFixedVar(6), csp.AddFixedVar(5)]
    csp.AddConstraint(OpConstraint(v[0], v[2], Op.Inf, 0))
    csp.AddConstraint(OpConstraint(v[0], v[3], Op.SupEqual, 0))
    csp.AddConstraint(OpConstraint(v[1], v[2], Op.InfEqual, 0))
    csp.AddConstraint(OpConstraint(v[1], v[3], Op.Sup, 0))
    csp.FinalizeModel()
    return csp


def _ring1022():                                           # the 1022-variable model of test_maximum_sizes_and_limits
    csp = CSP()
    n = 1022
    rng = random.Random(4)
    for i in range(n):
        csp.AddIntVar(0, 3 + (i * 7) % 3)
    for i in range(n):
        csp.AddConstraint(OpConstraint(i, (i + 1) % n, Op.NotEqual, 0))
    for _ in range(1100):
        a, b = rng.sample(range(n), 2)
        csp.AddConstraint(OpConstraint(a, b, Op.NotEqual, rng.choice([0, 1, -1])))
    csp.FinalizeModel()
    return csp


def _size(d):
    return len(d.values) if d.type == DomainType.Values else sum(d.values[i + 1] - d.values[i] for i in range(0, len(d.values), 2))


def _mixed(mode):
    """(name, CSP) in batch order: every word width and state size class.  The all-solutions trees of the rows+columns
    Sudoku scenarios are far too large to count, so they and the 1022-variable ring are in the FIRST batch only."""
    out = [("OpInequalityTest", _op_inequality()), ("NQueensTest8", nqueens(8)),
           ("Sudoku_boxes_alldiff", sudoku(REFERENCE_SUDOKU, boxes=True, alldiff=True)),
           ("Sudoku_boxes_binary", sudoku(REFERENCE_SUDOKU, boxes=True, alldiff=False))]
    if mode == "first":
        out += [("SudokuTest_rows_cols_alldiff", sudoku(REFERENCE_SUDOKU, boxes=False, alldiff=True)),
                ("Sudoku_rows_cols_binary", sudoku(REFERENCE_SUDOKU, boxes=False, alldiff=False)),
                ("ring1022", _ring1022())]
    out += [(f"queens{n}", nqueens(n)) for n in range(1, 14)]
    for s in range(40):                                    # 33..64 values: the 64-bit domain word launch
        csp = random_model(700 + s, 3 + s % 2, 3, 48)
        if max(_size(d) for d in csp.domains) > 32:
            out.append((f"wide{s}", csp))
    empty = CSP()
    empty.FinalizeModel()
    out.append(("empty", empty))
    return out


@pytest.fixture(scope="module", params=["first", "count"])
def mixed(request, product_lib):
    mode = request.param
    named = _mixed(mode)
    models = [api.Model(c) for _, c in named]
    assert sum(m.info()["max_dom"] > 32 for m in models) >= 5
    # the same handle twice
    named.append(("NQueensTest8 again", named[1][1]))
    models.append(models[1])
    return mode, named, models


@pytest.mark.gpu
def test_mixed_against_oracle(mixed):
    mode, named, models = mixed
    r = api.solve_models(models, mode)
    assert 1 <= r.n_split < len(models)
    names = [n for n, _ in named]
    # trees no warp budget below 2^20 can finish go through the split search
    assert r.nodes[names.index("SudokuTest_rows_cols_alldiff" if mode == "first" else "queens13")] > 1 << 20
    for i, (name, csp) in enumerate(named):
        if name == "empty":                                # IsComplete at entry: SAT, one solution, no node
            assert _got(r, i) == ("sat", 1, 0, []), name
            continue
        o = O.solve(csp, mode)
        assert _got(r, i) == (o.status, o.solutions, o.nodes, o.first), (mode, name)


@pytest.mark.gpu
def test_batch_equals_single_solves(mixed):
    mode, named, models = mixed
    before = [_tree(m.solve_tree(mode)) for m in models]
    r = api.solve_models(models, mode)
    after = [_tree(m.solve_tree(mode)) for m in models]
    for i, (name, _) in enumerate(named):
        assert _got(r, i) == before[i] == after[i], (mode, name)


def _raw(handles, **kw):
    o = api.dq_tree_opts(kw.get("mode", api.DQ_MODE_FIRST), kw.get("split_depth", 0), 0, kw.get("part_count", 1),
                         kw.get("node_budget", 0), kw.get("engine", 0), 0)
    n = len(handles)
    hs = (C.c_void_p * max(n, 1))(*handles)
    outcome = np.full(max(n, 1), 7, dtype=np.int32)
    u = np.zeros(max(n, 1), dtype=np.uint64)
    split = C.c_int64(-1)
    rc = api.lib().dq_solve_models(hs, n, C.byref(o), outcome.ctypes.data_as(C.POINTER(C.c_int32)), u.ctypes.data,
                                   u.ctypes.data, None, C.byref(split), None)
    return rc, outcome, split.value


def test_refusals(product_lib):
    """Options the batch does not serve, and malformed arguments, are refused before any device work."""
    m = api.Model(nqueens(6))
    h = [m._h.value]
    assert _raw(h, part_count=2)[0] == -2
    assert _raw(h, split_depth=3)[0] == -2
    assert _raw(h, node_budget=100)[0] == -2
    assert _raw(h, engine=api.ENGINE["lane"])[0] == -2
    assert _raw(h, engine=api.ENGINE["reg"])[0] == -2
    assert _raw(h, mode=5)[0] == -1
    assert _raw([h[0], None])[0] == -1
    rc, outcome, split = _raw([])
    assert rc == 0 and split == 0 and outcome[0] == 7


@pytest.mark.gpu
def test_repeated_rounds_give_back_memory(product_lib):
    import torch
    suite = model_suite(60, 1000)

    def round_():
        models = [api.Model(c) for c in suite] + [api.Model(nqueens(10))]
        r = api.solve_models(models, "count")
        for m in models:
            m.close()
        assert r.n_split >= 1
        return r.status, r.solutions, r.nodes, r.first

    want = round_()
    for _ in range(2):
        assert round_() == want
    free = torch.cuda.mem_get_info(0)[0]
    for _ in range(100):
        assert round_() == want
    assert torch.cuda.mem_get_info(0)[0] == free, "device memory not given back"


@pytest.mark.gpu
def test_dropin_solve_all(product_lib, tmp_path):
    out = str(tmp_path / "solve_all")
    libdir = os.path.join(ROOT, "dequan_b200", "lib")
    subprocess.check_call(["g++", "-std=c++11", "-O2", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o", out,
                           os.path.join(ROOT, "tests", "cpp", "solve_all.cpp"), "-L" + libdir, "-ldequan_b200", "-Wl,-rpath," + libdir])
    lines = [json.loads(l) for l in subprocess.run([out], capture_output=True, text=True, check=True, timeout=600).stdout.splitlines()]
    batch = [{k: v for k, v in l.items() if k != "path"} for l in lines if l["path"] == "all"]
    step = [{k: v for k, v in l.items() if k != "path"} for l in lines if l["path"] == "step"]
    assert len(batch) == len(step) == 17
    for b, s in zip(batch, step):
        assert b == s, b["name"]
    by_name = {b["name"]: b for b in batch}
    assert by_name["nqueens8"]["assigned_vars"] == 88 and by_name["op_inequality"]["ok"]
    assert by_name["shared_queens9_full"] == dict(by_name["shared_queens9_full_again"], name="shared_queens9_full")
    assert by_name["shared_queens9_col0_in_4_7"]["values"][0] in (4, 5, 6)
