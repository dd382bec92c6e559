"""GPU: the CUDA engines, through the C ABI, against the CPU oracle and the committed fixtures
captured from the unmodified reference.  Bit-exact: status, solution count, node count
(Assignment::AssignVar calls, dequan.h:416-423) and DFS-first solution."""
import hashlib
import os

import numpy as np
import pytest

import oracle_lib as O
from dequan_b200 import api
from dequan_b200 import generators as G
from dequan_b200.model import (CSP, AllDifferentConstraint, REFERENCE_SUDOKU, Op, OpConstraint, colouring, nqueens, sudoku,
                               sudoku_template)
from randmodels import model_suite, random_model

pytestmark = pytest.mark.gpu

ENGINES = ["warp", "lane", "auto"]


def _cmp_tree(got, want, what):
    assert (got.status, got.solutions, got.nodes, got.first) == (want.status, want.solutions, want.nodes, want.first), (what, got, want)


def test_device_is_blackwell(product_lib):
    info = api.device_info()
    assert info["cc"] >= 100, info


def test_reference_scenarios(golden, product_lib):
    """The three scenarios of /root/reference/test/main-test.cpp plus the boxed variants."""
    csp = CSP()
    v = [csp.AddIntVar(0, 10), csp.AddIntVar(0, 10), csp.AddFixedVar(6), csp.AddFixedVar(5)]
    csp.AddConstraint(OpConstraint(v[0], v[2], Op.Inf, 0))
    csp.AddConstraint(OpConstraint(v[0], v[3], Op.SupEqual, 0))
    csp.AddConstraint(OpConstraint(v[1], v[2], Op.InfEqual, 0))
    csp.AddConstraint(OpConstraint(v[1], v[3], Op.Sup, 0))
    cases = {
        "OpInequalityTest": csp,
        "NQueensTest8": nqueens(8),
        "SudokuTest_rows_cols_alldiff": sudoku(REFERENCE_SUDOKU, boxes=False, alldiff=True),
        "Sudoku_rows_cols_binary": sudoku(REFERENCE_SUDOKU, boxes=False, alldiff=False),
        "Sudoku_boxes_alldiff": sudoku(REFERENCE_SUDOKU, boxes=True, alldiff=True),
        "Sudoku_boxes_binary": sudoku(REFERENCE_SUDOKU, boxes=True, alldiff=False),
    }
    for name, model in cases.items():
        g = golden["reference_tests"][name]
        r = api.Model(model).solve_tree("first")
        assert (r.status, r.nodes, r.first) == (g["status"], g["nodes"], g["first"]), (name, r)


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("n", list(range(1, 14)))
def test_nqueens_count_and_first(golden, product_lib, engine, n):
    g = golden["nqueens"][str(n)]
    m = api.Model(nqueens(n))
    c = m.solve_tree("count", engine=engine)
    assert (c.solutions, c.nodes, c.first) == (g["count"]["solutions"], g["count"]["nodes"], g["count"]["first"]), c
    if engine == "lane":
        if n >= 3:          # (the bucket search wants three variables: smaller boards go to the generic engines)
            assert c.engine == "lane"
        with pytest.raises(api.DequanError):   # the lane engines serve COUNT_ALL only; FIRST runs on the warp engines
            m.solve_tree("first", engine=engine)
        return
    f = m.solve_tree("first", engine=engine)
    assert (f.status, f.nodes, f.first) == (g["first"]["status"], g["first"]["nodes"], g["first"]["first"]), f


@pytest.mark.parametrize("n", [15, 17, 18, 20, 22])
def test_queens_first_mode_on_the_class(product_lib, n):
    """FIRST mode on the N-Queens class: one warp walks the reference's DFS; solution and node count against the oracle
    (20-Queens: 145 151 nodes).  The count a later dq_tree_nodes_upto reports is the same."""
    csp = nqueens(n)
    want = O.solve(csp, "first")
    m = api.Model(csp)
    r = m.solve_tree("first")
    assert (r.status, r.nodes, r.first) == (want.status, want.nodes, want.first) and r.engine == "lane"
    assert m.nodes_upto(r.first_key) == want.nodes
    w = m.solve_tree("first", engine="warp")
    assert (w.status, w.nodes, w.first) == (want.status, want.nodes, want.first)


@pytest.mark.parametrize("engine", ENGINES)
def test_nqueens14_config(golden, product_lib, engine):
    """BASELINE config C2: 365 596 solutions, 19 787 662 nodes, first 0,2,4,6,11,9,12,3,13,8,1,5,7,10."""
    g = golden["nqueens"]["14"]["count"]
    c = api.Model(nqueens(14)).solve_tree("count", engine=engine)
    assert (c.solutions, c.nodes, c.first) == (365596, 19787662, g["first"]) == (g["solutions"], g["nodes"], g["first"])


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("depth", [1, 2, 3, 5])
def test_split_depth_invariance(golden, product_lib, engine, depth):
    g = golden["nqueens"]["9"]
    m = api.Model(nqueens(9))
    c = m.solve_tree("count", split_depth=depth, engine=engine)
    assert (c.solutions, c.nodes, c.first) == (g["count"]["solutions"], g["count"]["nodes"], g["count"]["first"])
    if engine != "lane":
        f = m.solve_tree("first", split_depth=depth, engine=engine)
        assert (f.nodes, f.first) == (g["first"]["nodes"], g["first"]["first"])


@pytest.mark.parametrize("mode", ["first", "count"])
def test_random_suite_vs_golden(golden, product_lib, mode):
    gs = golden["random_suite"]
    suite = model_suite(gs["n"], gs["seed0"])
    for i, (csp, g) in enumerate(zip(suite, gs[mode])):
        r = api.Model(csp).solve_tree(mode)
        assert (r.status, r.solutions, r.nodes, r.first) == (g["status"], g["solutions"], g["nodes"], g["first"]), (i, r, g)


def test_random_larger_models_vs_oracle(product_lib):
    for seed in range(5000, 5060):
        csp = random_model(seed, n_vars=12, n_cons=20, max_dom=7)
        for mode in ("first", "count"):
            _cmp_tree(api.Model(csp).solve_tree(mode), O.solve(csp, mode), (seed, mode))


@pytest.mark.parametrize("engine", ["warp", "lane"])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_partitions_sum_to_whole(golden, product_lib, world, engine):
    """Multi-GPU split emulated on one device: prefix i -> partition i % world."""
    g = golden["nqueens"]["10"]
    m = api.Model(nqueens(10))
    parts = [m.solve_tree("count", split_depth=3, part_rank=r, part_count=world, engine=engine) for r in range(world)]
    assert sum(p.solutions for p in parts) == g["count"]["solutions"]
    assert sum(p.nodes for p in parts) == g["count"]["nodes"]
    key = min(p.first_key for p in parts)
    assert [p.first for p in parts if p.first_key == key][0] == g["count"]["first"]
    if engine == "lane":
        return
    # FIRST mode: min key wins; node accounting re-asked for the global key
    for csp, want in ((nqueens(10), g["first"]), (nqueens(6), golden["nqueens"]["6"]["first"])):
        models = [api.Model(csp) for _ in range(world)]
        loc = [mm.solve_tree("first", split_depth=2, part_rank=r, part_count=world) for r, mm in enumerate(models)]
        key = min(p.first_key for p in loc)
        assert sum(mm.nodes_upto(key) for mm in models) == want["nodes"]
        assert [p.first for p in loc if p.first_key == key][0] == want["first"]


def test_edge_cases(product_lib):
    # no variables: IsComplete at entry (dequan.h:496-499)
    r = api.Model(CSP()).solve_tree("first")
    assert (r.status, r.nodes) == ("sat", 0)
    # one variable, empty domain
    csp = CSP()
    csp.AddIntVar(3, 3)
    _cmp_tree(api.Model(csp).solve_tree("first"), O.solve(csp, "first"), "empty domain")
    # unsat by a wiped-out given: two fixed vars that must differ but are equal
    csp = CSP()
    a, b, c = csp.AddFixedVar(2), csp.AddFixedVar(2), csp.AddIntVar(0, 3)
    csp.AddConstraint(OpConstraint(a, b, Op.NotEqual, 0))
    csp.AddConstraint(OpConstraint(b, c, Op.Inf, 0))
    for mode in ("first", "count"):
        _cmp_tree(api.Model(csp).solve_tree(mode), O.solve(csp, mode), "wiped given")
    # 32-value domains and 2-queens..3-queens (UNSAT trees)
    csp = CSP()
    xs = [csp.AddIntVar(0, 32) for _ in range(3)]
    csp.AddConstraint(OpConstraint(xs[0], xs[1], Op.Sup, 29))
    csp.AddConstraint(OpConstraint(xs[2], xs[1], Op.Equal, 1))
    for mode in ("first", "count"):
        _cmp_tree(api.Model(csp).solve_tree(mode), O.solve(csp, mode), "32-wide")
    with pytest.raises(api.DequanError):
        api.Model(nqueens(4)).solve_tree("first", node_budget=5)


@pytest.mark.parametrize("giv", [30, 40, 24])
def test_sudoku_batch_vs_golden(golden, product_lib, giv):
    g = golden[f"sudoku_g{giv}"]
    cells = G.sudoku_batch(g["n"], givens=giv, seed=g["seed"])
    r = api.Model(sudoku_template()).solve_batch_cells(cells)
    assert r.nodes.tolist() == g["nodes"]
    assert [api.OUTCOME[s] for s in r.status] == g["status"]
    assert ["".join(map(str, row)) for row in r.solution] == g["solution"]
    assert r.total_nodes == sum(g["nodes"]) and r.n_sat == g["n"]


def test_sudoku_batch_budget_and_unsat(product_lib):
    cells = G.sudoku_batch(64, givens=26)
    tmpl = api.Model(sudoku_template())
    full = tmpl.solve_batch_cells(cells)
    budget = int(np.median(full.nodes))
    r = tmpl.solve_batch_cells(cells, node_budget=budget)
    for i in range(64):
        o = O.solve(sudoku(cells[i]), "first", budget)
        assert (api.OUTCOME[r.status[i]], int(r.nodes[i])) == (o.status, o.nodes), i
        if o.status == "sat":
            assert r.solution[i].tolist() == o.first
        else:
            assert not r.solution[i].any()
    assert 0 < r.n_budget < 64
    # contradictory givens -> UNSAT with the reference's node count; bytes outside 1..9 -> status 3
    bad = cells[:4].copy()
    bad[0, 0], bad[0, 1] = 5, 5
    bad[1, 0] = 200
    r = tmpl.solve_batch_cells(bad)
    o = O.solve(sudoku(bad[0]), "first")
    assert (api.OUTCOME[r.status[0]], int(r.nodes[0])) == (o.status, o.nodes) and o.status == "unsat"
    assert r.status[1] == 3
    assert r.status[2] == 1 and r.status[3] == 1


def test_sudoku_batch_mixed_blank_counts(product_lib):
    """The lanes' stacks are sized for the batch's largest number of blanks: an empty grid (81 blanks), a solved grid (none)
    and a 17-given-like sparse grid next to 30-given puzzles, each against the oracle."""
    cells = G.sudoku_batch(24, givens=30, seed=3)
    tmpl = api.Model(sudoku_template())
    solved = tmpl.solve_batch_cells(cells[:1]).solution[0]
    cells[0] = 0
    cells[1] = solved
    sparse = solved.copy()
    sparse[np.arange(81) % 4 != 0] = 0          # 21 givens of a valid grid
    cells[2] = sparse
    r = tmpl.solve_batch_cells(cells)
    for i in range(len(cells)):
        o = O.solve(sudoku(cells[i]), "first", 3_000_000)
        assert (api.OUTCOME[r.status[i]], int(r.nodes[i])) == (o.status, o.nodes), i
        assert r.solution[i].tolist() == o.first, i
    assert int(r.nodes[1]) == 81


def test_sudoku_hard_batch_recycles_snapshots(product_lib):
    """Hard puzzles (24 givens, 2e4 nodes each on average) split into millions of pieces: the snapshot ring recycles its
    slots (round 1's linear pool ran out, after which no task could split).  The per-instance node counts do not depend
    on how the work was cut — default splitting against forced splitting every 64 nodes — and a sample agrees with the
    oracle."""
    n = 30_000
    cells = G.sudoku_batch(n, givens=24, seed=11)
    tmpl = api.Model(sudoku_template())
    a = tmpl.solve_batch_cells(cells)
    b = tmpl.solve_batch_cells(cells, task_nodes=64)
    assert a.n_sat == n and (a.status == 1).all()
    assert (a.nodes == b.nodes).all() and (a.solution == b.solution).all() and a.total_nodes == b.total_nodes
    order = np.argsort(a.nodes)
    for i in list(order[:3]) + list(order[n // 2: n // 2 + 3]):
        o = O.solve(sudoku(cells[i]), "first")
        assert (int(a.nodes[i]), a.solution[i].tolist()) == (o.nodes, o.first)


def test_sudoku_batch_unsolvable_without_clash(product_lib):
    """One given of each puzzle replaced by a value its row, column and box do not rule out: no clash for the digest to
    defer, but (mostly) no solution either — the lane pipeline's own unsat / budget paths (exhausted root level in the
    first stage, "whole parked stack" tasks in the counting stage) against the oracle."""
    n = 48
    cells = G.sudoku_batch(n, givens=30, seed=21)
    rng = np.random.default_rng(5)
    for i in range(n):
        g = cells[i].reshape(9, 9)
        given = np.argwhere(g != 0)
        for r, c in given[rng.permutation(len(given))]:
            seen = set(g[r, :]) | set(g[:, c]) | set(g[3 * (r // 3):3 * (r // 3) + 3, 3 * (c // 3):3 * (c // 3) + 3].ravel())
            free = [v for v in range(1, 10) if v not in seen]
            if free:
                g[r, c] = free[0]
                break
    budget = 400_000
    r = api.Model(sudoku_template()).solve_batch_cells(cells, node_budget=budget)
    seen_status = set()
    for i in range(n):
        o = O.solve(sudoku(cells[i]), "first", budget)
        assert (api.OUTCOME[r.status[i]], int(r.nodes[i])) == (o.status, o.nodes), i
        if o.status == "sat":
            assert r.solution[i].tolist() == o.first
        else:
            assert not r.solution[i].any()
        seen_status.add(o.status)
    assert "unsat" in seen_status


def test_sudoku_batch_large_properties(product_lib):
    """Size-independent properties at a size the oracle cannot cover."""
    n = 200_000
    cells = G.sudoku_batch(n, givens=32, seed=7)
    r = api.Model(sudoku_template()).solve_batch_cells(cells)
    assert r.n_sat == n and (r.status == 1).all()
    sol = r.solution.reshape(n, 9, 9)
    want = np.arange(1, 10)
    assert (np.sort(sol, axis=2) == want).all() and (np.sort(sol, axis=1) == want[:, None]).all()
    boxes = sol.reshape(n, 3, 3, 3, 3).transpose(0, 1, 3, 2, 4).reshape(n, 9, 9)
    assert (np.sort(boxes, axis=2) == want).all()
    assert (sol.reshape(n, 81)[cells != 0] == cells[cells != 0]).all()
    assert (r.nodes >= 81).all() and int(r.nodes.sum()) == r.total_nodes
    # idempotence: a solved grid is its own solution in exactly 81 nodes
    again = api.Model(sudoku_template()).solve_batch_cells(np.ascontiguousarray(r.solution[:1000]))
    assert (again.solution == r.solution[:1000]).all() and (again.nodes == 81).all()
    # spot-check 50 against the oracle
    for i in range(0, n, n // 50):
        o = O.solve(sudoku(cells[i]), "first")
        assert (int(r.nodes[i]), r.solution[i].tolist()) == (o.nodes, o.first)


def test_colouring_batch_vs_golden(golden, product_lib):
    for case in golden["colouring"]:
        off, edges = G.colouring_batch(case["count"], case["n_vertices"], case["c"])
        assert hashlib.sha256(edges.tobytes()).hexdigest() == case["sha256"]
        r = api.solve_batch_graphs(case["n_vertices"], case["k"], off, edges, node_budget=case["budget"])
        assert [api.OUTCOME[s] for s in r.status] == case["status"]
        assert r.nodes.tolist() == case["nodes"]
        for i, first in enumerate(case["first"]):
            if first is not None:
                assert r.solution[i].tolist() == first
            else:
                assert (r.solution[i] == 0xFF).all()


def test_colouring_200_vs_oracle(product_lib):
    """BASELINE config C4 shape: G(200, c/199), node budget, tri-state result."""
    off, edges = G.colouring_batch(24, 200, 3.6, seed=11)
    r = api.solve_batch_graphs(200, 3, off, edges, node_budget=50_000)
    for i in range(24):
        o = O.solve(colouring(200, 3, edges[off[i]:off[i + 1]]), "first", 50_000)
        assert (api.OUTCOME[r.status[i]], int(r.nodes[i])) == (o.status, o.nodes), i
        if o.status == "sat":
            assert r.solution[i].tolist() == o.first
            e = edges[off[i]:off[i + 1]]
            assert (r.solution[i][e[:, 0]] != r.solution[i][e[:, 1]]).all()
    # the same instances as single-tree models through dq_solve_tree agree too (no budget: only the solved ones)
    for i in range(24):
        if r.status[i] == 1 and r.nodes[i] < 20000:
            t = api.Model(colouring(200, 3, edges[off[i]:off[i + 1]])).solve_tree("first")
            assert (t.nodes, t.first) == (int(r.nodes[i]), r.solution[i].tolist())


def test_lane_engine_rejects_other_models(product_lib):
    with pytest.raises(api.DequanError):
        api.Model(nqueens(6)).solve_tree("first", engine="lane")
    with pytest.raises(api.DequanError):
        api.Model(sudoku(REFERENCE_SUDOKU)).solve_tree("count", engine="lane")


@pytest.mark.parametrize("n,k", [(15, 0), (16, 0), (18, 0), (12, 1), (12, 7), (13, 10), (13, 1), (14, 2), (16, 11)])
def test_lane_engine_larger_boards(golden, golden_large, product_lib, n, k):
    """N <= 14: tests/golden/reference.json; N = 15 .. 18: tests/golden/reference_large.json — both are outputs of the
    unmodified reference (solutions, stats.assigned_vars, DFS-first solution).  k = 0: the engine's own split depth (the
    bucket kernel compiled for its bucket count); (13, 1), (14, 2): nine buckets and (13, 10): none of its own, i.e. the
    general bucket kernel; (12, 7), (16, 11): two buckets."""
    g = (golden if n <= 14 else golden_large)["nqueens"][str(n)]["count"]
    r = api.Model(nqueens(n)).solve_tree("count", engine="lane", split_depth=k)
    assert (r.solutions, r.nodes, r.first) == (g["solutions"], g["nodes"], g["first"]) and r.engine == "lane"


@pytest.mark.parametrize("n", [15, 16])
def test_first_value_subtrees_vs_reference(golden_large, product_lib, n):
    """The reference's per-first-row-value runs (variable 0 fixed to v by a singleton domain: SURVEY.md section 8c) against
    the same models here: the fixed variable leaves the N-Queens class, so this is the generic path at 10^7-node size."""
    per = golden_large["nqueens"][str(n)]["per_first_value"]
    assert len(per) == n
    for v in (0, n // 2, n - 1):
        csp = nqueens(n)
        csp.domains[0] = type(csp.domains[0])(0, [v])          # Domain(Values, {v})
        r = api.Model(csp).solve_tree("count")
        assert (r.solutions, r.nodes) == (per[v]["solutions"], per[v]["nodes"]), (n, v, r)


def test_int_peak_microbenchmark(product_lib):
    ops, ms = api.measure_int_peak()
    assert 5e12 < ops < 4e13, ops


def test_caller_supplied_assign_order_vs_oracle(product_lib):
    """Assignment::assign_order is a public field (dequan.h:316): a caller-edited order reaches the engine."""
    import random
    for seed in range(7000, 7040):
        csp = random_model(seed, n_vars=9, n_cons=14, max_dom=6)
        order = list(range(9))
        random.Random(seed).shuffle(order)
        csp.assign_order = order
        m = api.Model(csp)
        assert m.order() == order
        for mode in ("first", "count"):
            _cmp_tree(m.solve_tree(mode), O.solve(csp, mode), (seed, mode))


def test_queens_with_caller_order_leaves_the_class_engine(product_lib):
    """The N-Queens class engine walks the variables in id order: a model whose caller-supplied assign_order is
    anything else must count through the generic engine, and agree with the oracle (node counts depend on the order)."""
    import random
    for n, seed in ((7, 1), (8, 2), (9, 3)):
        csp = nqueens(n)
        order = list(range(n))
        random.Random(seed).shuffle(order)
        csp.assign_order = order
        m = api.Model(csp)
        assert m.order() == order and m.info()["model_class"] != "queens"
        for mode in ("first", "count"):
            _cmp_tree(m.solve_tree(mode), O.solve(csp, mode), (n, mode))
        _cmp_tree(m.solve_tree("count", engine="lane"), O.solve(csp, "count"), (n, "generic lane engine"))
    csp = nqueens(8)
    csp.assign_order = list(range(8))                    # the identity, spelled out, still qualifies
    m = api.Model(csp)
    assert m.info()["model_class"] == "queens" and m.solve_tree("count").engine == "lane"


# ---- lane-per-instance Sudoku engine (dq_lane_sudoku.cuh): task splitting must not change any result ----

def _same_batch(a, b, what):
    assert (a.status == b.status).all(), what
    assert (a.nodes == b.nodes).all(), (what, np.nonzero(a.nodes != b.nodes)[0][:5])
    assert (a.solution == b.solution).all(), what
    assert (a.n_sat, a.n_unsat, a.n_budget, a.total_nodes) == (b.n_sat, b.n_unsat, b.n_budget, b.total_nodes), what


def test_sudoku_template_is_recognised(product_lib):
    assert api.Model(sudoku_template()).info()["model_class"] == "sudoku9"
    assert api.Model(sudoku([0] * 81, alldiff=True)).info()["model_class"] == "sudoku9"
    assert api.Model(sudoku_template(boxes=False)).info()["model_class"] == "ne_same"      # a Latin square is not a Sudoku
    assert api.Model(sudoku(REFERENCE_SUDOKU)).info()["model_class"] == "generic"          # givens baked into the template


@pytest.mark.parametrize("task_nodes", [16, 200, 3000, 0])
@pytest.mark.parametrize("giv", [24, 28, 36])
def test_sudoku_lane_engine_equals_warp_engine(product_lib, giv, task_nodes):
    """Whatever the split granularity, the lane engine reproduces the generic warp engine (itself pinned to the
    reference by the golden vectors) on every instance: status, node count, solution."""
    n = 1500 if giv == 24 else 6000
    cells = G.sudoku_batch(n, givens=giv, seed=99 + giv)
    tmpl = api.Model(sudoku_template())
    want = tmpl.solve_batch_cells(cells, engine="warp")
    got = tmpl.solve_batch_cells(cells, engine="lane", task_nodes=task_nodes)
    _same_batch(got, want, (giv, task_nodes))


def test_sudoku_lane_engine_unsat_budget_and_odd_inputs(product_lib):
    rng = np.random.default_rng(5)
    cells = G.sudoku_batch(3000, givens=27, seed=123)
    # no solution, but no two givens clash: overwrite one given with another value that is still free in its units
    broken = 0
    for i in range(0, 3000, 3):
        g = cells[i].reshape(9, 9)
        rs, cs = np.nonzero(g)
        for j in rng.permutation(len(rs)):
            r, c = rs[j], cs[j]
            used = set(g[r]) | set(g[:, c]) | set(g[r // 3 * 3:r // 3 * 3 + 3, c // 3 * 3:c // 3 * 3 + 3].ravel())
            free = [v for v in range(1, 10) if v not in used]
            if free:
                g[r, c] = free[0]
                broken += 1
                break
    assert broken > 900
    cells[1] = 0                                   # all blank
    cells[4] = G.sudoku_batch(1, givens=81, seed=4)[0]   # nothing blank
    cells[7, 0], cells[7, 1] = 5, 5                # clashing givens -> generic engine, exact node count
    cells[10, 3] = 77                              # a byte outside the template domain -> status 3
    tmpl = api.Model(sudoku_template())
    want = tmpl.solve_batch_cells(cells, engine="warp")
    assert want.n_unsat > 300 and want.status[10] == 3
    for tn in (32, 700, 0):
        _same_batch(tmpl.solve_batch_cells(cells, engine="lane", task_nodes=tn), want, tn)
    for budget in (60, 81, 300, 5000):
        wb = tmpl.solve_batch_cells(cells, engine="warp", node_budget=budget)
        for tn in (50, 0):
            _same_batch(tmpl.solve_batch_cells(cells, engine="lane", node_budget=budget, task_nodes=tn), wb, (budget, tn))
    # padded rows (stride > 81)
    wide = np.zeros((500, 96), dtype=np.uint8)
    wide[:, :81] = cells[:500]
    gw = tmpl.solve_batch_cells(wide, engine="lane", task_nodes=100)
    assert (gw.nodes == want.nodes[:500]).all() and (gw.solution[:, :81] == want.solution[:500]).all()
    with pytest.raises(api.DequanError):
        api.Model(sudoku_template(boxes=False)).solve_batch_cells(cells[:8], engine="lane")


def test_batches_from_on_disk_formats(product_lib):
    """81-character Sudoku lines and DIMACS .col text go through the parsers into the batch entry points."""
    cells = G.sudoku_batch(300, givens=31, seed=77)
    parsed = api.parse_sudoku_lines("\n".join(G.sudoku_lines(cells)) + "\n")
    tmpl = api.Model(sudoku_template())
    _same_batch(tmpl.solve_batch_cells(parsed), tmpl.solve_batch_cells(cells), "sudoku lines")
    edges = G.colouring_instance(60, 3.0, 20261018, 3)
    text = f"c G(60, 3/59)\np edge 60 {len(edges)}\n" + "".join(f"e {u + 1} {v + 1}\n" for u, v in edges)
    nv, pe = api.parse_dimacs_col(text)
    off = np.array([0, len(pe)], dtype=np.int64)
    r = api.solve_batch_graphs(nv, 3, off, pe, node_budget=20000)
    o = O.solve(colouring(60, 3, [tuple(e) for e in edges.tolist()]), "first", 20000)
    assert (api.OUTCOME[r.status[0]], int(r.nodes[0])) == (o.status, o.nodes)


def test_maximum_sizes_and_limits(product_lib):
    """254 variables (the widest batch template) and 1022 (the engine's limit) with mixed domain sizes; the first size
    beyond each limit (1023 variables, 65 values) is refused with an error, not approximated; empty batches are no-ops."""
    import random
    rng = random.Random(3)
    csp = CSP()
    n = 254
    for i in range(n):
        csp.AddIntVar(0, 32 if i % 50 == 0 else 2)
    for i in range(n - 1):
        csp.AddConstraint(OpConstraint(i, i + 1, Op.NotEqual, 0))
    for _ in range(40):
        a, b = rng.sample(range(n), 2)
        csp.AddConstraint(OpConstraint(a, b, Op.NotEqual, rng.choice([0, 1])))
    _cmp_tree(api.Model(csp).solve_tree("first"), O.solve(csp, "first"), "254 variables")
    # 1022 variables: a ring of different-neighbour constraints with 1100 chords, domains of 3..5 values
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
    m = api.Model(csp)
    want = O.solve(csp, "first")
    _cmp_tree(m.solve_tree("first"), want, "1022 variables")
    _cmp_tree(m.solve_tree("first", split_depth=5), want, "1022 variables, split")
    # a 16x16 Sudoku (256 variables on 1..16), 4 of every 7 cells blank: 514 140 nodes to the first solution
    base = [[(4 * (r % 4) + r // 4 + c) % 16 + 1 for c in range(16)] for r in range(16)]
    s16 = CSP()
    for r in range(16):
        for c in range(16):
            if (r * 16 + c) % 7 < 4:
                s16.AddIntVar(1, 17)
            else:
                s16.AddFixedVar(base[r][c])
    groups = [[r * 16 + c for c in range(16)] for r in range(16)] + [[r * 16 + c for r in range(16)] for c in range(16)]
    groups += [[(4 * (b // 4) + i // 4) * 16 + 4 * (b % 4) + i % 4 for i in range(16)] for b in range(16)]
    for g in groups:
        s16.AddConstraint(AllDifferentConstraint(g))
    s16.FinalizeModel()
    want = O.solve(s16, "first")
    assert want.status == "sat" and want.first == [base[r][c] for r in range(16) for c in range(16)]
    _cmp_tree(api.Model(s16).solve_tree("first"), want, "16x16 sudoku")
    big = CSP()
    for _ in range(1023):
        big.AddIntVar(0, 2)
    with pytest.raises(api.DequanError):
        api.Model(big)
    wide = CSP()
    wide.AddIntVar(0, 65)
    with pytest.raises(api.DequanError):
        api.Model(wide)
    tmpl = api.Model(sudoku_template())
    r = tmpl.solve_batch_cells(np.zeros((0, 81), dtype=np.uint8))
    assert (r.n_sat, r.n_unsat, r.total_nodes, len(r.nodes)) == (0, 0, 0, 0)
    r = api.solve_batch_graphs(5, 3, np.zeros(1, dtype=np.int64), np.zeros((0, 2), dtype=np.uint8))
    assert len(r.status) == 0
    # a single instance, and a batch smaller than a warp
    one = G.sudoku_batch(1, givens=30, seed=9)
    _same_batch(tmpl.solve_batch_cells(one), tmpl.solve_batch_cells(one, engine="warp"), "single instance")
    few = G.sudoku_batch(7, givens=26, seed=10)
    _same_batch(tmpl.solve_batch_cells(few), tmpl.solve_batch_cells(few, engine="warp"), "seven instances")


def _graph_lists(nv, c, count, seed=4242):
    lists = [G.colouring_instance(nv, c, seed, i) if nv > 1 else np.zeros((0, 2), dtype=np.uint8) for i in range(count)]
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    for i, e in enumerate(lists):
        off[i + 1] = off[i] + len(e)
    edges = np.ascontiguousarray(np.concatenate(lists, axis=0).astype(np.uint8)) if off[-1] else np.zeros((0, 2), dtype=np.uint8)
    return off, edges


@pytest.mark.parametrize("nv,k,c,budget", [(200, 3, 4.2, 30000), (200, 4, 7.0, 30000), (60, 3, 3.5, 0), (33, 2, 1.2, 0), (1, 3, 0.0, 0),
                                           (254, 4, 6.0, 5000), (64, 1, 0.5, 0), (2, 2, 1.0, 0), (17, 4, 9.0, 0)])
def test_colouring_engines_agree(product_lib, nv, k, c, budget):
    """The lane-per-instance engine (dq_group_graphs.cuh) and the register-resident warp engine (dq_reg_graphs.cuh)
    against the generic warp engine, itself pinned to the reference."""
    off, edges = _graph_lists(nv, c, 96)
    b = api.solve_batch_graphs(nv, k, off, edges, node_budget=budget, engine="warp")
    a = api.solve_batch_graphs(nv, k, off, edges, node_budget=budget, engine="lane")
    _same_batch(a, b, (nv, k, c, budget, "lane"))
    assert a.launches == 3
    _same_batch(api.solve_batch_graphs(nv, k, off, edges, node_budget=budget), b, (nv, k, c, budget, "auto"))
    r = api.solve_batch_graphs(nv, k, off, edges, node_budget=budget, engine="reg")
    _same_batch(r, b, (nv, k, c, budget, "reg"))
    assert r.launches == 1 and b.launches == 2
    with pytest.raises(api.DequanError):        # a self-loop has no lowering (the reference would fail every value of that vertex)
        api.solve_batch_graphs(3, 3, np.array([0, 1], dtype=np.int64), np.array([[1, 1]], dtype=np.uint8))


@pytest.mark.parametrize("engine", ["lane", "reg"])
def test_colouring_c4_vs_reference(golden_large, product_lib, engine):
    """BASELINE config C4 as stated — G(200, c/199), k=3 c in {4.0, 4.2, 4.4, 4.69}, k=4 c in {6, 7}, 64 instances each,
    budget 100 000 nodes — against what the unmodified reference returns (tests/golden/make_golden_large.py):
    status, node count and colours per instance."""
    assert len(golden_large["colouring200"]) == 6
    for case in golden_large["colouring200"]:
        off, edges = G.colouring_batch(case["count"], case["n_vertices"], case["c"])
        assert hashlib.sha256(edges.tobytes()).hexdigest() == case["sha256"]
        r = api.solve_batch_graphs(case["n_vertices"], case["k"], off, edges, node_budget=case["budget"], engine=engine)
        assert [api.OUTCOME[s] for s in r.status] == case["status"], (case["k"], case["c"])
        assert r.nodes.tolist() == case["nodes"], (case["k"], case["c"])
        for i, first in enumerate(case["first"]):
            if first is not None:
                assert r.solution[i].tolist() == first
            else:
                assert (r.solution[i] == 0xFF).all()
        assert (r.n_sat, r.n_unsat, r.n_budget) == tuple(case["status"].count(x) for x in ("sat", "unsat", "budget"))
        assert r.total_nodes == sum(case["nodes"])


def test_colouring_device_resident_entry(product_lib):
    """dq_solve_batch_graphs_dev (edge lists and outputs in HBM) against the host-buffer entry point; malformed lists
    are refused by the device-side check."""
    import torch
    off, edges = _graph_lists(60, 3.5, 300)
    want = api.solve_batch_graphs(60, 3, off, edges, node_budget=5000, engine="warp")
    dev = torch.device("cuda", 0)
    pad = (-edges.size) % 16
    d_edges = torch.from_numpy(np.concatenate([edges.reshape(-1), np.zeros(pad, dtype=np.uint8)])).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_col = torch.zeros((300, 60), dtype=torch.uint8, device=dev)
    d_nodes = torch.zeros(300, dtype=torch.int64, device=dev)
    d_status = torch.zeros(300, dtype=torch.uint8, device=dev)
    st = api.solve_batch_graphs_ptr(60, 3, off, d_off.data_ptr(), d_edges.data_ptr(), d_col.data_ptr(), d_nodes.data_ptr(),
                                    d_status.data_ptr(), node_budget=5000, device=True)
    torch.cuda.synchronize()
    assert (d_col.cpu().numpy() == want.solution).all() and (d_nodes.cpu().numpy().astype(np.uint64) == want.nodes).all()
    assert (d_status.cpu().numpy() == want.status).all()
    assert (st.n_sat, st.n_unsat, st.n_budget, st.total_nodes) == (want.n_sat, want.n_unsat, want.n_budget, want.total_nodes)
    bad = d_edges.clone()
    bad[3] = 77                                           # vertex 77 of 60
    with pytest.raises(api.DequanError):
        api.solve_batch_graphs_ptr(60, 3, off, d_off.data_ptr(), bad.data_ptr(), d_col.data_ptr(), d_nodes.data_ptr(),
                                   d_status.data_ptr(), node_budget=5000, device=True)


def test_colouring_group_engine_odd_inputs(product_lib):
    """Duplicate edges, reversed endpoints, empty instances between full ones, a ragged batch that ends in an empty graph."""
    rng = np.random.default_rng(5)
    lists = []
    for i in range(40):
        if i % 7 == 3:
            lists.append(np.zeros((0, 2), dtype=np.uint8))
            continue
        e = G.colouring_instance(40, 3.2, 77, i).astype(np.uint8)
        e = np.concatenate([e, e[: len(e) // 3][:, ::-1]], axis=0)          # duplicates, endpoints swapped
        lists.append(e[rng.permutation(len(e))])
    lists.append(np.zeros((0, 2), dtype=np.uint8))
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    for i, e in enumerate(lists):
        off[i + 1] = off[i] + len(e)
    edges = np.ascontiguousarray(np.concatenate(lists, axis=0))
    b = api.solve_batch_graphs(40, 3, off, edges, engine="warp")
    _same_batch(api.solve_batch_graphs(40, 3, off, edges, engine="lane"), b, "odd")
    _same_batch(api.solve_batch_graphs(40, 3, off, edges), b, "odd, auto")
    for i in (3, 40):
        assert b.status[i] == 1 and b.nodes[i] == 40 and (b.solution[i] == 0).all()
    # budgets on the boundary: an instance that needs exactly B nodes is solved with budget B, and busts with B - 1
    need = int(b.nodes[0])
    one = (off[:2].copy(), edges[: off[1]])
    for budget in (need, need - 1, 1):
        _same_batch(api.solve_batch_graphs(40, 3, *one, node_budget=budget, engine="lane"), api.solve_batch_graphs(40, 3, *one, node_budget=budget, engine="warp"), budget)
    assert api.solve_batch_graphs(40, 3, *one, node_budget=need, engine="lane").status[0] == b.status[0]
    r = api.solve_batch_graphs(40, 3, *one, node_budget=need - 1, engine="lane")
    assert r.status[0] == 2 and r.nodes[0] == need and (r.solution[0] == 0xFF).all()


def test_register_tree_engine_equals_generic_engine(product_lib):
    """dq_small_tree.cuh (domains in registers, models of at most 32 variables) against the generic warp engine and the
    oracle: random models with every constraint kind, both modes, several split depths and partitions."""
    used = 0
    for seed in range(9000, 9120):
        csp = random_model(seed, n_vars=5 + seed % 9, n_cons=6 + seed % 13, max_dom=3 + seed % 5)
        m = api.Model(csp)
        for mode in ("first", "count"):
            want = O.solve(csp, mode)
            a = m.solve_tree(mode, engine="warp")
            _cmp_tree(a, want, (seed, mode, "warp"))
            b = m.solve_tree(mode)
            _cmp_tree(b, want, (seed, mode, "auto"))
            used += b.engine == "reg"
            if b.engine == "reg":
                for depth in (1, 3):
                    _cmp_tree(m.solve_tree(mode, split_depth=depth, engine="reg"), want, (seed, mode, depth))
    print('register engine used', used)
    assert used > 60
    used = 0
    for seed in range(9200, 9260):             # not-equal models: many solutions, the DFS kernel always runs
        csp = random_model(seed, n_vars=7 + seed % 4, n_cons=10 + seed % 9, max_dom=4 + seed % 2, kinds="ne")
        m = api.Model(csp)
        for mode in ("first", "count"):
            want = O.solve(csp, mode)
            b = m.solve_tree(mode)
            _cmp_tree(b, want, (seed, mode, "auto"))
            _cmp_tree(m.solve_tree(mode, engine="warp"), want, (seed, mode, "warp"))
            used += b.engine == "reg"
    assert used > 80
    m = api.Model(nqueens(11))
    g = O.solve(nqueens(11), "count")
    parts = [m.solve_tree("count", split_depth=3, part_rank=r, part_count=3, engine="reg") for r in range(3)]
    assert (sum(p.solutions for p in parts), sum(p.nodes for p in parts)) == (g.solutions, g.nodes)
    for engine, used_engine in (("reg", "reg"), ("auto", "lane")):     # (auto: the class's own first-solution warp)
        f = m.solve_tree("first", engine=engine)
        assert f.engine == used_engine and f.launches == 1 and (f.nodes, f.first) == (O.solve(nqueens(11), "first").nodes, O.solve(nqueens(11), "first").first)
    big = CSP()
    for _ in range(40):
        big.AddIntVar(0, 3)
    with pytest.raises(api.DequanError):
        api.Model(big).solve_tree("first", engine="reg")


def test_enumeration_in_reference_order(product_lib):
    """dq_enumerate_solutions: every solution, in the order the reference's search visits them — against the golden
    lists recorded from the unmodified reference and against the oracle, on both tree engines, split and partitioned."""
    import json
    from enum_models import enum_models
    with open(os.path.join(os.path.dirname(__file__), "golden", "enumerate_reference.json")) as f:
        gold = json.load(f)
    used_reg = 0
    for name, csp in enum_models():
        g = gold["models"][name]
        want, total = O.enumerate_solutions(csp, 100000)
        assert total == g["solutions"] and want[:gold["cap"]] == g["all"], name
        m = api.Model(csp)
        for engine in ("warp", "auto"):
            for depth in (0, 1, 2):
                got, r = m.enumerate_solutions(max(total, 1), split_depth=depth, engine=engine)
                assert got.tolist() == want, (name, engine, depth)
                assert (r.solutions, r.nodes) == (g["solutions"], g["nodes"]), (name, engine, depth)
                used_reg += r.engine == "reg"
        if total > 1:
            with pytest.raises(api.DequanError):
                m.enumerate_solutions(total - 1)
            parts = [m.enumerate_solutions(total, split_depth=2, part_rank=k, part_count=3)[0].tolist() for k in range(3)]
            assert sorted(sum(parts, [])) == sorted(want), name
            pos = {tuple(s): i for i, s in enumerate(want)}
            for p in parts:                                   # each partition's list keeps the global order
                idx = [pos[tuple(s)] for s in p]
                assert idx == sorted(idx), name
    assert used_reg > 100
    csp = nqueens(10)
    want, total = O.enumerate_solutions(csp, 1000)
    got, r = api.Model(csp).enumerate_solutions(1000)
    assert total == 724 and got.tolist() == want and r.nodes == O.solve(csp, "count").nodes


def _max_dom(csp):
    return max(len(d.values) if d.type.name == "Values" else sum(d.values[i + 1] - d.values[i] for i in range(0, len(d.values), 2))
               for d in csp.domains)


def test_domains_up_to_64_values(product_lib):
    """Models whose largest domain has 33..64 values run the generic engine on 64-bit domain words: same counts,
    node counts and first solutions as the oracle, through every split depth and partition count."""
    wide = 0
    for seed in range(9500, 9580):
        csp = random_model(seed, n_vars=3 + seed % 3, n_cons=3 + seed % 5, max_dom=40 + seed % 25)
        m = api.Model(csp)
        is_wide = _max_dom(csp) > 32
        wide += is_wide
        for mode in ("first", "count"):
            want = O.solve(csp, mode)
            _cmp_tree(m.solve_tree(mode), want, (seed, mode))
            for depth in (1, 2):
                _cmp_tree(m.solve_tree(mode, split_depth=depth), want, (seed, mode, depth))
            if is_wide:
                assert m.solve_tree(mode).engine == "warp"
                with pytest.raises(api.DequanError):
                    m.solve_tree(mode, engine="reg")
        if is_wide and seed % 4 == 0:
            g = O.solve(csp, "count")
            parts = [m.solve_tree("count", split_depth=2, part_rank=r, part_count=3) for r in range(3)]
            assert (sum(p.solutions for p in parts), sum(p.nodes for p in parts)) == (g.solutions, g.nodes), seed
    assert wide > 25
    # seven queens on a 50-column board (test/main-test.cpp:36-49 with a wider domain): first solution, node count, and
    # the count of the tree below a fixed first queen
    board = CSP()
    for _ in range(7):
        board.AddIntVar(0, 50)
    for i in range(7):
        for j in range(i + 1, 7):
            for off in (0, j - i, i - j):
                board.AddConstraint(OpConstraint(i, j, Op.NotEqual, off))
    board.FinalizeModel()
    _cmp_tree(api.Model(board).solve_tree("first"), O.solve(board, "first"), "board first")
    # 64 values exactly, and one more is refused
    edge = CSP()
    a = edge.AddIntVar(0, 64); b = edge.AddIntVar(-10, 54); c = edge.AddIntVar(5, 20)
    edge.AddConstraint(OpConstraint(a, b, Op.Equal, 3)); edge.AddConstraint(OpConstraint(c, a, Op.Sup, 40)); edge.AddConstraint(OpConstraint(b, c, Op.NotEqual, -7))
    edge.FinalizeModel()
    for mode in ("first", "count"):
        _cmp_tree(api.Model(edge).solve_tree(mode), O.solve(edge, mode), ("edge", mode))
    big = CSP()
    big.AddIntVar(0, 65); big.AddIntVar(0, 3)
    big.FinalizeModel()
    with pytest.raises(api.DequanError):
        api.Model(big)
    tmpl = CSP()
    for _ in range(4):
        tmpl.AddIntVar(1, 41)
    tmpl.AddConstraint(OpConstraint(0, 1, Op.NotEqual, 0))
    tmpl.FinalizeModel()
    with pytest.raises(api.DequanError):            # batches take 32-bit templates
        api.Model(tmpl).solve_batch_cells(np.zeros((2, 4), dtype=np.uint8))


def test_queens_graph_replay_and_recapture(product_lib):
    """The N-Queens solve queue is replayed as a CUDA graph from the second identical solve on; a change of split depth
    or partition re-captures it.  Every call returns the same exact counts."""
    csp = nqueens(12)
    g = O.solve(csp, "count")
    m = api.Model(csp)
    for _ in range(4):                                          # call-by-call, capture, replay, replay
        r = m.solve_tree("count")
        assert (r.solutions, r.nodes, r.first) == (g.solutions, g.nodes, g.first)
    for rounds in range(2):
        parts = [m.solve_tree("count", part_rank=k, part_count=2) for k in (0, 1, 0, 1)]
        assert (parts[0].solutions + parts[1].solutions, parts[0].nodes + parts[1].nodes) == (g.solutions, g.nodes)
        assert (parts[2].solutions, parts[2].nodes, parts[3].solutions, parts[3].nodes) == \
               (parts[0].solutions, parts[0].nodes, parts[1].solutions, parts[1].nodes)
        for depth in (4, 6, 4, 4):
            r = m.solve_tree("count", split_depth=depth)
            assert (r.solutions, r.nodes, r.first) == (g.solutions, g.nodes, g.first), depth
    t = m.solve_tree("count", time_kernels=True)
    assert (t.solutions, t.nodes) == (g.solutions, g.nodes) and t.search_kernel_ms > 0
    m.solve_tree("count")                                        # first time round for this queue again: call by call
    assert m.solve_tree("count").search_kernel_ms == 0          # replayed: the graph is timed from outside only


def test_17_queens_in_four_partitions(golden_large, product_lib):
    """BASELINE config C5 at full size, the way four GPUs split it (split depth 9): the partitions' counts add up to what
    the unmodified reference returns for 17-Queens (tests/golden/reference_large.json: 17 single-threaded runs of
    oracle/_ref/dequan_ref, one per first-row value), and the lowest first-solution key belongs to its first solution."""
    g = golden_large["nqueens"]["17"]["count"]
    assert g["solutions"] == 95815104                      # OEIS A000170(17), for the record
    csp = nqueens(17)
    m = api.Model(csp)
    parts = [m.solve_tree("count", part_rank=k, part_count=4) for k in range(4)]
    assert sum(p.solutions for p in parts) == g["solutions"] and sum(p.nodes for p in parts) == g["nodes"]
    best = min(parts, key=lambda p: p.first_key)
    assert best.first == g["first"] == O.solve(csp, "first").first
    whole = m.solve_tree("count")
    assert (whole.solutions, whole.nodes, whole.first) == (g["solutions"], g["nodes"], g["first"])


def test_single_process_multi_device_solve(golden, product_lib):
    """dq_solve_tree_multi: one call deals the prefix-split tree to several devices (worker thread + model clone each)
    and reduces the tail itself.  A device may be named more than once, so the partition / reduction logic is
    exercised on a one-GPU box too; with two or more GPUs the same list of checks runs across real devices."""
    import torch
    lists = [(0,), (0, 0), (0, 0, 0)]
    if torch.cuda.device_count() >= 2:
        lists += [(0, 1), tuple(range(torch.cuda.device_count()))]
    for n in (8, 12):
        g = golden["nqueens"][str(n)]
        m = api.Model(nqueens(n))
        for devs in lists:
            c = m.solve_tree_multi("count", devs)
            assert (c.solutions, c.nodes, c.first) == (g["count"]["solutions"], g["count"]["nodes"], g["count"]["first"]), (n, devs, c)
            f = m.solve_tree_multi("first", devs)
            assert (f.status, f.nodes, f.first) == (g["first"]["status"], g["first"]["nodes"], g["first"]["first"]), (n, devs, f)
    for seed in range(9100, 9130):
        csp = random_model(seed, n_vars=10, n_cons=15, max_dom=6)
        m = api.Model(csp)
        for mode in ("first", "count"):
            want = O.solve(csp, mode)
            for devs in lists[1:]:
                _cmp_tree(m.solve_tree_multi(mode, devs, split_depth=2), want, (seed, mode, devs))
    with pytest.raises(api.DequanError):
        api.Model(nqueens(6)).solve_tree_multi("count", (0, 99))


def test_duplicate_values_vs_reference(product_lib):
    """Values domains that list a value more than once (SURVEY.md par. 9 Q2): every copy is a position of the domain
    word, Exclude erases the first copy still present, Intersect leaves one — against the unmodified reference."""
    import json
    from randmodels import dup_suite
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_dups.json")))["duplicate_values"]
    suite = dup_suite(g["n"], g["seed0"])
    for mode in ("first", "count"):
        for i, (csp, want) in enumerate(zip(suite, g[mode])):
            m = api.Model(csp)
            assert m.order() == want["order"]
            for engine in ("auto", "warp"):
                r = m.solve_tree(mode, engine=engine)
                assert (r.status, r.solutions, r.nodes, r.first) == (want["status"], want["solutions"], want["nodes"], want["first"]), (mode, i, engine, r)


def _queens_plus(n, extra):
    """N-Queens with one more constraint: no longer the structure the class engine recognises."""
    csp = nqueens(n)
    csp.constraints = list(csp.constraints)
    csp.AddConstraint(extra)
    csp.FinalizeModel()
    return csp


@pytest.mark.parametrize("n", [9, 11, 12])
def test_generic_lane_tree_engine(product_lib, n):
    """dq_lane_tree.cuh (lane per prefix subtree, small models with plain AND filters): COUNT_ALL against the oracle and
    against the warp-cooperative engines on models just outside the N-Queens class."""
    for extra in (OpConstraint(0, n - 1, Op.Inf, 0), OpConstraint(1, 2, Op.NotEqual, 3), OpConstraint(0, 3, Op.SupEqual, -2)):
        csp = _queens_plus(n, extra)
        m = api.Model(csp)
        assert m.info()["model_class"] != "queens"
        want = O.solve(csp, "count")
        for engine, depth in (("auto", 0), ("lane", 0), ("lane", 4), ("reg", 0), ("warp", 0)):
            got = m.solve_tree("count", engine=engine, split_depth=depth)
            _cmp_tree(got, want, (n, engine, depth))
        if n >= 12:
            assert m.solve_tree("count", engine="lane").engine == "lane"
        parts = [m.solve_tree("count", engine="lane", part_rank=r, part_count=3) for r in range(3)]
        assert (sum(p.solutions for p in parts), sum(p.nodes for p in parts)) == (want.solutions, want.nodes)
        assert min(parts, key=lambda p: p.first_key).first == want.first


def test_generic_path_on_the_queens_class(golden, product_lib):
    """DQ_NO_CLASS=1 sends the N-Queens model itself down the generic path (lane tree engine): same counts as the
    reference.  The variable is read once per process, hence the subprocess."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); from dequan_b200 import api; from dequan_b200.model import nqueens\n"
            "for n in (10, 13):\n"
            "    r = api.Model(nqueens(n)).solve_tree('count'); print(n, r.solutions, r.nodes, r.first, r.engine)\n"
            % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, DQ_NO_CLASS="1"), capture_output=True, text=True,
                         check=True, timeout=300).stdout.splitlines()
    for line in out:
        n = int(line.split()[0])
        g = golden["nqueens"][str(n)]["count"]
        want_engine = "lane" if n >= 13 else line.split()[-1]      # (a tree of a few thousand prefixes stays on the warp-cooperative engines)
        assert line == f"{n} {g['solutions']} {g['nodes']} {g['first']} {want_engine}", line


@pytest.mark.parametrize("var", ["DQ_QUEENS_PLAIN_ROWS"])
def test_queens_bucket_kernel_variants(golden, product_lib, var):
    """The bucket kernels a 17-Queens solve does not pick: forward-check rows all in plain form (what boards of 23 and
    more queens get).  The variable is read once per process, hence the subprocess."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); from dequan_b200 import api; from dequan_b200.model import nqueens\n"
            "for n in (5, 9, 12, 14):\n"
            "    r = api.Model(nqueens(n)).solve_tree('count'); print(n, r.solutions, r.nodes, r.first, r.engine)\n"
            % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **{var: "1"}), capture_output=True, text=True,
                         check=True, timeout=300).stdout.splitlines()
    assert len(out) == 4
    for line in out:
        n = int(line.split()[0])
        g = golden["nqueens"][str(n)]["count"]
        assert line == f"{n} {g['solutions']} {g['nodes']} {g['first']} lane", line


def test_sudoku_10k_vs_reference(golden_large, product_lib):
    """The first 10 000 puzzles of the 1 M batch (config C3): node count and solution of every puzzle against the
    unmodified reference (810 binary NotEqual constraints, tests/golden/make_golden_large.py)."""
    g = golden_large["sudoku10k"]
    cells = G.sudoku_batch(g["n"], givens=g["givens"])
    assert hashlib.sha256(cells.tobytes()).hexdigest() == g["sha256"]
    tmpl = api.Model(sudoku_template())
    for engine in ("auto", "warp"):
        r = tmpl.solve_batch_cells(cells, engine=engine)
        assert (r.status == 1).all()
        assert r.nodes.tolist() == g["nodes"], engine
        got = "".join(map(str, r.solution.reshape(-1).tolist()))
        assert hashlib.sha256(got.encode()).hexdigest() == g["solutions_sha256"] and got == g["solutions"], engine
