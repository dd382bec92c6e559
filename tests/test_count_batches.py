"""Counting batches: `dq_count_batch_cells` / `dq_count_batch_graphs` instance by instance against the CPU oracle.

Expected answers come from `dqo_count_limit` (tests/oracle_count_limit.c, the CPU oracle's search with a solution
limit): the instance the FIRST-mode batch builds (givens fixed with AddFixedVar, the template's caller order kept),
searched with the counting constraint linked last that passes the L-th solution, under the Budget constraint
evaluated before it.  Every output array is compared element by element:
solutions, the DFS-first solution bytes, nodes and status, and the batch totals."""
import atexit
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import oracle_lib as O
from dequan_b200 import api
from dequan_b200 import generators as G
from dequan_b200.model import CSP, colouring, sudoku, sudoku_template
from randmodels import dup_suite, filter_suite, model_suite, random_filter_model
from test_batch_generic import (_satisfiable, _tile, colour_lists, family_cases, instance_csp, make_rows, order_cases,
                                valid_row)

STATUS = {"unsat": 0, "sat": 1, "budget": 2}
LIMITS = (0, 1, 2, 7)
DQ_ERR_INVALID, DQ_ERR_UNSUPPORTED = -1, -2


# ---- the oracle's search with a solution limit (tests/oracle_count_limit.c, built here into a temporary directory) --

_LIMIT_LIB = None


def _olib():
    global _LIMIT_LIB
    if _LIMIT_LIB is None:
        here = os.path.dirname(os.path.abspath(__file__))
        tmp = tempfile.mkdtemp(prefix="dq_count_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libdq_count_limit.so")
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-Wall",
                               "-I" + os.path.join(os.path.dirname(here), "include"), "-o", out,
                               os.path.join(here, "oracle_count_limit.c")])
        L = C.CDLL(out)
        L.dqo_count_limit.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(O.dqo_result), C.POINTER(C.c_int32)]
        L.dqo_count_limit.restype = C.c_int
        _LIMIT_LIB = L
    return _LIMIT_LIB


def oracle_count(csp: CSP, limit: int, budget: int = 0):
    """(status, solutions, nodes, first solution or None) of dqo_count_limit."""
    desc, keep = csp.desc()
    nv = len(csp.domains)
    first = np.zeros(max(nv, 1), dtype=np.int32)
    r = O.dqo_result()
    rc = _olib().dqo_count_limit(C.byref(desc), budget, limit, C.byref(r), first.ctypes.data_as(C.POINTER(C.c_int32)))
    assert rc == 0
    del keep
    return O.STATUS[r.outcome], r.solutions, r.nodes, first[:nv].tolist() if r.solutions else None


_TEMPLATES = {}


@functools.lru_cache(maxsize=None)
def _cell_expected(key, row_bytes: bytes, limit: int, budget: int):
    t = _TEMPLATES[key]
    nv = len(t.domains)
    row = np.frombuffer(row_bytes, dtype=np.uint8)
    if not valid_row(t, row):
        return 3, 0, 0, bytes(nv)
    st, sols, nodes, first = oracle_count(instance_csp(t, row), limit, budget)
    return STATUS[st], sols, nodes, bytes(x & 0xFF for x in first) if first else bytes(nv)


def cell_expected(key, t: CSP, rows: np.ndarray, limit: int, budget: int):
    """(status, solutions, nodes, first bytes) per row; repeated rows are searched once."""
    _TEMPLATES[key] = t
    nv = len(t.domains)
    out = [_cell_expected(key, bytes(r[:nv]), limit, budget) for r in rows]
    return (np.array([o[0] for o in out], dtype=np.uint8), np.array([o[1] for o in out], dtype=np.uint64),
            np.array([o[2] for o in out], dtype=np.uint64),
            np.frombuffer(b"".join(o[3] for o in out), dtype=np.uint8).reshape(len(rows), nv))


def check(got, want, what):
    st, sols, nodes, first = want
    nv = first.shape[1]
    bad = np.nonzero((got.status != st) | (got.solutions != sols) | (got.nodes != nodes)
                     | (got.first[:, :nv] != first).any(axis=1))[0]
    assert len(bad) == 0, (what, f"{len(bad)} of {len(st)} differ",
                           [(int(i), int(got.status[i]), int(st[i]), int(got.solutions[i]), int(sols[i]), int(got.nodes[i]),
                             int(nodes[i])) for i in bad[:5]])
    assert (got.n_sat, got.n_unsat, got.n_budget) == (int((st == 1).sum()), int((st == 0).sum() + (st == 3).sum()),
                                                     int((st == 2).sum())), what
    assert got.total_nodes == int(nodes.sum()), what


# ---- CPU: the oracle's limit entry point against its FIRST and COUNT_ALL modes ---------------------------------------

def _oracle_models():
    return model_suite(60, 1000) + dup_suite(40, 5000) + filter_suite(40, 20000)


def test_oracle_limit_identities():
    """L = 1 is FIRST mode (status, nodes, first), L = 0 is COUNT_ALL, n_solutions = min(total, L), node counts do not
    decrease as L grows, and the budget ends a search at exactly B + 1 nodes."""
    seen_budget = seen_limit = 0
    for csp in _oracle_models():
        f, c = O.solve(csp, "first"), O.solve(csp, "count")
        assert oracle_count(csp, 1) == (f.status, f.solutions, f.nodes, f.first)
        assert oracle_count(csp, 0) == (c.status, c.solutions, c.nodes, c.first)
        prev = 0
        for L in (1, 2, 3, 7, 50):
            st, sols, nodes, first = oracle_count(csp, L)
            assert sols == min(c.solutions, L) and first == c.first and nodes >= prev
            assert st == ("sat" if sols else "unsat")
            seen_limit += 0 < L < c.solutions
            prev = nodes
        assert prev <= c.nodes
        for B in sorted({1, 2, max(1, c.nodes // 3), max(1, c.nodes - 1), c.nodes}):
            for L in (0, 1, 2):
                st, sols, nodes, first = oracle_count(csp, L, B)
                whole = oracle_count(csp, L)
                if whole[2] <= B:                     # the unbudgeted search fits: the same answer
                    assert (st, sols, nodes, first) == whole
                else:
                    seen_budget += 1
                    assert st == "budget" and nodes == B + 1 and sols <= whole[1]
                    assert first == (whole[3] if sols else None)
                fb = O.solve(csp, "first", B)
                if L == 1:
                    assert (st, nodes, first) == (fb.status, fb.nodes, fb.first)
    assert seen_budget > 50 and seen_limit > 50


# ---- CPU: refusals before any device call -----------------------------------------------------------------------------

def _cells_rc(m, cells, stride=None, opts=None, nsol=True, n=None):
    cells = np.ascontiguousarray(cells, dtype=np.uint8)
    n = len(cells) if n is None else n
    stride = cells.shape[1] if stride is None else stride
    bufs = [np.zeros(max(len(cells), 1), dtype=np.uint64), np.zeros(max(cells.size, 1), dtype=np.uint8),
            np.zeros(max(len(cells), 1), dtype=np.uint64), np.zeros(max(len(cells), 1), dtype=np.uint8)]
    ptrs = [b.ctypes.data for b in bufs]
    if not nsol:
        ptrs[0] = None
    st = api.dq_batch_stats()
    st.n_sat = 99
    rc = api.lib().dq_count_batch_cells(m._h if m is not None else None, cells.ctypes.data, n, stride,
                                        C.byref(opts) if opts is not None else None, *ptrs, C.byref(st))
    return rc, st


def _graphs_rc(nv, k, off, edges, opts=None, nsol=True, edges_ptr=True):
    n = len(off) - 1
    bufs = [np.zeros(max(n, 1), dtype=np.uint64), np.zeros(max(n * max(nv, 1), 1), dtype=np.uint8),
            np.zeros(max(n, 1), dtype=np.uint64), np.zeros(max(n, 1), dtype=np.uint8)]
    ptrs = [b.ctypes.data for b in bufs]
    if not nsol:
        ptrs[0] = None
    edges = np.ascontiguousarray(edges, dtype=np.uint8)
    return api.lib().dq_count_batch_graphs(nv, k, off.ctypes.data, edges.ctypes.data if edges_ptr else None, n,
                                           C.byref(opts) if opts is not None else None, *ptrs, None)


def test_count_refusals_without_device(product_lib):
    t = sudoku_template()
    m = api.Model(t)
    cells = G.sudoku_batch(4, givens=30, seed=1)
    for eng in (api.ENGINE["lane"], api.ENGINE["reg"]):
        rc, _ = _cells_rc(m, cells, opts=api.dq_count_opts(0, 2, eng))
        assert rc == DQ_ERR_UNSUPPORTED and "warp engine" in api.lib().dq_last_error().decode()
    for eng in (-1, 4, 99):
        assert _cells_rc(m, cells, opts=api.dq_count_opts(0, 2, eng))[0] == DQ_ERR_INVALID
    assert _cells_rc(None, cells)[0] == DQ_ERR_INVALID
    assert _cells_rc(m, cells, n=-1)[0] == DQ_ERR_INVALID
    assert _cells_rc(m, cells, stride=80)[0] == DQ_ERR_INVALID
    assert _cells_rc(m, cells, nsol=False)[0] == DQ_ERR_INVALID
    wide = CSP()
    for _ in range(3):
        wide.AddIntVar(0, 40)
    assert _cells_rc(api.Model(wide), np.zeros((2, 3), dtype=np.uint8))[0] == DQ_ERR_UNSUPPORTED
    with pytest.raises(api.DequanError):
        m.count_batch_cells(cells, engine="lane")
    # an empty batch needs no device: zero stats
    rc, st = _cells_rc(m, np.zeros((0, 81), dtype=np.uint8), opts=api.dq_count_opts(0, 0, 0))
    assert rc == 0 and st.n_sat == 0
    r = m.count_batch_cells(np.zeros((0, 81), dtype=np.uint8), solution_limit=2)
    assert r.solutions.shape == (0,) and r.first.shape == (0, 81) and (r.n_sat, r.n_unsat, r.n_budget, r.total_nodes) == (0, 0, 0, 0)

    off = np.array([0, 2, 3], dtype=np.int64)
    edges = np.array([[0, 1], [1, 2], [2, 3]], dtype=np.uint8)
    for eng in (api.ENGINE["lane"], api.ENGINE["reg"]):
        assert _graphs_rc(5, 3, off, edges, opts=api.dq_count_opts(0, 0, eng)) == DQ_ERR_UNSUPPORTED
        assert "warp engine" in api.lib().dq_last_error().decode()
    assert _graphs_rc(5, 3, off, edges, opts=api.dq_count_opts(0, 0, 5)) == DQ_ERR_INVALID
    for nv, k in ((0, 3), (255, 3), (5, 0), (5, 33)):
        assert _graphs_rc(nv, k, off, edges) == DQ_ERR_INVALID, (nv, k)
    assert _graphs_rc(5, 3, off, edges, nsol=False) == DQ_ERR_INVALID
    assert _graphs_rc(5, 3, np.array([1, 2, 3], dtype=np.int64), edges) == DQ_ERR_INVALID
    assert _graphs_rc(5, 3, np.array([0, 2, 1], dtype=np.int64), edges) == DQ_ERR_INVALID
    assert _graphs_rc(5, 3, off, edges, edges_ptr=False) == DQ_ERR_INVALID
    assert _graphs_rc(3, 3, off, edges) == DQ_ERR_INVALID                       # endpoint 3 of 3 vertices
    assert _graphs_rc(5, 3, off, np.array([[0, 1], [1, 2], [4, 4]], dtype=np.uint8)) == DQ_ERR_UNSUPPORTED
    assert _graphs_rc(5, 3, np.zeros(1, dtype=np.int64), edges) == 0           # empty batch
    with pytest.raises(api.DequanError):
        api.count_batch_graphs(5, 3, off, edges, engine="reg")


def test_count_families_are_not_vacuous():
    """(CPU) The GPU families below see, at their limits and budgets, every status and instances with more than 7
    solutions, so that each limit cuts some search short."""
    for fam in CELL_FAMILIES:
        seen, many = set(), 0
        for key, t, rows, cap in cell_cases(fam):
            for L in LIMITS:
                st, sols, _, _ = cell_expected(key, t, rows, L, cap)
                seen |= set(st.tolist())
                if L == 0:
                    many += int((sols > 7).sum())
            seen |= set(cell_expected(key, t, rows, 0, mid_budget(key, t, rows, cap))[0].tolist())
        assert {1, 2, 3} <= seen, (fam, seen)
        assert many > 0, fam


# ---- the GPU families -------------------------------------------------------------------------------------------------

CELL_FAMILIES = ["sudoku9", "sudoku_generic", "latin_colour", "filters", "all", "dups", "user_filters"]


def _sudoku_rows(n: int, seed: int) -> np.ndarray:
    """22 to 30 givens (many puzzles have several solutions), a few rows with a clash or a foreign byte."""
    rows = np.concatenate([G.sudoku_batch(n // 9 + 1, givens=g, seed=seed + g) for g in range(22, 31)])[:n]
    rows = np.ascontiguousarray(rows)
    rows[::37, 0] = 0xEE                                    # not a value of the template domain: status 3
    return rows


@functools.lru_cache(maxsize=None)
def cell_cases(family: str):
    """[(key, template, distinct rows, node budget that bounds the oracle's work)]."""
    if family == "sudoku9":
        return [("sudoku9", sudoku_template(), _sudoku_rows(270, 11), 40_000)]
    if family == "sudoku_generic":
        return [("sudoku_alldiff", sudoku([0] * 81, alldiff=True), _sudoku_rows(180, 12), 40_000)]
    if family == "latin_colour":
        out = []
        for key, t, rows, _, _ in family_cases("ne_same"):
            if key in ("latin9", "col31", "col200"):
                out.append((key, t, np.ascontiguousarray(rows[:250]), 3000))
        return out
    if family == "user_filters":
        picks = _satisfiable(lambda s: random_filter_model(s, 6 + s % 3 * 2, 5 + s % 3 * 2, 6), range(30000, 30600), 3)
        return [(f"uf{i}", t, make_rows(t, sols, 300, seed=70 + i), 3000) for i, (t, sols) in enumerate(picks)]
    return [(key, t, np.ascontiguousarray(rows[:300]), 3000) for key, t, rows, _, _ in family_cases(family)]


def mid_budget(key, t, rows, cap):
    """The median node count of the rows' searches to the end, at most a quarter of cap."""
    nodes = cell_expected(key, t, rows, 0, cap)[2]
    return min(max(1, int(np.median(nodes[nodes > 0]))) if (nodes > 0).any() else 1, cap // 4)


def _budget_boundaries(m, key, t, rows, cap, what):
    """Budgets that land exactly on the L-th solution and one node before it (inside the last level): a few rows with
    at least L solutions, each alone."""
    for L in (1, 2, 7):
        st, sols, nodes, first = cell_expected(key, t, rows, L, cap)
        hit = np.nonzero((st == 1) & (sols == L))[0]
        for i in hit[:: max(1, len(hit) // 4)][:4]:
            one, need = np.ascontiguousarray(rows[i:i + 1]), int(nodes[i])
            a = m.count_batch_cells(one, solution_limit=L, node_budget=need)
            assert (a.status[0], int(a.solutions[0]), int(a.nodes[0])) == (1, L, need), (what, L, int(i))
            assert a.first[0].tobytes() == first[i].tobytes(), (what, L, int(i))
            if need > 1:
                b = m.count_batch_cells(one, solution_limit=L, node_budget=need - 1)
                check(b, cell_expected(key, t, one, L, need - 1), (what, L, int(i), need - 1))
                assert (b.status[0], int(b.solutions[0]), int(b.nodes[0])) == (2, L - 1, need), (what, L, int(i))


@pytest.mark.gpu
@pytest.mark.parametrize("family", CELL_FAMILIES)
def test_count_cells_vs_oracle(product_lib, family):
    for key, t, rows, cap in cell_cases(family):
        m = api.Model(t)
        batch = _tile(rows, 4 * len(rows), len(rows))
        for L in LIMITS:
            r = m.count_batch_cells(batch, solution_limit=L, node_budget=cap)
            check(r, cell_expected(key, t, batch, L, cap), (key, L, cap))
            assert r.launches == 1
        # a budget near the median node count: many searches end inside a last level
        mid = mid_budget(key, t, rows, cap)
        for L in (0, 2, 7):
            check(m.count_batch_cells(batch, solution_limit=L, node_budget=mid), cell_expected(key, t, batch, L, mid),
                  (key, L, mid))
        _budget_boundaries(m, key, t, rows, cap, key)


@pytest.mark.gpu
def test_count_cells_layouts(product_lib):
    """A caller assign_order, a stride wider than the template (padding bytes the kernel must not read), batches
    smaller than a warp and an empty batch."""
    for key, t, rows, budget in order_cases():
        m = api.Model(t)
        cap = budget or 3000
        for L in (0, 2):
            check(m.count_batch_cells(rows, solution_limit=L, node_budget=cap), cell_expected(key, t, rows, L, cap), (key, L))
    key, t, rows, cap = cell_cases("all")[0]
    m = api.Model(t)
    nv = len(t.domains)
    r = m.count_batch_cells(rows, solution_limit=7, node_budget=cap)
    wide = np.random.default_rng(5).integers(1, 256, size=(len(rows), nv + 13), dtype=np.uint8)
    wide[:, :nv] = rows
    w = m.count_batch_cells(wide, solution_limit=7, node_budget=cap)
    assert (w.solutions == r.solutions).all() and (w.nodes == r.nodes).all() and (w.status == r.status).all()
    assert (w.first[:, :nv] == r.first).all()
    for n in (1, 5, 31):
        check(m.count_batch_cells(np.ascontiguousarray(rows[:n]), solution_limit=2, node_budget=cap),
              cell_expected(key, t, rows[:n], 2, cap), (key, n))
    e = m.count_batch_cells(np.zeros((0, nv), dtype=np.uint8), solution_limit=2)
    assert e.solutions.size == 0 and (e.n_sat, e.n_unsat, e.n_budget, e.total_nodes) == (0, 0, 0, 0)


# ---- graphs ----------------------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def graph_lists(nv: int, k: int, seed: int):
    """test_batch_generic's lists (cliques, empty and complete graphs, repeated and reversed edges) and random graphs of
    average degree 0.8 k to 2.2 k, where counts range from none to past the node cap."""
    off, edges = colour_lists(nv, k, seed)
    rng = np.random.default_rng(seed)
    iu, ju = np.triu_indices(nv, 1)
    lists = [edges[off[i]:off[i + 1]] for i in range(len(off) - 1)]
    for f in (0.8, 1.0, 1.2, 1.4, 1.6, 1.8, 2.0, 2.2):
        sel = rng.random(iu.size) < min(1.0, f * k / max(nv - 1, 1))
        lists.append(np.stack([iu[sel], ju[sel]], axis=1).astype(np.uint8))
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in lists])
    return off, np.ascontiguousarray(np.concatenate(lists).reshape(-1, 2))


@functools.lru_cache(maxsize=None)
def _graph_expected(nv, k, seed, i, limit, budget):
    off, edges = graph_lists(nv, k, seed)
    st, sols, nodes, first = oracle_count(colouring(nv, k, edges[off[i]:off[i + 1]]), limit, budget)
    return STATUS[st], sols, nodes, bytes(first) if first else b"\xff" * nv


def graph_expected(nv, k, seed, limit, budget):
    off, _ = graph_lists(nv, k, seed)
    out = [_graph_expected(nv, k, seed, i, limit, budget) for i in range(len(off) - 1)]
    return (np.array([o[0] for o in out], dtype=np.uint8), np.array([o[1] for o in out], dtype=np.uint64),
            np.array([o[2] for o in out], dtype=np.uint64),
            np.frombuffer(b"".join(o[3] for o in out), dtype=np.uint8).reshape(len(out), nv))


GRAPH_CASES = [(nv, k) for k in (3, 5, 9) for nv in (1, 2, 10, 16, 24, 33, 40)]
GRAPH_CAP = 4000


@pytest.mark.gpu
@pytest.mark.parametrize("k", [3, 5, 9])
def test_count_graphs_vs_oracle(product_lib, k):
    for nv, kk in GRAPH_CASES:
        if kk != k:
            continue
        seed = nv * 100 + k
        off, edges = graph_lists(nv, k, seed)
        for L in LIMITS:
            for budget in (GRAPH_CAP, 150):
                r = api.count_batch_graphs(nv, k, off, edges, solution_limit=L, node_budget=budget)
                assert r.launches == 2
                check(r, graph_expected(nv, k, seed, L, budget), (nv, k, L, budget))
        # budgets on the L-th solution and one node before it
        for L in (1, 2, 7):
            st, sols, nodes, first = graph_expected(nv, k, seed, L, GRAPH_CAP)
            for i in np.nonzero((st == 1) & (sols == L))[0][:3]:
                one = (np.array([0, off[i + 1] - off[i]], dtype=np.int64), np.ascontiguousarray(edges[off[i]:off[i + 1]]))
                need = int(nodes[i])
                a = api.count_batch_graphs(nv, k, *one, solution_limit=L, node_budget=need)
                assert (a.status[0], int(a.solutions[0]), int(a.nodes[0]), a.first[0].tobytes()) == (1, L, need, first[i].tobytes())
                if need > 1:
                    b = api.count_batch_graphs(nv, k, *one, solution_limit=L, node_budget=need - 1)
                    assert (b.status[0], int(b.solutions[0]), int(b.nodes[0])) == (2, L - 1, need)
                    assert b.first[0].tobytes() == (first[i].tobytes() if L > 1 else b"\xff" * nv)


# ---- L = 1 is the FIRST-mode batch, on whichever engine it picks -------------------------------------------------------

def _same_as_first(c, f, nv, what):
    assert (c.status == f.status).all() and (c.nodes == f.nodes).all(), what
    assert (c.first[:, :nv] == f.solution[:, :nv]).all(), what
    assert (c.solutions == (f.status == 1)).all(), what
    assert (c.n_sat, c.n_unsat, c.n_budget, c.total_nodes) == (f.n_sat, f.n_unsat, f.n_budget, f.total_nodes), what


@pytest.mark.gpu
def test_limit_one_is_the_first_mode_batch(product_lib):
    m = api.Model(sudoku_template())
    cells = G.sudoku_batch(100_000, givens=30, seed=20261018)
    cells[::997, 5] = 0xEE                                   # status 3 rows
    for budget in (0, 300):
        f = m.solve_batch_cells(cells, node_budget=budget)
        c = m.count_batch_cells(cells, solution_limit=1, node_budget=budget)
        _same_as_first(c, f, 81, ("sudoku", budget))
    for count, engine_picked in ((4096, "lane"), (1000, "reg")):
        off, edges = G.colouring_batch(count, 200, 4.2)
        f = api.solve_batch_graphs(200, 3, off, edges, node_budget=100_000)
        assert f.launches == (3 if engine_picked == "lane" else 1)
        c = api.count_batch_graphs(200, 3, off, edges, solution_limit=1, node_budget=100_000)
        _same_as_first(c, f, 200, ("colouring", count))


# ---- L = 0 against a second device path: dq_solve_models on each instance ---------------------------------------------

@pytest.mark.gpu
def test_count_all_matches_solve_models(product_lib):
    for fam in ("sudoku9", "all", "user_filters", "latin_colour"):
        key, t, rows, cap = cell_cases(fam)[0]
        st, sols, nodes, first = cell_expected(key, t, rows, 0, cap)
        pick = [i for i in range(len(rows)) if st[i] in (0, 1)][:48]
        r = api.Model(t).count_batch_cells(np.ascontiguousarray(rows[pick]), node_budget=0)
        ms = [api.Model(instance_csp(t, rows[i])) for i in pick]
        want = api.solve_models(ms, mode="count")
        assert [int(x) for x in r.solutions] == want.solutions, fam
        assert [int(x) for x in r.nodes] == want.nodes, fam
        assert [api.OUTCOME[int(x)] for x in r.status] == want.status, fam
        for j, f in enumerate(want.first):
            assert (r.first[j].tolist()[:len(t.domains)] == [x & 0xFF for x in f]) if f else (r.first[j] == 0).all(), (fam, j)
