"""The batch entry points on everything but the 9x9 Sudoku template, instance by instance against the CPU oracle.

`dq_solve_batch_cells` sends every template other than the 9x9 Sudoku class to the generic batch kernel
(`k_batch_cells<HAS_F, HAS_TABLE>`); `dq_solve_batch_graphs` with more than four colours runs only the generic warp
engine (`k_graphs_build` + `k_batch_graphs`).  Expected answers: one instance = the template with each given
v -> Domain(Values, [byte]) (AddFixedVar, dequan.h:467-471), solved by the oracle in FIRST mode with the same node
budget; status, node count and the first solution, value as byte."""
import functools
import random

import numpy as np
import pytest

import oracle_lib as O
from dequan_b200 import api
from dequan_b200 import generators as G
from dequan_b200.model import (CSP, AllDifferentConstraint, Domain, DomainType, EqualityConstraint, Op, OpConstraint,
                               OrRangeConstraint, TableConstraint, colouring, sudoku, sudoku_template)
from randmodels import random_domain, random_model, random_model_dups

SMS = 148                   # B200
STATUS = {"unsat": 0, "sat": 1, "budget": 2}


# ---- reference for one batch instance ----------------------------------------------------------------------------

def instance_csp(template: CSP, row) -> CSP:
    """Instance `row` of a cell batch: a copy of the template in which every variable v with row[v] != 0 is fixed to that
    value (AddFixedVar).  The caller's assign_order, if any, is kept."""
    nv = len(template.domains)
    doms = [Domain(DomainType.Values, [int(row[v])]) if row[v] else Domain(DomainType(d.type), list(d.values))
            for v, d in enumerate(template.domains[:nv])]
    order = list(template.assign_order) if template.assign_order is not None else None
    return CSP(doms, list(template.constraints), order)


def domain_values(d: Domain):
    if d.type == DomainType.Values:
        return list(d.values)
    return [x for a, b in zip(d.values[::2], d.values[1::2]) for x in range(a, b)]


def valid_row(template: CSP, row) -> bool:
    """Every given byte is a value of its variable's template domain (else the kernel answers status 3)."""
    return all(not row[v] or int(row[v]) in domain_values(d) for v, d in enumerate(template.domains))


@functools.lru_cache(maxsize=None)
def _expected(template_key, row_bytes: bytes, budget: int):
    template = _TEMPLATES[template_key]
    row = np.frombuffer(row_bytes, dtype=np.uint8)
    nv = len(template.domains)
    if not valid_row(template, row):
        return 3, 0, bytes(nv)
    o = O.solve(instance_csp(template, row), "first", budget)
    sol = bytes(x & 0xFF for x in o.first) if o.status == "sat" else bytes(nv)
    return STATUS[o.status], o.nodes, sol


_TEMPLATES = {}


def expected(key, template: CSP, rows: np.ndarray, budget: int):
    """(status, nodes, solution bytes) per row from the oracle; rows that repeat are solved once."""
    _TEMPLATES[key] = template
    nv = len(template.domains)
    out = [_expected(key, bytes(r[:nv]), budget) for r in rows]
    return (np.array([s for s, _, _ in out], dtype=np.uint8), np.array([n for _, n, _ in out], dtype=np.uint64),
            np.frombuffer(b"".join(s for _, _, s in out), dtype=np.uint8).reshape(len(rows), nv))


# ---- templates and rows --------------------------------------------------------------------------------------------

def latin_template(n: int) -> CSP:
    csp = CSP()
    for _ in range(n * n):
        csp.AddIntVar(1, n + 1)
    for r in range(n):
        for a in range(n):
            for b in range(a + 1, n):
                csp.AddConstraint(OpConstraint(r * n + a, r * n + b, Op.NotEqual, 0))
                csp.AddConstraint(OpConstraint(a * n + r, b * n + r, Op.NotEqual, 0))
    return csp


def colouring_template(nv: int, k: int, c: float, seed: int) -> CSP:
    """k-colouring on values 1..k (so that every colour is a possible given byte)."""
    edges = G.colouring_instance(nv, c, seed, 0) if nv > 1 else np.zeros((0, 2), dtype=np.uint8)
    csp = CSP()
    for _ in range(nv):
        csp.AddIntVar(1, k + 1)
    for u, v in edges:
        csp.AddConstraint(OpConstraint(int(u), int(v), Op.NotEqual, 0))
    return csp


def filter_model(seed: int, n_vars: int, n_cons: int) -> CSP:
    """Pair filters without an F word: NotEqual with a non-zero offset and the four order relations (K_AND)."""
    rng = random.Random(seed)
    csp = CSP()
    for _ in range(n_vars):
        csp.AddIntVar(random_domain(rng, 1, 9, 6))
    for _ in range(n_cons):
        a, b = rng.sample(range(n_vars), 2)
        op = rng.choice([Op.NotEqual, Op.SupEqual, Op.Sup, Op.InfEqual, Op.Inf])
        csp.AddConstraint(OpConstraint(a, b, op, rng.choice([-2, -1, 1, 2]) if op == Op.NotEqual else rng.randint(-2, 2)))
    return csp


def latin_solutions(n: int, count: int, rng: np.random.Generator) -> np.ndarray:
    """Latin squares on 1..n: the cyclic square with rows, columns and symbols permuted."""
    base = (np.arange(n)[:, None] + np.arange(n)[None, :]) % n
    out = np.zeros((count, n * n), dtype=np.uint8)
    for i in range(count):
        sq = base[rng.permutation(n)][:, rng.permutation(n)]
        out[i] = (rng.permutation(n)[sq] + 1).reshape(-1)
    return out


def make_rows(template: CSP, solutions: np.ndarray, n: int, seed: int, p_keep=(0.2, 0.9), p_rand=(0.05, 0.4)) -> np.ndarray:
    """n distinct-ish rows: 45 % a random subset of a solution's values, 40 % random givens from the template domains,
    10 % all-zero (the template itself), the rest with one byte that is not in its variable's domain."""
    rng = np.random.default_rng(seed)
    nv = len(template.domains)
    doms = [[x for x in domain_values(d) if 1 <= x <= 255] for d in template.domains]
    rows = np.zeros((n, nv), dtype=np.uint8)
    for i in range(n):
        u = rng.random()
        if u < 0.45 and len(solutions):
            s = solutions[rng.integers(len(solutions))]
            keep = rng.random(nv) < rng.uniform(*p_keep)
            rows[i] = np.where(keep & (s >= 1) & (s <= 255), s, 0).astype(np.uint8)
        elif u < 0.85:
            p = rng.uniform(*p_rand)
            for v in range(nv):
                if doms[v] and rng.random() < p:
                    rows[i, v] = doms[v][rng.integers(len(doms[v]))]
        elif u < 0.95:
            pass
        else:
            v = int(rng.integers(nv))
            bad = [x for x in range(1, 256) if x not in set(domain_values(template.domains[v]))]
            rows[i, v] = bad[rng.integers(len(bad))]
    return rows


def _satisfiable(make, seeds, want: int, min_solutions: int = 20):
    """The first `want` templates make(seed) with at least `min_solutions` solutions (so that rows drawn from
    solutions are mostly sat), with up to 300 of their solutions."""
    out = []
    for seed in seeds:
        t = make(seed)
        sols, total = O.enumerate_solutions(t, 300)
        if total >= min_solutions:
            out.append((t, np.array(sols, dtype=np.int64).reshape(len(sols), len(t.domains))))
            if len(out) == want:
                return out
    raise AssertionError("not enough satisfiable templates")


def _with_every_kind(seed: int) -> CSP:
    t = random_model(seed, 12, 9, 6)
    t.AddConstraint(EqualityConstraint(0, 1))
    t.AddConstraint(OrRangeConstraint(2, 3, 1, 4))
    t.AddConstraint(TableConstraint(4, 5, [(a, b) for a in range(-3, 12) for b in range(-3, 12) if (a + b) % 3]))
    t.AddConstraint(AllDifferentConstraint([6, 7, 8]))
    return t


def _random_cases(family: str):
    if family == "filters":                       # k_batch_cells<false, true>
        picks = (_satisfiable(lambda s: random_model(s, 8 + s % 3 * 4, 10 + s % 3 * 4, 6, "ne"), range(700, 800), 2)
                 + _satisfiable(lambda s: filter_model(s, 10 + s % 2 * 8, 9 + s % 2 * 8), range(800, 900), 2))
    elif family == "all":                         # k_batch_cells<true, true>: Equal -> K_WEQ, Table / OrRange -> K_CHK
        picks = (_satisfiable(lambda s: random_model(s, 6 + s % 4 * 4, 6 + s % 4 * 4, 6), range(900, 1100), 4)
                 + _satisfiable(_with_every_kind, range(1100, 1300), 1))
    else:                                         # duplicates: ENT_FIRST masks, the byte -> value-index map on repeats
        picks = _satisfiable(lambda s: random_model_dups(s, 5 + s % 4 * 2, 5 + s % 4 * 2, 5), range(1300, 1500), 6)
    return [(f"{family}{i}", t, sols) for i, (t, sols) in enumerate(picks)]


@functools.lru_cache(maxsize=None)
def family_cases(family: str):
    """[(key, template, distinct rows, model class, cap)]: cap is the "unbounded" node budget, 0 (none) where every row
    of the family finishes quickly; the Latin squares and large colourings have rows the oracle needs minutes for."""
    if family == "ne_same":
        out = []
        rng = np.random.default_rng(9)
        for n, count in ((9, 2500), (12, 1200)):
            t = latin_template(n) if n == 12 else sudoku_template(boxes=False)
            rows = make_rows(t, latin_solutions(n, 200, rng), count, seed=n, p_keep=(0.3, 0.9), p_rand=(0.05, 0.3))
            out.append((f"latin{n}", t, rows, "ne_same", 200_000))
        for i, nv in enumerate((1, 31, 32, 33, 200, 254)):
            t = colouring_template(nv, 4, 2.0, 300 + i)
            o = O.solve(t, "first")
            sols = np.array([o.first], dtype=np.int64) if o.first else np.zeros((0, nv), dtype=np.int64)
            rows = make_rows(t, sols, 600 if nv < 200 else 300, seed=40 + i, p_rand=(0.01, 0.1))
            out.append((f"col{nv}", t, rows, "ne_same", 200_000))
        return out
    out = []
    for key, t, sols in _random_cases(family):
        rows = make_rows(t, sols, 1500, seed=sum(map(ord, key)))
        out.append((key, t, rows, "generic", 0))
    return out


FAMILIES = ["ne_same", "filters", "all", "dups"]


def median_budget(key, t, rows, cap):
    """A node budget near the median of the template's node counts (at least 1)."""
    _, nodes, _ = expected(key, t, rows, cap)
    return max(1, int(np.median(nodes)))


# ---- CPU ------------------------------------------------------------------------------------------------------------

def test_instance_reference_and_family_outcomes():
    """instance_csp on the Sudoku template is exactly the construction of the Sudoku goldens (model.sudoku), and every
    template family gets sat, unsat and budget answers from the oracle (at its median budget) and some status-3 rows."""
    for row in G.sudoku_batch(20, givens=28, seed=3):
        got, want = instance_csp(sudoku_template(), row).arrays(), sudoku(row).arrays()
        assert all(np.array_equal(a, b) for a, b in zip(got, want))
    for fam in FAMILIES:
        seen = set()
        for key, t, rows, _, cap in family_cases(fam):
            st, _, _ = expected(key, t, rows, median_budget(key, t, rows, cap))
            seen |= set(st.tolist())
        assert seen == {0, 1, 2, 3}, (fam, seen)


# ---- GPU: generic templates (k_batch_cells) --------------------------------------------------------------------------

# Four times as many instances as a B200 has warps at the highest occupancy k_batch_cells reaches (16 CTAs of 4 warps
# per SM): every warp runs instance after instance in the same shared state.
BATCH = 4 * SMS * 16 * 4


def _tile(rows: np.ndarray, n: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    b = np.tile(rows, (-(-n // len(rows)), 1))
    return np.ascontiguousarray(b[rng.permutation(len(b))])


def _check_batch(got, want, what):
    st, nodes, sol = want
    nv = sol.shape[1]
    bad = np.nonzero((got.status != st) | (got.nodes != nodes) | (got.solution[:, :nv] != sol).any(axis=1))[0]
    assert len(bad) == 0, (what, f"{len(bad)} of {len(st)} instances differ", [(int(i), int(got.status[i]), int(st[i]), int(got.nodes[i]), int(nodes[i])) for i in bad[:5]])
    assert (got.n_sat, got.n_unsat, got.n_budget) == (int((st == 1).sum()), int((st == 0).sum() + (st == 3).sum()), int((st == 2).sum())), what
    assert got.n_sat + got.n_unsat + got.n_budget == len(st) and got.total_nodes == int(got.nodes.sum()) == int(nodes.sum()), what


def _same_outputs(a, b, nv, what):
    assert (a.status == b.status).all() and (a.nodes == b.nodes).all(), what
    assert (a.solution[:, :nv] == b.solution[:, :nv]).all(), what
    assert (a.n_sat, a.n_unsat, a.n_budget, a.total_nodes) == (b.n_sat, b.n_unsat, b.n_budget, b.total_nodes), what


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_generic_batch_vs_oracle(product_lib, family):
    """Every instance of each template's batch against the oracle, without a budget (or far above the median where some
    rows take the oracle minutes) and at the median; then the same batch permuted, padded to a wider stride, and the
    budget boundary of a few instances."""
    for key, t, rows, cls, cap in family_cases(family):
        nv = len(t.domains)
        m = api.Model(t)
        assert m.info()["model_class"] == cls, key
        batch = _tile(rows, BATCH, len(rows))
        budget = median_budget(key, t, rows, cap)
        full = m.solve_batch_cells(batch, node_budget=cap)
        _check_batch(full, expected(key, t, batch, cap), (key, cap))
        assert full.launches == 1
        r = m.solve_batch_cells(batch, node_budget=budget)
        _check_batch(r, expected(key, t, batch, budget), (key, budget))
        # a permutation of the rows permutes the answers
        perm = np.random.default_rng(nv).permutation(len(batch))
        p = m.solve_batch_cells(np.ascontiguousarray(batch[perm]), node_budget=budget)
        assert (p.status == r.status[perm]).all() and (p.nodes == r.nodes[perm]).all() and (p.solution == r.solution[perm]).all(), key
        assert (p.n_sat, p.n_unsat, p.n_budget, p.total_nodes) == (r.n_sat, r.n_unsat, r.n_budget, r.total_nodes), key
        # stride > n_vars: the padding columns hold non-zero bytes the kernel must not read
        wide = np.random.default_rng(nv + 1).integers(1, 256, size=(len(batch), nv + 13), dtype=np.uint8)
        wide[:, :nv] = batch
        _same_outputs(m.solve_batch_cells(wide, node_budget=budget), r, nv, (key, "stride"))
        # an instance that needs exactly N nodes is solved with budget N and runs out with N - 1
        st, nodes, sol = expected(key, t, rows, cap)
        sat = np.nonzero(st == 1)[0]
        for i in sat[np.argsort(nodes[sat])][[0, len(sat) // 2, -1]]:
            one, need = np.ascontiguousarray(rows[i:i + 1]), int(nodes[i])
            a = m.solve_batch_cells(one, node_budget=need)
            assert (a.status[0], int(a.nodes[0]), a.solution[0].tobytes()) == (1, need, sol[i].tobytes()), (key, i)
            if need > 1:
                b = m.solve_batch_cells(one, node_budget=need - 1)
                _check_batch(b, expected(key, t, one, need - 1), (key, i, need - 1))
                assert (b.status[0], int(b.nodes[0])) == (2, need), (key, i)


@pytest.mark.gpu
def test_generic_batch_device_entry(product_lib):
    """dq_solve_batch_cells_dev on a generic template (torch buffers) equals the host entry; the lane engine refuses it."""
    import torch
    key, t, rows, _, cap = family_cases("all")[-1]
    m = api.Model(t)
    batch = _tile(rows, 20000, 3)
    n, nv = batch.shape
    budget = median_budget(key, t, rows, cap)
    want = m.solve_batch_cells(batch, node_budget=budget)
    dev = torch.device("cuda", 0)
    d_cells = torch.from_numpy(batch).to(dev)
    d_sol = torch.zeros((n, nv), dtype=torch.uint8, device=dev)
    d_nodes = torch.zeros(n, dtype=torch.int64, device=dev)
    d_status = torch.zeros(n, dtype=torch.uint8, device=dev)
    st = m.solve_batch_cells_ptr(d_cells.data_ptr(), n, nv, d_sol.data_ptr(), d_nodes.data_ptr(), d_status.data_ptr(),
                                 node_budget=budget, device=True)
    torch.cuda.synchronize()
    assert (d_sol.cpu().numpy() == want.solution).all() and (d_status.cpu().numpy() == want.status).all()
    assert (d_nodes.cpu().numpy().astype(np.uint64) == want.nodes).all()
    assert (st.n_sat, st.n_unsat, st.n_budget, st.total_nodes) == (want.n_sat, want.n_unsat, want.n_budget, want.total_nodes)
    assert 0 < want.n_budget < n and want.n_sat > 0
    for tmpl in (t, sudoku_template(boxes=False)):
        with pytest.raises(api.DequanError):
            api.Model(tmpl).solve_batch_cells(batch[:8] if tmpl is t else np.zeros((8, 81), dtype=np.uint8), engine="lane")


# ---- caller-supplied assign_order ------------------------------------------------------------------------------------

def _with_order(t: CSP, order) -> CSP:
    return CSP([Domain(DomainType(d.type), list(d.values)) for d in t.domains], list(t.constraints), list(order))


@functools.lru_cache(maxsize=None)
def order_cases():
    """[(key, template with a caller order, rows, budget)]: rows whose oracle answer in the caller's order differs from
    the one in Reset's order of the instance (the givens first), so that a batch that drops the order fails on each."""
    rng = random.Random(17)
    sud = sudoku_template()
    shuffled = lambda t: rng.sample(range(len(t.domains)), len(t.domains))
    cases = [("sudoku_shuffled", _with_order(sud, shuffled(sud)), G.sudoku_batch(20, givens=28, seed=3), 20_000),
             ("sudoku_identity", _with_order(sud, range(81)), G.sudoku_batch(20, givens=28, seed=3), 20_000)]
    l12 = latin_template(12)
    cases.append(("latin12_shuffled", _with_order(l12, shuffled(l12)),
                  make_rows(l12, latin_solutions(12, 40, np.random.default_rng(5)), 60, seed=6, p_keep=(0.4, 0.8), p_rand=(0.02, 0.05)),
                  20_000))
    for i, (t, sols) in enumerate(_satisfiable(lambda s: random_model(s, 10 + s % 2 * 4, 6 + s % 2 * 3, 6), range(2000, 2400), 2)):
        cases.append((f"random{i}_shuffled", _with_order(t, shuffled(t)), make_rows(t, sols, 400, seed=60 + i), 0))
    out = []
    for key, t, rows, budget in cases:
        plain = CSP(t.domains, t.constraints)
        keep = [r for r in rows if valid_row(t, r)
                and _expected(_reg(key, t), bytes(r), budget) != _expected(_reg(key + "_reset", plain), bytes(r), budget)]
        out.append((key, t, np.ascontiguousarray(np.array(keep, dtype=np.uint8).reshape(len(keep), len(t.domains))), budget))
    return out


def _reg(key, t):
    _TEMPLATES[key] = t
    return key


def test_caller_order_cases_are_order_sensitive():
    """(CPU) The caller-order batches below are not vacuous: each keeps enough rows whose answer depends on the order."""
    for key, t, rows, _ in order_cases():
        assert len(rows) >= (20 if key.startswith("sudoku") else 15), (key, len(rows))


@pytest.mark.gpu
def test_caller_order_is_kept_in_batches(product_lib):
    """A template compiled with assign_order searches every instance in that order, even when it is the identity (Reset
    would put the givens first).  The 81-variable Sudoku with a caller order is not the Sudoku class."""
    for key, t, rows, budget in order_cases():
        m = api.Model(t)
        assert m.order() == list(t.assign_order)
        if key.startswith("sudoku"):
            assert m.info()["model_class"] == "ne_same"
        batch = _tile(rows, 4096, 1)
        _check_batch(m.solve_batch_cells(batch, node_budget=budget), expected(key, t, batch, budget), key)


# ---- colouring with k > 4 (k_graphs_build + k_batch_graphs) ----------------------------------------------------------

COLOUR_NV = [1, 2, 31, 32, 33, 64, 200, 254]
COLOUR_K = [5, 6, 8, 16, 31, 32]
COLOUR_BUDGET = 3000


def warp_state_bytes(nv: int, trail: int) -> int:       # dq_warp_engine.cuh
    nvp, tp = (nv + 3) & ~3, (trail + 3) & ~3
    return (nvp * 4 * 3 + tp * 4 + tp * 2 + nvp * 2 + nvp * 5 + 15) & ~15


def fits(nv: int, k: int) -> bool:
    """The per-warp state of the warp engine (trail nv * k + 32) for four warps fits the 200 KB it may use per CTA."""
    return warp_state_bytes(nv, nv * k + 32) * 4 <= 200 * 1024


def _clique(m: int):
    return [(u, v) for u in range(m) for v in range(u + 1, m)]


def colour_lists(nv: int, k: int, seed: int):
    """Random graphs with average degree from a third to 1.3 times k's colourability threshold (about 2 k ln k), the
    cliques K_k and K_(k+1), empty and complete graphs between them, and one list with duplicate and reversed edges."""
    rng = np.random.default_rng(seed)
    iu, ju = np.triu_indices(nv, 1)
    thr = 2 * k * np.log(k)
    lists = []
    for f in (0.3, 0.6, 0.8, 0.9, 1.0, 1.0, 1.1, 1.1, 1.2, 1.3):
        p = min(1.0, f * thr / max(nv - 1, 1))
        sel = rng.random(iu.size) < p
        lists.append(np.stack([iu[sel], ju[sel]], axis=1))
    lists.insert(3, np.zeros((0, 2)))
    lists.insert(6, np.stack([iu, ju], axis=1))
    for m in (k, k + 1):
        if m <= nv:
            lists.append(np.array(_clique(m)).reshape(-1, 2))
    e = lists[5]
    lists.append(np.concatenate([e, e[: len(e) // 2][:, ::-1], e[: len(e) // 3]])[rng.permutation(len(e) + len(e) // 2 + len(e) // 3)])
    lists.append(np.zeros((0, 2)))
    lists = [np.asarray(x, dtype=np.uint8).reshape(-1, 2) for x in lists]
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in lists])
    return off, np.ascontiguousarray(np.concatenate(lists))


@functools.lru_cache(maxsize=None)
def colour_expected(nv: int, k: int, budget: int, i: int):
    off, edges = colour_lists(nv, k, nv * 100 + k)
    o = O.solve(colouring(nv, k, edges[off[i]:off[i + 1]]), "first", budget)
    return STATUS[o.status], o.nodes, o.first


@pytest.mark.gpu
@pytest.mark.parametrize("k", COLOUR_K)
def test_colouring_more_than_four_colours_vs_oracle(product_lib, k):
    seen = set()
    for nv in COLOUR_NV:
        off, edges = colour_lists(nv, k, nv * 100 + k)
        n = len(off) - 1
        if not fits(nv, k):
            assert k > 16
            with pytest.raises(api.DequanError):
                api.solve_batch_graphs(nv, k, off, edges, node_budget=COLOUR_BUDGET, engine="warp")
            continue
        r = api.solve_batch_graphs(nv, k, off, edges, node_budget=COLOUR_BUDGET, engine="warp")
        assert r.launches == 2
        _same_outputs(api.solve_batch_graphs(nv, k, off, edges, node_budget=COLOUR_BUDGET), r, nv, (nv, k, "auto"))
        for i in range(n):
            st, nodes, first = colour_expected(nv, k, COLOUR_BUDGET, i)
            assert (int(r.status[i]), int(r.nodes[i])) == (st, nodes), (nv, k, i)
            if st == 1:
                assert r.solution[i].tolist() == first, (nv, k, i)
                e = edges[off[i]:off[i + 1]]
                assert (r.solution[i][e[:, 0]] != r.solution[i][e[:, 1]]).all()
            else:
                assert (r.solution[i] == 0xFF).all(), (nv, k, i)
            seen.add(st)
        assert (r.n_sat, r.n_unsat, r.n_budget) == tuple(int((r.status == s).sum()) for s in (1, 0, 2))
        assert r.total_nodes == int(r.nodes.sum())
        if nv >= k + 1:                                  # K_k is sat in nv nodes; K_(k+1) is unsat if the budget lets FC prove it
            ck, ck1 = n - 4, n - 3
            assert (r.status[ck], r.nodes[ck]) == (1, nv)
            assert r.status[ck1] == (0 if k <= 6 else 2)
        # budget boundary on the instance with the most nodes among the solved ones
        sat = np.nonzero(r.status == 1)[0]
        i = int(sat[np.argmax(r.nodes[sat])])
        need = int(r.nodes[i])
        one = (np.array([0, off[i + 1] - off[i]], dtype=np.int64), np.ascontiguousarray(edges[off[i]:off[i + 1]]))
        a = api.solve_batch_graphs(nv, k, *one, node_budget=need, engine="warp")
        assert (a.status[0], int(a.nodes[0]), a.solution[0].tolist()) == (1, need, r.solution[i].tolist())
        if need > 1:
            b = api.solve_batch_graphs(nv, k, *one, node_budget=need - 1, engine="warp")
            assert (b.status[0], int(b.nodes[0])) == (2, need) and (b.solution[0] == 0xFF).all()
        for engine in ("lane", "reg"):
            with pytest.raises(api.DequanError):
                api.solve_batch_graphs(nv, k, off, edges, engine=engine)
    assert seen == ({0, 1, 2} if k <= 6 else {1, 2}), seen        # (FC proves no larger-k instance unsat in the budget)


@pytest.mark.gpu
def test_colouring_more_than_four_colours_device_entry_refused(product_lib):
    import torch
    off, edges = colour_lists(31, 5, 7)
    dev = torch.device("cuda", 0)
    d_edges = torch.zeros(((edges.size + 15) // 16) * 16, dtype=torch.uint8, device=dev)
    d_edges[:edges.size] = torch.from_numpy(edges.reshape(-1)).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    n = len(off) - 1
    d_col = torch.zeros((n, 31), dtype=torch.uint8, device=dev)
    d_nodes = torch.zeros(n, dtype=torch.int64, device=dev)
    d_status = torch.zeros(n, dtype=torch.uint8, device=dev)
    with pytest.raises(api.DequanError):
        api.solve_batch_graphs_ptr(31, 5, off, d_off.data_ptr(), d_edges.data_ptr(), d_col.data_ptr(), d_nodes.data_ptr(),
                                   d_status.data_ptr(), device=True)


def test_colouring_state_limit():
    """(CPU) Which shapes the warp engine must refuse: at most k = 30 fits 254 vertices, every k <= 16 fits every size."""
    assert all(fits(nv, k) for nv in COLOUR_NV for k in COLOUR_K if k <= 16)
    assert [k for k in COLOUR_K if not fits(254, k)] == [31, 32]
    assert all(fits(nv, k) for nv in COLOUR_NV[:-1] for k in COLOUR_K)


# ---- k <= 4 warp engine against the reference -----------------------------------------------------------------------

@pytest.mark.gpu
def test_colouring_warp_engine_vs_reference(golden, golden_large, product_lib):
    for case in golden["colouring"] + golden_large["colouring200"]:
        off, edges = G.colouring_batch(case["count"], case["n_vertices"], case["c"])
        r = api.solve_batch_graphs(case["n_vertices"], case["k"], off, edges, node_budget=case["budget"], engine="warp")
        assert r.launches == 2
        assert [api.OUTCOME[s] for s in r.status] == case["status"], (case["k"], case["c"])
        assert r.nodes.tolist() == case["nodes"], (case["k"], case["c"])
        for i, first in enumerate(case["first"]):
            assert r.solution[i].tolist() == (first if first is not None else [0xFF] * case["n_vertices"]), i
        assert (r.n_sat, r.n_unsat, r.n_budget) == tuple(case["status"].count(x) for x in ("sat", "unsat", "budget"))
        assert r.total_nodes == sum(case["nodes"])
