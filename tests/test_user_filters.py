"""Filtering user constraints (DQ_CON_FILTER): a user-defined binary constraint that overrides AplyArcConsistency, lowered
to two tables, the pairs its Evaluate accepts (a K_CHK mask) and, per direction, the pairs its filter keeps (a K_AND
mask).  A value the filter removes is never visited; a value the filter keeps but Evaluate rejects is visited, counted
as a node, and fails.  So node counts are only right if the two tables stay apart.

CPU: the oracle against the four reference scenarios with a filtering user constraint, restatement identities, the
compiler's refusals and the drop-in header's refusals.  GPU: every engine and entry point against the oracle on random
FILTER models whose keep sets are equal to, stronger than, weaker than or unrelated to their allow sets."""
import json
import os
import random
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from dequan_b200 import api
from dequan_b200.model import (CSP, UNASSIGNED, AllDifferentConstraint, ConKind, Domain, DomainType, FilterConstraint, Op,
                               OpConstraint, TableConstraint, colouring, nqueens, sudoku_template)
from randmodels import domain_values, filter_suite, model_suite, random_domain, random_filter, random_filter_model
from test_batch_generic import instance_csp, make_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
LIBDIR = os.path.join(ROOT, "dequan_b200", "lib")


def tabulate(x, y, xs, ys, evaluate, keep01, keep10) -> FilterConstraint:
    """A user constraint on (x, y) as include/dequan.h's TabulateUserConstraint lowers it: the pairs Evaluate accepts, and
    per direction the pairs its AplyArcConsistency keeps, over the value lists xs and ys."""
    return FilterConstraint(x, y, [(a, b) for a in xs for b in ys if evaluate(a, b)],
                            [(a, b) for a in xs for b in ys if keep01(a, b)],
                            [(a, b) for b in ys for a in xs if keep10(a, b)])


def ordered(csp, x, y, gap):
    """tests/cpp/dropin_scenarios.cpp OrderedConstraint: Evaluate x + gap <= y; assigning x: ExcludeInf(x + gap) on y;
    assigning y: ExcludeSup(y - gap + 1) on x."""
    xs, ys = domain_values(csp.domains[x]), domain_values(csp.domains[y])
    return tabulate(x, y, xs, ys, lambda a, b: a + gap <= b, lambda a, b: b >= a + gap, lambda a, b: a < b - gap + 1)


def gap_table(csp, x, y, gap):
    """tests/cpp/dropin_scenarios.cpp GapConstraint (check-only): |x - y| != gap."""
    xs, ys = domain_values(csp.domains[x]), domain_values(csp.domains[y])
    return TableConstraint(x, y, [(a, b) for a in xs for b in ys if abs(a - b) != gap])


def user_filter_scenario(n, g, reverse_domains, extra_gap) -> CSP:
    """tests/cpp/dropin_scenarios.cpp user_filter."""
    csp = CSP()
    for i in range(n):
        if i % 2 == 0:
            csp.AddIntVar(0, n + 3)
        else:
            csp.AddIntVar(Domain(DomainType.Values, [n + 2 - k if reverse_domains else k for k in range(n + 3)]))
    for i in range(n - 1):
        csp.AddConstraint(ordered(csp, i, i + 1, g if i % 2 else 1))
    csp.AddConstraint(AllDifferentConstraint(list(range(n))))
    if extra_gap:
        csp.AddConstraint(gap_table(csp, 0, n - 1, extra_gap))
    csp.AddConstraint(OpConstraint(1, n - 2, Op.NotEqual, -3))
    csp.FinalizeModel()
    return csp


SCENARIOS = {"user_filter_sat": (5, 2, False, 0), "user_filter_reversed_domains": (6, 1, True, 4),
             "user_filter_unsat": (6, 3, False, 0), "user_filter_gap": (5, 1, True, 6)}


def _tree(r):
    return (r.status, r.solutions, r.nodes, r.first)


def _cmp(got, want, what):
    assert _tree(got) == _tree(want), (what, got, want)


def _keep_classes(csp):
    """How each FILTER direction's keep set relates to its allow set: equal, stronger (a subset), weaker (a superset) or
    other."""
    seen = set()
    for c in csp.constraints:
        if isinstance(c, FilterConstraint):
            allow = set(c.allow)
            for keep in (set(c.keep01), set(c.keep10)):
                seen.add("equal" if keep == allow else "stronger" if keep < allow else "weaker" if keep > allow else "other")
    return seen


# ---- CPU: the oracle ---------------------------------------------------------------------------------------------------

def test_oracle_matches_reference_user_filter_scenarios():
    """The oracle's FILTER against the four user_filter scenarios the unmodified reference ran (drop-in goldens): outcome,
    stats.assigned_vars, solution and assign_order."""
    gold = {}
    for line in open(os.path.join(GOLD, "dropin_reference.jsonl")):
        if line.strip():
            d = json.loads(line)
            gold[d["name"]] = d
    for name, args in SCENARIOS.items():
        want = gold[name]
        o = O.solve(user_filter_scenario(*args), "first")
        assert (o.status == "sat") == want["ok"], name
        assert o.nodes == want["assigned_vars"], name
        assert (o.first or [UNASSIGNED] * len(want["values"])) == want["values"], name
        assert o.order == want["assign_order"], name


def fc_filters_only(csp: CSP, mode: str):
    """A plain forward-checking search (ForwardCheckingStep, dequan.h:494-571) for models whose constraints are all
    FILTERs and whose domains list no value twice -> (status, solutions, nodes, first).  Its filter reads keep01 when v0
    is assigned and keep10 when v1 is: the one property the reference scenarios cannot pin, because their filters keep
    the same pairs in both directions."""
    nv = len(csp.domains)
    order = sorted(range(nv), key=lambda v: (len(domain_values(csp.domains[v])), v))
    links = [[c for c in csp.constraints if v in (c.v0, c.v1)] for v in range(nv)]
    inst = [None] * nv
    st = {"nodes": 0, "count": 0, "first": None}

    def step(k, doms):
        if k == nv:
            return True
        v = order[k]
        for val in doms[v]:
            st["nodes"] += 1
            inst[v] = val
            ok = all(inst[c.v0] is None or inst[c.v1] is None or (inst[c.v0], inst[c.v1]) in set(c.allow) for c in links[v])
            if ok and mode == "count" and k == nv - 1:       # the counting constraint, linked last
                st["count"] += 1
                st["first"] = st["first"] or list(inst)
                ok = False
            if ok:
                nd = list(doms)
                for c in links[v]:
                    if (inst[c.v0] is None) == (inst[c.v1] is None):
                        continue
                    if inst[c.v0] is not None:
                        nd[c.v1] = [w for w in nd[c.v1] if (inst[c.v0], w) in set(c.keep01)]
                        ok = bool(nd[c.v1])
                    else:
                        nd[c.v0] = [w for w in nd[c.v0] if (w, inst[c.v1]) in set(c.keep10)]
                        ok = bool(nd[c.v0])
                    if not ok:
                        break
                if ok and step(k + 1, nd):
                    return True
            inst[v] = None
        return False

    found = step(0, [domain_values(d) for d in csp.domains])
    if mode == "count":
        return ("sat" if st["count"] else "unsat"), st["count"], st["nodes"], st["first"]
    return ("sat" if found else "unsat"), int(found), st["nodes"], list(inst) if found else None


def test_oracle_filter_directions():
    """The oracle against fc_filters_only on models of FILTERs only, with keep sets that differ by direction."""
    asym = 0
    for seed in range(300):
        rng = random.Random(seed)
        csp = CSP()
        for _ in range(rng.randint(2, 6)):
            csp.AddIntVar(random_domain(rng, -3, 6, 5))
        vals = [domain_values(d) for d in csp.domains]
        for _ in range(rng.randint(1, 7)):
            a, b = rng.sample(range(len(vals)), 2)
            csp.AddConstraint(random_filter(rng, a, b, vals[a], vals[b]))
        csp.FinalizeModel()
        asym += any(set(c.keep01) != set(c.keep10) for c in csp.constraints)
        for mode in ("first", "count"):
            assert _tree(O.solve(csp, mode)) == fc_filters_only(csp, mode), (seed, mode)
    assert asym > 200


def _op_keeps(op, y, t):
    """The built-in filter (OpConstraint DoCheck, dequan.h:636-669): does y survive `y (op) t`?"""
    return {Op.NotEqual: y != t, Op.SupEqual: y >= t, Op.Sup: y >= t + 1, Op.InfEqual: y < t + 1, Op.Inf: y < t}[op]


def _op_evaluate(op, a, b, off):
    return {Op.NotEqual: a != b + off, Op.SupEqual: a >= b + off, Op.Sup: a > b + off, Op.InfEqual: a <= b + off,
            Op.Inf: a < b + off}[op]


REVERSE = {Op.NotEqual: Op.NotEqual, Op.SupEqual: Op.InfEqual, Op.Sup: Op.Inf, Op.InfEqual: Op.SupEqual, Op.Inf: Op.Sup}


def op_as_filter(csp, c: OpConstraint) -> FilterConstraint:
    """An OpConstraint restated as a user filter: keep sets from the built-in filter (v0 = a assigned: v1 filtered with the
    reversed op against a - off; v1 = b assigned: v0 filtered with the op against b + off), allow set from Evaluate."""
    xs, ys = domain_values(csp.domains[c.v0]), domain_values(csp.domains[c.v1])
    op, off = c.op, c.offset
    return tabulate(c.v0, c.v1, xs, ys, lambda a, b: _op_evaluate(op, a, b, off),
                    lambda a, b: _op_keeps(REVERSE[op], b, a - off), lambda a, b: _op_keeps(op, a, b + off))


def _restated(csp, fn) -> CSP:
    out = CSP([Domain(d.type, list(d.values)) for d in csp.domains], [fn(c) for c in csp.constraints], csp.assign_order)
    out.FinalizeModel()
    return out


@pytest.mark.parametrize("op", [Op.NotEqual, Op.SupEqual, Op.Sup, Op.InfEqual, Op.Inf])
def test_op_constraint_restated_as_filter(op):
    """Each non-Equal OpConstraint, offsets -2..2, on Values and Ranges domains, restated as a FILTER: same status, nodes,
    solution count and first solution."""
    for off in range(-2, 3):
        for dt in (DomainType.Values, DomainType.Ranges):
            for seed in range(6):
                rng = random.Random(f"{int(op)} {off} {int(dt)} {seed}")
                csp = CSP()
                for _ in range(5):
                    k = rng.randint(2, 6)
                    if dt == DomainType.Values:
                        csp.AddIntVar(Domain(DomainType.Values, rng.sample(range(-3, 9), k)))
                    else:
                        a = rng.randint(-3, 4)
                        csp.AddIntVar(Domain(DomainType.Ranges, [a, a + k] if rng.random() < 0.6 else [a, a + 2, a + 3, a + k + 2]))
                for _ in range(4):
                    a, b = rng.sample(range(5), 2)
                    csp.AddConstraint(OpConstraint(a, b, op, off))
                a, b = rng.sample(range(5), 2)
                csp.AddConstraint(OpConstraint(a, b, Op.Equal, rng.randint(-1, 1)))
                csp.AddConstraint(AllDifferentConstraint(rng.sample(range(5), 3)))
                csp.FinalizeModel()
                filt = _restated(csp, lambda c: op_as_filter(csp, c) if isinstance(c, OpConstraint) and c.op != Op.Equal else c)
                for mode in ("first", "count"):
                    assert _tree(O.solve(filt, mode)) == _tree(O.solve(csp, mode)), (op, off, dt, seed, mode)


def test_table_restated_as_keep_all_filter():
    """A TABLE is a FILTER whose filter keeps everything."""
    n = 0
    for csp in model_suite(200, 1000):
        if not any(isinstance(c, TableConstraint) for c in csp.constraints):
            continue
        n += 1

        def restate(c):
            if not isinstance(c, TableConstraint):
                return c
            xs, ys = domain_values(csp.domains[c.v0]), domain_values(csp.domains[c.v1])
            allow = set(c.pairs)
            return tabulate(c.v0, c.v1, xs, ys, lambda a, b: (a, b) in allow, lambda a, b: True, lambda a, b: True)

        filt = _restated(csp, restate)
        for mode in ("first", "count"):
            assert _tree(O.solve(filt, mode)) == _tree(O.solve(csp, mode)), mode
    assert n > 50


def test_generator_covers_every_keep_class():
    """filter_suite draws keep sets equal to, stronger than, weaker than and unrelated to the allow set, and its filters
    change answers: replacing each FILTER by a TABLE of its allow set changes the node count of many models."""
    seen, changed = set(), 0
    for csp in filter_suite(200):
        seen |= _keep_classes(csp)

        def as_table(c):
            return TableConstraint(c.v0, c.v1, c.allow) if isinstance(c, FilterConstraint) else c

        changed += O.solve(csp, "count").nodes != O.solve(_restated(csp, as_table), "count").nodes
    assert seen == {"equal", "stronger", "weaker", "other"}, seen
    assert changed > 80, changed


# ---- CPU: refusals -------------------------------------------------------------------------------------------------------

class Raw:
    def __init__(self, kind, payload):
        self.kind, self.payload = kind, payload

    def lower(self):
        return self.kind, list(self.payload)


def _compile_code(payload, nv=3):
    csp = CSP()
    for _ in range(nv):
        csp.AddIntVar(0, 4)
    csp.AddConstraint(Raw(ConKind.FILTER, payload))
    try:
        api.Model(csp)
    except api.DequanError as e:
        return e.code
    return 0


def test_compiler_refusals(product_lib):
    ok = [0, 1, 1, 1, 1, 0, 1, 0, 2, 1, 0]                    # one allowed pair, one kept pair per direction
    assert _compile_code(ok) == 0
    assert _compile_code(ok[:-1]) == -1                       # payload one short
    assert _compile_code(ok + [3]) == -1                      # one long
    assert _compile_code([0, 1, 0, 0]) == -1                  # no counts
    assert _compile_code([0, 1, -1, 1, 1, 0, 1]) == -1         # negative counts whose sum still fits the length
    assert _compile_code([0, 1, 1, -1, 1, 0, 1]) == -1
    assert _compile_code([0, 1, 1, 1, -1, 0, 1]) == -1
    assert _compile_code([1, 1] + ok[2:]) == -2               # v0 == v1
    assert _compile_code([0, 3] + ok[2:]) == -1               # out of range
    assert _compile_code([-1, 1] + ok[2:]) == -1


def _ne_filter(csp, c: OpConstraint):
    """A NotEqual-0 pair as a FILTER whose keep mask is exactly "different value"; Evaluate accepts the same pairs."""
    xs, ys = domain_values(csp.domains[c.v0]), domain_values(csp.domains[c.v1])
    return tabulate(c.v0, c.v1, xs, ys, lambda a, b: a != b, lambda a, b: a != b, lambda a, b: a != b)


def test_filter_models_are_never_a_class(product_lib):
    """The class engines know nothing of K_CHK: a model with a FILTER is generic even when its keep mask is exactly
    "different value" (K_NE_SAME) and its allow set says the same."""
    q = nqueens(7)
    s = sudoku_template()
    c = colouring(12, 3, [(i, (i + 1) % 12) for i in range(12)] + [(i, (i + 5) % 12) for i in range(12)])
    for base, cls in ((q, "queens"), (s, "sudoku9"), (c, "ne_same")):
        assert api.Model(base).info()["model_class"] == cls
        first = base.constraints[0]
        one = _restated(base, lambda k: _ne_filter(base, k) if k is first else k)
        assert api.Model(one).info()["model_class"] == "generic", cls
        keep_all_allow_ne = _restated(base, lambda k: tabulate(k.v0, k.v1, domain_values(base.domains[k.v0]),
                                                               domain_values(base.domains[k.v1]), lambda a, b: True,
                                                               lambda a, b: a != b, lambda a, b: a != b) if k is first else k)
        assert api.Model(keep_all_allow_ne).info()["model_class"] == "generic", cls


@pytest.fixture(scope="module")
def dropin_bin(product_lib, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("user_filters") / "user_filters")
    subprocess.check_call(["g++", "-std=c++11", "-O2", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o", out,
                           os.path.join(ROOT, "tests", "cpp", "user_filters.cpp"), "-L" + LIBDIR, "-ldequan_b200",
                           "-Wl,-rpath," + LIBDIR])
    return out


def test_dropin_refuses_illegal_filters(dropin_bin):
    """The lowering runs before any device call: each illegal filter throws dequan::b200::Error with its reason."""
    got = [json.loads(l) for l in subprocess.run([dropin_bin, "refusals"], capture_output=True, text=True, check=True,
                                                 timeout=60).stdout.splitlines()]
    want = {"touches_third": "changes a domain other than its unassigned endpoint's",
            "true_when_empty": "must answer false exactly when it empties the domain",
            "depends_on_others": "depends on the other values of the domain it filters"}
    assert [g["name"] for g in got] == list(want)
    for g in got:
        assert g["thrown"] and want[g["name"]] in g["what"], g


# ---- GPU ------------------------------------------------------------------------------------------------------------------

def _suite():
    return filter_suite(160) + [random_filter_model(30000 + s, 10 + s % 6, 12 + s % 7, 5 + s % 3) for s in range(40)]


@pytest.mark.gpu
def test_random_filter_models_every_engine(product_lib):
    """auto / warp / reg, FIRST and COUNT_ALL, split depths 0-3, against the oracle; the register engine (pattern
    AND / WEQ / CHK per pair) serves a share of them."""
    used = solves = 0
    for i, csp in enumerate(_suite()):
        m = api.Model(csp)
        for mode in ("first", "count"):
            want = O.solve(csp, mode)
            b = m.solve_tree(mode)
            _cmp(b, want, (i, mode, "auto"))
            solves += 1
            used += b.engine == "reg"
            _cmp(m.solve_tree(mode, engine="warp"), want, (i, mode, "warp"))
            try:
                r = m.solve_tree(mode, engine="reg")
            except api.DequanError:
                assert b.engine != "reg"
            else:
                _cmp(r, want, (i, mode, "reg"))
            for depth in (1, 2, 3):
                _cmp(m.solve_tree(mode, split_depth=depth), want, (i, mode, depth))
                _cmp(m.solve_tree(mode, split_depth=depth, engine="warp"), want, (i, mode, depth, "warp"))
    print("register engine used", used, "of", solves)
    assert used > solves // 4


def _wide_models():
    out = []
    for seed in range(40000, 40100):
        csp = random_filter_model(seed, 3 + seed % 2, 3 + seed % 4, 40 + seed % 25)
        if max(len(domain_values(d)) for d in csp.domains) <= 32:
            continue
        if O.solve(csp, "count", budget=200_000).status == "budget":     # keep the oracle quick
            continue
        out.append(csp)
    return out


@pytest.mark.gpu
def test_wide_filter_models(product_lib):
    """33..64 values (64-bit domain words, the warp engine): FIRST and COUNT_ALL, partitioned counts that add up, and
    FIRST-mode node accounting across partitions."""
    models = _wide_models()
    assert len(models) >= 20
    for i, csp in enumerate(models):
        m = api.Model(csp)
        for mode in ("first", "count"):
            want = O.solve(csp, mode)
            r = m.solve_tree(mode)
            _cmp(r, want, (i, mode))
            assert r.engine == "warp"
            _cmp(m.solve_tree(mode, split_depth=2), want, (i, mode, 2))
        g = O.solve(csp, "count")
        parts = [m.solve_tree("count", split_depth=2, part_rank=k, part_count=3) for k in range(3)]
        assert (sum(p.solutions for p in parts), sum(p.nodes for p in parts)) == (g.solutions, g.nodes), i
        f = O.solve(csp, "first")
        hs = [api.Model(csp) for _ in range(3)]
        loc = [h.solve_tree("first", split_depth=1, part_rank=k, part_count=3) for k, h in enumerate(hs)]
        key = min(p.first_key for p in loc)
        if f.status == "sat":
            assert [p.first for p in loc if p.first_key == key][0] == f.first, i
            assert sum(h.nodes_upto(key) for h in hs) == f.nodes, i
        else:
            assert all(p.status == "unsat" for p in loc) and sum(p.nodes for p in loc) == f.nodes, i


@pytest.mark.gpu
def test_enumeration_in_oracle_order(product_lib):
    """Every solution in the oracle's visiting order, whole (warp and auto, split depths 0-2) and partitioned."""
    checked = 0
    for i, csp in enumerate(filter_suite(400, 50000)):
        want, total = O.enumerate_solutions(csp, 20000)
        if total > 20000:
            continue
        checked += total > 1
        m = api.Model(csp)
        for engine in ("warp", "auto"):
            for depth in (0, 1, 2):
                got, r = m.enumerate_solutions(max(total, 1), split_depth=depth, engine=engine)
                assert got.tolist() == want and r.solutions == total, (i, engine, depth)
                assert r.nodes == O.solve(csp, "count").nodes, (i, engine, depth)
        if total > 1:
            parts = [m.enumerate_solutions(total, split_depth=2, part_rank=k, part_count=3)[0].tolist() for k in range(3)]
            assert sorted(sum(parts, [])) == sorted(want), i
            pos = {tuple(s): j for j, s in enumerate(want)}
            for p in parts:
                idx = [pos[tuple(s)] for s in p]
                assert idx == sorted(idx), i
    assert checked > 30


def pigeonhole_filters(holes: int) -> CSP:
    """holes + 1 pigeons, pairwise different through FILTERs: unsat, and far more than a warp's budget of nodes."""
    csp = CSP()
    for _ in range(holes + 1):
        csp.AddIntVar(0, holes)
    xs = list(range(holes))
    for a in range(holes + 1):
        for b in range(a + 1, holes + 1):
            csp.AddConstraint(tabulate(a, b, xs, xs, lambda p, q: p != q, lambda p, q: p != q, lambda p, q: p != q))
    csp.FinalizeModel()
    return csp


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["first", "count"])
def test_solve_models_batch(product_lib, mode):
    """api.solve_models on a mixed batch of FILTER models, one of which outgrows the in-batch node budget and goes
    through the split search: every entry equals the oracle and a single solve_tree of the same handle."""
    csps = filter_suite(80, 60000) + _wide_models()[:8] + [pigeonhole_filters(8)]
    models = [api.Model(c) for c in csps]
    r = api.solve_models(models, mode)
    assert r.n_split >= 1
    assert r.nodes[-1] > 1 << 14
    for i, (csp, m) in enumerate(zip(csps, models)):
        want = O.solve(csp, mode)
        got = (r.status[i], r.solutions[i], r.nodes[i], r.first[i])
        assert got == _tree(want) == _tree(m.solve_tree(mode)), (mode, i)


# ---- GPU: cell batches ------------------------------------------------------------------------------------------------

BATCH = 4 * 148 * 16 * 4
STATUS = {"unsat": 0, "sat": 1, "budget": 2}


def _batch_templates():
    out = []
    for seed in range(70000, 70200):
        t = random_filter_model(seed, 8 + seed % 5, 5 + seed % 4, 6, lo=1, hi=9)
        sols, total = O.enumerate_solutions(t, 300)
        if total >= 20:
            out.append((t, np.array(sols, dtype=np.int64).reshape(len(sols), len(t.domains))))
            if len(out) == 4:
                return out
    raise AssertionError("not enough satisfiable templates")


def _expected(t, rows, budget, cache):
    nv = len(t.domains)
    st, nodes, sol = [], [], []
    for r in rows:
        key = (bytes(r[:nv]), budget)
        if key not in cache:
            if not all(not r[v] or int(r[v]) in domain_values(d) for v, d in enumerate(t.domains)):
                cache[key] = (3, 0, bytes(nv))
            else:
                o = O.solve(instance_csp(t, r), "first", budget)
                cache[key] = (STATUS[o.status], o.nodes, bytes(x & 0xFF for x in o.first) if o.status == "sat" else bytes(nv))
        s, n, b = cache[key]
        st.append(s), nodes.append(n), sol.append(b)
    return (np.array(st, dtype=np.uint8), np.array(nodes, dtype=np.uint64),
            np.frombuffer(b"".join(sol), dtype=np.uint8).reshape(len(rows), nv))


def _check_batch(got, want, what):
    st, nodes, sol = want
    nv = sol.shape[1]
    bad = np.nonzero((got.status != st) | (got.nodes != nodes) | (got.solution[:, :nv] != sol).any(axis=1))[0]
    assert len(bad) == 0, (what, f"{len(bad)} of {len(st)} instances differ",
                           [(int(i), int(got.status[i]), int(st[i]), int(got.nodes[i]), int(nodes[i])) for i in bad[:5]])
    assert got.total_nodes == int(nodes.sum()), what


@pytest.mark.gpu
def test_cell_batches_with_filter_templates(product_lib):
    """dq_solve_batch_cells on FILTER templates (the generic batch kernel, one launch): every instance against the oracle
    without a budget and at the median budget; an instance needing N nodes finishes with budget N, runs out with N - 1."""
    seen = set()
    for j, (t, sols) in enumerate(_batch_templates()):
        cache = {}
        m = api.Model(t)
        assert m.info()["model_class"] == "generic"
        rows = make_rows(t, sols, 1200, seed=j)
        rng = np.random.default_rng(j)
        batch = np.tile(rows, (-(-BATCH // len(rows)), 1))
        batch = np.ascontiguousarray(batch[rng.permutation(len(batch))])
        full = m.solve_batch_cells(batch)
        _check_batch(full, _expected(t, batch, 0, cache), (j, 0))
        assert full.launches == 1
        st, nodes, sol = _expected(t, rows, 0, cache)
        budget = max(1, int(np.median(nodes)))
        r = m.solve_batch_cells(batch, node_budget=budget)
        _check_batch(r, _expected(t, batch, budget, cache), (j, budget))
        seen |= set(r.status.tolist())
        sat = np.nonzero(st == 1)[0]
        for i in sat[np.argsort(nodes[sat])][[0, len(sat) // 2, -1]]:
            one, need = np.ascontiguousarray(rows[i:i + 1]), int(nodes[i])
            a = m.solve_batch_cells(one, node_budget=need)
            assert (a.status[0], int(a.nodes[0]), a.solution[0].tobytes()) == (1, need, sol[i].tobytes()), (j, i)
            if need > 1:
                b = m.solve_batch_cells(one, node_budget=need - 1)
                assert (b.status[0], int(b.nodes[0])) == (2, need), (j, i)
    assert seen == {0, 1, 2, 3}, seen


@pytest.mark.gpu
def test_multi_device_solve(product_lib):
    """dq_solve_tree_multi with the device list (0, 0): the split tree dealt to two workers and reduced."""
    for i, csp in enumerate(filter_suite(40, 80000)):
        m = api.Model(csp)
        for mode in ("first", "count"):
            _cmp(m.solve_tree_multi(mode, (0, 0), split_depth=2), O.solve(csp, mode), (i, mode))


# ---- GPU: the drop-in header end to end ---------------------------------------------------------------------------------

REL = [lambda a, b, g: a + g <= b, lambda a, b, g: a + g < b, lambda a, b, g: a + g - 2 <= b,
       lambda a, b, g: (a + b + g) % 3 != 0, lambda a, b, g: True, lambda a, b, g: a != b + g]


@pytest.mark.gpu
def test_dropin_filters_stronger_and_weaker_than_evaluate(dropin_bin):
    """User filters that keep more or fewer pairs than their Evaluate accepts, through ForwardCheckingStep and SolveAll
    (TabulateUserConstraint with keep != allow): both paths agree, and each model rebuilt from FilterConstraints gives
    the oracle's outcome, node count, solution and order."""
    lines = [json.loads(l) for l in subprocess.run([dropin_bin], capture_output=True, text=True, check=True,
                                                   timeout=300).stdout.splitlines()]
    step = [l for l in lines if l["path"] == "step"]
    batch = [l for l in lines if l["path"] == "all"]
    assert len(step) == len(batch) == 22
    classes = set()
    for s, b in zip(step, batch):
        assert dict(s, path="") == dict(b, path=""), s["name"]
        csp = CSP()
        for d in s["domains"]:
            csp.AddIntVar(Domain(DomainType(d["t"]), d["v"]))
        for x, y, ev, k01, k10, g in s["rels"]:
            xs, ys = domain_values(csp.domains[x]), domain_values(csp.domains[y])
            csp.AddConstraint(tabulate(x, y, xs, ys, lambda a, b, e=ev, g=g: REL[e](a, b, g),
                                       lambda a, b, k=k01, g=g: REL[k](a, b, g), lambda a, b, k=k10, g=g: REL[k](a, b, g)))
        if s["alldiff"]:
            csp.AddConstraint(AllDifferentConstraint(list(range(len(s["domains"])))))
        csp.FinalizeModel()
        classes |= _keep_classes(csp)
        o = O.solve(csp, "first")
        assert (o.status == "sat") == s["ok"] and o.nodes == s["assigned_vars"] and o.order == s["assign_order"], s["name"]
        assert (o.first or [UNASSIGNED] * len(s["values"])) == s["values"], s["name"]
    assert {"stronger", "weaker", "other"} <= classes, classes
