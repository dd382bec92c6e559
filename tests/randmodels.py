"""Seeded random binary CSPs exercising every constraint kind / domain quirk the engine supports."""
from __future__ import annotations

import random
from typing import List

from dequan_b200.model import (CSP, AllDifferentConstraint, Domain, DomainType, EqualityConstraint, FilterConstraint, Op,
                               OpConstraint, OrRangeConstraint, TableConstraint)


def random_domain(rng: random.Random, lo: int, hi: int, max_size: int) -> Domain:
    kind = rng.random()
    if kind < 0.4:  # single range
        a = rng.randint(lo, hi - 1)
        b = min(hi, a + rng.randint(1, max_size))
        return Domain(DomainType.Ranges, [a, b])
    if kind < 0.6:  # two ranges (ascending, disjoint)
        a = rng.randint(lo, hi - 3)
        b = a + rng.randint(1, max(1, max_size // 2))
        c = b + rng.randint(1, 3)
        d = c + rng.randint(1, max(1, max_size // 2))
        return Domain(DomainType.Ranges, [a, b, c, d])
    if kind < 0.9:  # explicit values, unsorted (SURVEY §9 Q2), no duplicates
        n = rng.randint(1, max_size)
        vals = rng.sample(range(lo, hi + max_size), n)
        return Domain(DomainType.Values, vals)
    return Domain(DomainType.Values, [rng.randint(lo, hi)])  # fixed var


def random_model(seed: int, n_vars: int = 6, n_cons: int = 8, max_dom: int = 6, kinds: str = "all") -> CSP:
    rng = random.Random(seed)
    csp = CSP()
    for _ in range(n_vars):
        csp.AddIntVar(random_domain(rng, -3, 6, max_dom))
    for _ in range(n_cons):
        a, b = rng.sample(range(n_vars), 2)
        r = rng.random()
        if kinds == "ne":
            csp.AddConstraint(OpConstraint(a, b, Op.NotEqual, rng.choice([0, 0, 1, -1, 2])))
        elif r < 0.45:
            csp.AddConstraint(OpConstraint(a, b, Op(rng.randint(0, 5)), rng.randint(-2, 2)))
        elif r < 0.55:
            csp.AddConstraint(EqualityConstraint(a, b))
        elif r < 0.70:
            m = rng.randint(2, min(4, n_vars))
            csp.AddConstraint(AllDifferentConstraint(rng.sample(range(n_vars), m)))
        elif r < 0.80:
            lo = rng.randint(-3, 4)
            csp.AddConstraint(OrRangeConstraint(a, b, lo, lo + rng.randint(1, 5)))
        else:
            pairs = [(x, y) for x in range(-3, 13) for y in range(-3, 13) if rng.random() < 0.6]
            csp.AddConstraint(TableConstraint(a, b, pairs))
    csp.FinalizeModel()
    return csp


def model_suite(n: int = 200, seed0: int = 1000) -> List[CSP]:
    out = []
    for i in range(n):
        rng = random.Random(seed0 + i)
        nv = rng.randint(2, 9)
        nc = rng.randint(1, 14)
        out.append(random_model(seed0 + i, nv, nc, rng.randint(2, 7), "ne" if i % 5 == 0 else "all"))
    return out


def random_model_dups(seed: int, n_vars: int = 6, n_cons: int = 9, max_dom: int = 5) -> CSP:
    """random_model with Values domains that list some values more than once (SURVEY.md par. 9 Q2: iteration visits every
    copy, Domain::Exclude erases the first match only, Domain::Intersect leaves one copy)."""
    csp = random_model(seed, n_vars, n_cons, max_dom)
    rng = random.Random(seed * 7919 + 13)
    for d in csp.domains:
        if d.type == DomainType.Values and rng.random() < 0.7:
            for _ in range(rng.randint(1, 3)):
                d.values.insert(rng.randint(0, len(d.values)), rng.choice(d.values))
    return csp


def dup_suite(n: int = 150, seed0: int = 5000) -> List[CSP]:
    out = []
    for i in range(n):
        rng = random.Random(seed0 + i)
        out.append(random_model_dups(seed0 + i, rng.randint(2, 8), rng.randint(2, 12), rng.randint(2, 5)))
    return out


def domain_values(d: Domain) -> List[int]:
    """The values of a domain in iteration order."""
    if d.type == DomainType.Values:
        return list(d.values)
    return [x for a, b in zip(d.values[::2], d.values[1::2]) for x in range(a, b)]


KEEP_CLASSES = ("equal", "stronger", "weaker", "unrelated")


def random_filter(rng: random.Random, v0: int, v1: int, xs: List[int], ys: List[int]) -> FilterConstraint:
    """A FILTER on (v0, v1) over the value lists xs, ys.  Each direction's keep set is drawn from one class relative to
    the allow set: equal to it, a subset (the filter is stronger than Evaluate), a superset (Evaluate rejects the rest)
    or unrelated; a quarter of the constraints use one class for both directions.  Some values of the assigned side
    then keep nothing (an immediate wipe-out) and some keep everything.  A few pairs name values outside the domains,
    and some pairs are listed twice: both must be ignored."""
    pairs = [(a, b) for a in xs for b in ys]
    allow = [p for p in pairs if rng.random() < rng.choice((0.3, 0.6, 0.9))]

    def keep_set(cls: str, side: int):
        if cls == "equal":
            keep = list(allow)
        elif cls == "stronger":
            keep = [p for p in allow if rng.random() < 0.7]
        elif cls == "weaker":
            keep = list(allow) + [p for p in pairs if p not in allow and rng.random() < 0.5]
        else:
            keep = [p for p in pairs if rng.random() < 0.6]
        for v in (xs if side == 0 else ys):              # per assigned value: keep nothing / keep everything
            u = rng.random()
            at = (lambda p, v=v: p[0] == v) if side == 0 else (lambda p, v=v: p[1] == v)
            if u < 0.08:
                keep = [p for p in keep if not at(p)]
            elif u < 0.16:
                keep = [p for p in keep if not at(p)] + [p for p in pairs if at(p)]
        rng.shuffle(keep)
        return keep

    c01 = rng.choice(KEEP_CLASSES)
    c10 = c01 if rng.random() < 0.25 else rng.choice(KEEP_CLASSES)
    keep01, keep10 = keep_set(c01, 0), keep_set(c10, 1)
    for lst in (allow, keep01, keep10):
        if lst and rng.random() < 0.3:
            lst.append(rng.choice(lst))                  # listed twice
        if rng.random() < 0.3:
            lst.append((max(xs) + 100, rng.choice(ys)))  # a value v0 never takes
            lst.append((rng.choice(xs), min(ys) - 100))  # a value v1 never takes
    rng.shuffle(allow)
    return FilterConstraint(v0, v1, allow, keep01, keep10)


def random_filter_model(seed: int, n_vars: int = 6, n_cons: int = 8, max_dom: int = 6, lo: int = -3, hi: int = 6) -> CSP:
    """random_model's kinds mixed with FILTERs (about half the constraints).  Some FILTERs share their pair with an
    Equal OpConstraint or an EqualityConstraint, in either link order, or with a TABLE or an order OpConstraint.  No
    duplicate values: the filter of a user constraint on a repeated value is not defined by the tabulation rules."""
    rng = random.Random(seed)
    csp = CSP()
    for _ in range(n_vars):
        csp.AddIntVar(random_domain(rng, lo, hi, max_dom))
    vals = [domain_values(d) for d in csp.domains]
    for _ in range(n_cons):
        a, b = rng.sample(range(n_vars), 2)
        r = rng.random()
        if r < 0.35:
            csp.AddConstraint(random_filter(rng, a, b, vals[a], vals[b]))
        elif r < 0.55:                                   # FILTER + Equal on the same pair, both orders
            eq = (OpConstraint(a, b, Op.Equal, rng.randint(-1, 1)) if rng.random() < 0.5
                  else EqualityConstraint(*rng.sample((a, b), 2)))
            f = random_filter(rng, a, b, vals[a], vals[b])
            for con in ((f, eq) if rng.random() < 0.5 else (eq, f)):
                csp.AddConstraint(con)
        elif r < 0.65:                                   # FILTER + TABLE or OP on the same pair
            if rng.random() < 0.5:
                other = TableConstraint(b, a, [(x, y) for x in vals[b] for y in vals[a] if rng.random() < 0.7])
            else:
                other = OpConstraint(b, a, Op(rng.randint(1, 5)), rng.randint(-2, 2))
            f = random_filter(rng, a, b, vals[a], vals[b])
            for con in ((f, other) if rng.random() < 0.5 else (other, f)):
                csp.AddConstraint(con)
        elif r < 0.8:
            csp.AddConstraint(OpConstraint(a, b, Op(rng.randint(0, 5)), rng.randint(-2, 2)))
        elif r < 0.9:
            m = rng.randint(2, min(4, n_vars))
            csp.AddConstraint(AllDifferentConstraint(rng.sample(range(n_vars), m)))
        else:
            c = rng.randint(lo, hi)
            csp.AddConstraint(OrRangeConstraint(a, b, c, c + rng.randint(1, 5)))
    csp.FinalizeModel()
    return csp


def filter_suite(n: int = 200, seed0: int = 20000) -> List[CSP]:
    out = []
    for i in range(n):
        rng = random.Random(seed0 + i)
        out.append(random_filter_model(seed0 + i, rng.randint(2, 9), rng.randint(1, 12), rng.randint(2, 7)))
    return out
