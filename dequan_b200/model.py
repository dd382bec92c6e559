"""Python mirror of dequan's modelling API, lowered to the flat `dq_model_desc`.

The product's host side is C++ (include/dequan.h over include/dequan_b200.h); this
module exists so the tests and bench.py can state models with the reference's own
vocabulary (`CSP.AddIntVar`, `OpConstraint(v0, v1, Op.NotEqual, off)` ...,
/root/reference/dequan.h:328-355, 174-268) and hand the identical descriptor to the
C ABI, to the CPU oracle and (as text) to the reference driver.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from enum import IntEnum
from typing import List, Sequence

import numpy as np

UNASSIGNED = -(2**31 - 1)  # InstVar::UNASSIGNED == -INT_MAX, dequan.h:122


class DomainType(IntEnum):  # dequan.h:70-74
    Values = 0
    Ranges = 1


class Op(IntEnum):  # OpConstraint::Op, dequan.h:176-184
    Equal = 0
    NotEqual = 1
    SupEqual = 2
    Sup = 3
    InfEqual = 4
    Inf = 5


class ConKind(IntEnum):  # include/dequan_b200.h dq_con_kind
    OP = 0
    EQ = 1
    ALLDIFF = 2
    ORRANGE = 3
    TABLE = 4
    FILTER = 5


@dataclass
class Domain:  # dequan.h:76-96
    type: DomainType
    values: List[int]


@dataclass
class OpConstraint:  # v0 (op) v1 + offset, dequan.h:173-197
    v0: int
    v1: int
    op: Op
    offset: int = 0

    def lower(self):
        return ConKind.OP, [self.v0, self.v1, int(self.op), self.offset]

    def text(self):
        return f"op {self.v0} {self.v1} {int(self.op)} {self.offset}"


@dataclass
class EqualityConstraint:  # dequan.h:200-211
    v0: int
    v1: int

    def lower(self):
        return ConKind.EQ, [self.v0, self.v1]

    def text(self):
        return f"eq {self.v0} {self.v1}"


@dataclass
class OrRangeConstraint:  # dequan.h:242-254
    v0: int
    v1: int
    min: int
    max: int

    def lower(self):
        return ConKind.ORRANGE, [self.v0, self.v1, self.min, self.max]

    def text(self):
        return f"orrange {self.v0} {self.v1} {self.min} {self.max}"


@dataclass
class AllDifferentConstraint:  # dequan.h:257-268
    vars: List[int]

    def lower(self):
        return ConKind.ALLDIFF, list(self.vars)

    def text(self):
        return f"alldiff {len(self.vars)} " + " ".join(map(str, self.vars))


@dataclass
class TableConstraint:
    """A user-defined binary `dequan::Constraint` (dequan.h:134-148) whose Evaluate has been
    tabulated into allowed (v0, v1) value pairs; check-only, like the base-class default
    AplyArcConsistency (dequan.h:147)."""
    v0: int
    v1: int
    pairs: List[tuple]

    def lower(self):
        flat = [self.v0, self.v1]
        for a, b in self.pairs:
            flat += [a, b]
        return ConKind.TABLE, flat

    def text(self):
        return f"table {self.v0} {self.v1} {len(self.pairs)} " + " ".join(f"{a} {b}" for a, b in self.pairs)


@dataclass
class FilterConstraint:
    """A user-defined binary `dequan::Constraint` that overrides AplyArcConsistency (dequan.h:145-147), tabulated the
    way include/dequan.h's TabulateUserConstraint does it: `allow` = the (v0, v1) value pairs its Evaluate accepts;
    `keep01` = the pairs (a, b) such that assigning v0 = a leaves b in v1's domain; `keep10` = the pairs (a, b) such that
    assigning v1 = b leaves a in v0's domain.  Every pair is (value of v0, value of v1)."""
    v0: int
    v1: int
    allow: List[tuple]
    keep01: List[tuple]
    keep10: List[tuple]

    def lower(self):
        flat = [self.v0, self.v1, len(self.allow), len(self.keep01), len(self.keep10)]
        for pairs in (self.allow, self.keep01, self.keep10):
            for a, b in pairs:
                flat += [a, b]
        return ConKind.FILTER, flat

    def text(self):
        raise NotImplementedError("the reference driver's .dqm format has no filtering user constraint")


class dq_model_desc(C.Structure):  # include/dequan_b200.h
    _fields_ = [
        ("n_vars", C.c_int32),
        ("dom_type", C.POINTER(C.c_int32)),
        ("dom_off", C.POINTER(C.c_int32)),
        ("dom_vals", C.POINTER(C.c_int32)),
        ("n_cons", C.c_int32),
        ("con_kind", C.POINTER(C.c_int32)),
        ("con_off", C.POINTER(C.c_int32)),
        ("con_data", C.POINTER(C.c_int32)),
        ("assign_order", C.POINTER(C.c_int32)),
    ]


@dataclass
class CSP:  # dequan.h:328-355
    domains: List[Domain] = field(default_factory=list)
    constraints: list = field(default_factory=list)
    assign_order: List[int] = None  # explicit Assignment::assign_order (dequan.h:316); None = Reset's sort

    def AddIntVar(self, a, b=None) -> int:  # dequan.h:454-466
        if b is None:
            dom = a
        else:
            dom = Domain(DomainType.Ranges, [a, b])
        self.domains.append(Domain(DomainType(dom.type), list(dom.values)))
        return len(self.domains) - 1

    def AddFixedVar(self, val: int) -> int:  # dequan.h:467-471
        return self.AddIntVar(Domain(DomainType.Values, [val]))

    def AddBoolVar(self) -> int:  # dequan.h:472-476
        return self.AddIntVar(Domain(DomainType.Values, [0, 1]))

    def AddConstraint(self, con) -> None:  # dequan.h:477-483
        self.constraints.append(con)

    def FinalizeModel(self) -> None:  # dequan.h:484-492 (linking happens in dq_compile)
        pass

    # ---- lowering -----------------------------------------------------------------------
    def arrays(self):
        nv = len(self.domains)
        dom_type = np.array([int(d.type) for d in self.domains], dtype=np.int32).reshape(nv)
        dom_off = np.zeros(nv + 1, dtype=np.int32)
        vals: List[int] = []
        for i, d in enumerate(self.domains):
            vals += d.values
            dom_off[i + 1] = len(vals)
        dom_vals = np.array(vals if vals else [0], dtype=np.int32)
        nc = len(self.constraints)
        con_kind = np.zeros(max(nc, 1), dtype=np.int32)
        con_off = np.zeros(nc + 1, dtype=np.int32)
        data: List[int] = []
        for i, c in enumerate(self.constraints):
            k, payload = c.lower()
            con_kind[i] = int(k)
            data += payload
            con_off[i + 1] = len(data)
        con_data = np.array(data if data else [0], dtype=np.int32)
        return dom_type, dom_off, dom_vals, con_kind, con_off, con_data

    def desc(self):
        """Returns (dq_model_desc, keepalive) — keepalive owns the numpy buffers."""
        arrs = self.arrays()
        p = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
        order = None
        if self.assign_order is not None:
            order = np.array(self.assign_order, dtype=np.int32)
            arrs = arrs + (order,)
        d = dq_model_desc(len(self.domains), p(arrs[0]), p(arrs[1]), p(arrs[2]),
                          len(self.constraints), p(arrs[3]), p(arrs[4]), p(arrs[5]),
                          p(order) if order is not None else None)
        return d, arrs

    def to_text(self) -> str:
        """`.dqm` text consumed by oracle/ref_driver.cpp (read_model)."""
        out = [f"dqm {len(self.domains)} {len(self.constraints)}"]
        for d in self.domains:
            out.append(("R" if d.type == DomainType.Ranges else "V") + f" {len(d.values)} " + " ".join(map(str, d.values)))
        out += [c.text() for c in self.constraints]
        return "\n".join(out) + "\n"


# ---- model builders for BASELINE.json's configs ---------------------------------------------

def nqueens(n: int) -> CSP:
    """/root/reference/test/main-test.cpp:32-50 — 3 NotEqual OpConstraints per pair."""
    csp = CSP()
    q = [csp.AddIntVar(0, n) for _ in range(n)]
    for i in range(n):
        for j in range(i + 1, n):
            csp.AddConstraint(OpConstraint(q[i], q[j], Op.NotEqual, 0))
            csp.AddConstraint(OpConstraint(q[i], q[j], Op.NotEqual, j - i))
            csp.AddConstraint(OpConstraint(q[i], q[j], Op.NotEqual, i - j))
    csp.FinalizeModel()
    return csp


def sudoku_groups(boxes: bool = True) -> List[List[int]]:
    g = [[r * 9 + c for c in range(9)] for r in range(9)]
    g += [[r * 9 + c for r in range(9)] for c in range(9)]
    if boxes:
        g += [[(b // 3 * 3 + k // 3) * 9 + (b % 3 * 3 + k % 3) for k in range(9)] for b in range(9)]
    return g


def sudoku_peer_pairs(boxes: bool = True) -> List[tuple]:
    """Unordered peer pairs in the order oracle/ref_driver.cpp's sudoku_model emits them."""
    seen, out = set(), []
    for grp in sudoku_groups(boxes):
        for a in range(len(grp)):
            for b in range(a + 1, len(grp)):
                u, v = sorted((grp[a], grp[b]))
                if (u, v) not in seen:
                    seen.add((u, v))
                    out.append((u, v))
    return out


def sudoku(cells: Sequence[int], boxes: bool = True, alldiff: bool = False) -> CSP:
    """main-test.cpp:110-149 (givens -> AddFixedVar, blanks -> AddIntVar(1,10)); with `boxes`
    the 9 box groups the reference test omits; all-different either native or as binary !=."""
    csp = CSP()
    for g in cells:
        if g:
            csp.AddFixedVar(int(g))
        else:
            csp.AddIntVar(1, 10)
    if alldiff:
        for grp in sudoku_groups(boxes):
            csp.AddConstraint(AllDifferentConstraint(grp))
    else:
        for u, v in sudoku_peer_pairs(boxes):
            csp.AddConstraint(OpConstraint(u, v, Op.NotEqual, 0))
    csp.FinalizeModel()
    return csp


def sudoku_template(boxes: bool = True) -> CSP:
    """All-blank Sudoku: the constraint graph shared by a batch (dq_solve_batch_cells)."""
    return sudoku([0] * 81, boxes=boxes)


def colouring(n: int, k: int, edges: Sequence[tuple]) -> CSP:
    csp = CSP()
    for _ in range(n):
        csp.AddIntVar(0, k)
    for u, v in edges:
        csp.AddConstraint(OpConstraint(int(u), int(v), Op.NotEqual, 0))
    csp.FinalizeModel()
    return csp


REFERENCE_SUDOKU = [int(ch) for ch in  # main-test.cpp:92-105
                    "003020600900305001001806400008102900700000008006708200002609500800203009005010300"]
