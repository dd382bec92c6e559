"""ctypes binding of the C ABI (include/dequan_b200.h -> dequan_b200/lib/libdequan_b200.so).

Used by tests/ and bench.py; the product's host side is the C++ drop-in header.  There is no
fallback: if the CUDA library is missing or no device is present every solve raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from .model import CSP, UNASSIGNED, dq_model_desc

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libdequan_b200.so")
U64_MAX = 2**64 - 1

DQ_MODE_FIRST, DQ_MODE_COUNT_ALL = 0, 1
ENGINE = {"auto": 0, "warp": 1, "lane": 2, "reg": 3}
ENGINE_NAME = {v: k for k, v in ENGINE.items()}
OUTCOME = {0: "unsat", 1: "sat", 2: "budget", 3: "invalid"}
MODEL_CLASS = {0: "generic", 1: "ne_same", 2: "queens", 3: "sudoku9"}


class DequanError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"dequan_b200 error {code}: {msg}")
        self.code = code


class dq_tree_opts(C.Structure):
    _fields_ = [("mode", C.c_int32), ("split_depth", C.c_int32), ("part_rank", C.c_int32), ("part_count", C.c_int32),
                ("node_budget", C.c_uint64), ("engine", C.c_int32), ("flags", C.c_int32)]


class dq_tree_result(C.Structure):
    _fields_ = [("outcome", C.c_int32), ("n_prefixes", C.c_int32), ("n_solutions", C.c_uint64), ("n_nodes", C.c_uint64),
                ("first_key", C.c_uint64), ("nodes_before_first", C.c_uint64), ("kernel_ms", C.c_double),
                ("engine_used", C.c_int32), ("split_depth_used", C.c_int32), ("kernel_launches", C.c_uint64),
                ("search_kernel_ms", C.c_double), ("frontier_nodes", C.c_uint64)]


class dq_batch_opts(C.Structure):
    _fields_ = [("node_budget", C.c_uint64), ("engine", C.c_int32), ("task_nodes", C.c_int32)]


class dq_count_opts(C.Structure):
    _fields_ = [("node_budget", C.c_uint64), ("solution_limit", C.c_uint64), ("engine", C.c_int32)]


class dq_batch_stats(C.Structure):
    _fields_ = [("n_sat", C.c_uint64), ("n_unsat", C.c_uint64), ("n_budget", C.c_uint64), ("total_nodes", C.c_uint64),
                ("kernel_ms", C.c_double), ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("search_kernel_ms", C.c_double)]


EXPORTS = ["dq_device_info", "dq_set_device", "dq_compile", "dq_free", "dq_model_info", "dq_model_order", "dq_model_table_bytes", "dq_solve_tree",
           "dq_solve_tree_multi", "dq_solve_models", "dq_tree_nodes_upto", "dq_enumerate_solutions", "dq_solve_batch_cells", "dq_solve_batch_cells_dev", "dq_solve_batch_graphs", "dq_solve_batch_graphs_dev",
           "dq_count_batch_cells", "dq_count_batch_graphs",
           "dq_measure_int_peak", "dq_last_error", "dq_version", "dq_parse_sudoku_lines", "dq_parse_dimacs_col"]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DequanError(-3, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32p, u8p, u64p = C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p
    L.dq_device_info.argtypes = [i32p, i32p, C.c_char_p, C.c_size_t]
    L.dq_set_device.argtypes = [C.c_int32]
    L.dq_compile.argtypes = [C.POINTER(dq_model_desc), C.POINTER(vp)]
    L.dq_free.argtypes = [vp]
    L.dq_free.restype = None
    L.dq_model_info.argtypes = [vp, i32p, i32p, i32p, i32p]
    L.dq_model_order.argtypes = [vp, i32p]
    L.dq_model_table_bytes.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.dq_solve_tree.argtypes = [vp, C.POINTER(dq_tree_opts), C.POINTER(dq_tree_result), i32p]
    L.dq_solve_tree_multi.argtypes = [vp, C.POINTER(dq_tree_opts), C.c_int32, i32p, C.POINTER(dq_tree_result), i32p]
    L.dq_solve_models.argtypes = [C.POINTER(vp), C.c_int64, C.POINTER(dq_tree_opts), i32p, u64p, u64p, i32p,
                                  C.POINTER(C.c_int64), C.POINTER(dq_batch_stats)]
    L.dq_tree_nodes_upto.argtypes = [vp, C.c_uint64, C.POINTER(C.c_uint64)]
    L.dq_enumerate_solutions.argtypes = [vp, C.POINTER(dq_tree_opts), C.POINTER(dq_tree_result), i32p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.dq_solve_batch_cells.argtypes = [vp, u8p, C.c_int64, C.c_int32, C.POINTER(dq_batch_opts), u8p, u64p, u8p,
                                       C.POINTER(dq_batch_stats)]
    L.dq_solve_batch_cells_dev.argtypes = L.dq_solve_batch_cells.argtypes
    L.dq_solve_batch_graphs.argtypes = [C.c_int32, C.c_int32, C.c_void_p, u8p, C.c_int64, C.POINTER(dq_batch_opts),
                                        u8p, u64p, u8p, C.POINTER(dq_batch_stats)]
    L.dq_solve_batch_graphs_dev.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, u8p, C.c_int64, C.POINTER(dq_batch_opts),
                                            u8p, u64p, u8p, C.POINTER(dq_batch_stats)]
    L.dq_count_batch_cells.argtypes = [vp, u8p, C.c_int64, C.c_int32, C.POINTER(dq_count_opts), u64p, u8p, u64p, u8p,
                                       C.POINTER(dq_batch_stats)]
    L.dq_count_batch_graphs.argtypes = [C.c_int32, C.c_int32, C.c_void_p, u8p, C.c_int64, C.POINTER(dq_count_opts),
                                        u64p, u8p, u64p, u8p, C.POINTER(dq_batch_stats)]
    L.dq_measure_int_peak.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.dq_parse_sudoku_lines.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    L.dq_parse_dimacs_col.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_int32), C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    L.dq_last_error.restype = C.c_char_p
    L.dq_version.restype = C.c_char_p
    for name in EXPORTS:
        if name not in ("dq_free", "dq_last_error", "dq_version"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise DequanError(rc, lib().dq_last_error().decode())


def device_info():
    sm, cc = C.c_int32(), C.c_int32()
    name = C.create_string_buffer(128)
    _check(lib().dq_device_info(C.byref(sm), C.byref(cc), name, 128))
    return {"sm_count": sm.value, "cc": cc.value, "name": name.value.decode()}


def set_device(ordinal: int):
    _check(lib().dq_set_device(ordinal))


def measure_int_peak():
    ops, ms = C.c_double(), C.c_double()
    _check(lib().dq_measure_int_peak(C.byref(ops), C.byref(ms)))
    return ops.value, ms.value


@dataclass
class TreeResult:
    status: str
    solutions: int
    nodes: int
    first: Optional[List[int]]
    first_key: int
    n_prefixes: int
    split_depth: int
    kernel_ms: float
    engine: str
    launches: int
    search_kernel_ms: float = 0.0
    frontier_nodes: int = 0


@dataclass
class BatchResult:
    solution: np.ndarray
    nodes: np.ndarray
    status: np.ndarray
    n_sat: int
    n_unsat: int
    n_budget: int
    total_nodes: int
    kernel_ms: float
    launches: int
    h2d_bytes: int
    d2h_bytes: int
    search_kernel_ms: float = 0.0


@dataclass
class CountResult:
    """Per instance of a counting batch: `solutions` (uint64; min(total, limit) when limit > 0), `first` (the DFS-first
    solution in the layout of the FIRST-mode batch, written whenever solutions >= 1), `nodes` and `status` (0 unsat,
    1 sat, 2 budget, 3 bad given); then the batch totals."""
    solutions: np.ndarray
    first: np.ndarray
    nodes: np.ndarray
    status: np.ndarray
    n_sat: int
    n_unsat: int
    n_budget: int
    total_nodes: int
    kernel_ms: float
    launches: int
    h2d_bytes: int
    d2h_bytes: int
    search_kernel_ms: float = 0.0


def _count_result(sols, first, nodes, status, st) -> CountResult:
    return CountResult(sols, first, nodes, status, st.n_sat, st.n_unsat, st.n_budget, st.total_nodes, st.kernel_ms,
                       st.kernel_launches, st.h2d_bytes, st.d2h_bytes, st.search_kernel_ms)


class Model:
    """A compiled model: `dq_compile` of a CSP (CSP::FinalizeModel + Assignment::Reset)."""

    def __init__(self, csp: CSP, desc_keep=None):
        """`desc_keep` = a (dq_model_desc, keepalive) pair from an earlier `csp.desc()`: compile straight from the
        host arrays (what the C++ drop-in header hands to dq_compile) without rebuilding them in Python."""
        desc, keep = desc_keep if desc_keep is not None else csp.desc()
        h = C.c_void_p()
        _check(lib().dq_compile(C.byref(desc), C.byref(h)))
        del keep
        self._h = h
        self.n_vars = len(csp.domains)

    def close(self):
        if self._h:
            lib().dq_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        nv, kd, na, mc = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        _check(lib().dq_model_info(self._h, C.byref(nv), C.byref(kd), C.byref(na), C.byref(mc)))
        return {"n_vars": nv.value, "max_dom": kd.value, "n_arcs": na.value, "model_class": MODEL_CLASS[mc.value]}

    def order(self) -> List[int]:
        o = np.zeros(max(self.n_vars, 1), dtype=np.int32)
        _check(lib().dq_model_order(self._h, o.ctypes.data_as(C.POINTER(C.c_int32))))
        return o[:self.n_vars].tolist()

    def solve_tree(self, mode: str = "first", split_depth: int = 0, part_rank: int = 0, part_count: int = 1,
                   engine: str = "auto", node_budget: int = 0, time_kernels: bool = False) -> TreeResult:
        """time_kernels: DQ_TREE_TIME_KERNELS (search_kernel_ms from CUDA events; the queue is not replayed as a graph)."""
        o = dq_tree_opts(DQ_MODE_COUNT_ALL if mode == "count" else DQ_MODE_FIRST, split_depth, part_rank, part_count,
                         node_budget, ENGINE[engine], 1 if time_kernels else 0)
        r = dq_tree_result()
        first = np.zeros(max(self.n_vars, 1), dtype=np.int32)
        _check(lib().dq_solve_tree(self._h, C.byref(o), C.byref(r), first.ctypes.data_as(C.POINTER(C.c_int32))))
        have = r.first_key != U64_MAX and (self.n_vars == 0 or first[0] != UNASSIGNED)
        return TreeResult(OUTCOME[r.outcome], r.n_solutions, r.n_nodes, first[:self.n_vars].tolist() if have else None,
                          r.first_key, r.n_prefixes, r.split_depth_used, r.kernel_ms,
                          ENGINE_NAME.get(r.engine_used, "?"), r.kernel_launches, r.search_kernel_ms, r.frontier_nodes)

    def solve_tree_multi(self, mode: str = "first", devices=(0,), split_depth: int = 0, engine: str = "auto",
                         time_kernels: bool = False) -> TreeResult:
        """dq_solve_tree_multi: one process, one partition of the prefix-split tree per entry of `devices`."""
        o = dq_tree_opts(DQ_MODE_COUNT_ALL if mode == "count" else DQ_MODE_FIRST, split_depth, 0, 1, 0, ENGINE[engine],
                         1 if time_kernels else 0)
        r = dq_tree_result()
        first = np.zeros(max(self.n_vars, 1), dtype=np.int32)
        devs = np.array(list(devices), dtype=np.int32)
        _check(lib().dq_solve_tree_multi(self._h, C.byref(o), len(devs), devs.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(r),
                                         first.ctypes.data_as(C.POINTER(C.c_int32))))
        have = r.first_key != U64_MAX and (self.n_vars == 0 or first[0] != UNASSIGNED)
        return TreeResult(OUTCOME[r.outcome], r.n_solutions, r.n_nodes, first[:self.n_vars].tolist() if have else None,
                          r.first_key, r.n_prefixes, r.split_depth_used, r.kernel_ms,
                          ENGINE_NAME.get(r.engine_used, "?"), r.kernel_launches, r.search_kernel_ms, r.frontier_nodes)

    def enumerate_solutions(self, cap: int, split_depth: int = 0, part_rank: int = 0, part_count: int = 1,
                            engine: str = "auto"):
        """All solutions in the reference's DFS order -> (int32[n, n_vars], TreeResult).  Raises DequanError
        (DQ_ERR_NOMEM) when there are more than `cap`."""
        o = dq_tree_opts(DQ_MODE_COUNT_ALL, split_depth, part_rank, part_count, 0, ENGINE[engine], 0)
        r = dq_tree_result()
        out = np.zeros((max(cap, 1), max(self.n_vars, 1)), dtype=np.int32)
        n = C.c_uint64()
        _check(lib().dq_enumerate_solutions(self._h, C.byref(o), C.byref(r), out.ctypes.data_as(C.POINTER(C.c_int32)),
                                            cap, C.byref(n)))
        res = TreeResult(OUTCOME[r.outcome], r.n_solutions, r.n_nodes, None, r.first_key, r.n_prefixes, r.split_depth_used,
                         r.kernel_ms, ENGINE_NAME.get(r.engine_used, "?"), r.kernel_launches, r.search_kernel_ms, r.frontier_nodes)
        return out[:n.value, :self.n_vars].copy(), res

    def table_bytes(self) -> int:
        n = C.c_uint64()
        _check(lib().dq_model_table_bytes(self._h, C.byref(n)))
        return n.value

    def nodes_upto(self, key: int) -> int:
        n = C.c_uint64()
        _check(lib().dq_tree_nodes_upto(self._h, key, C.byref(n)))
        return n.value

    def solve_batch_cells(self, cells: np.ndarray, node_budget: int = 0, engine: str = "auto",
                          out: Optional[tuple] = None, task_nodes: int = 0) -> BatchResult:
        """cells: uint8[n, stride] host array (0 = keep template domain)."""
        assert cells.dtype == np.uint8 and cells.ndim == 2 and cells.flags.c_contiguous
        n, stride = cells.shape
        if out is None:
            sol = np.zeros((n, stride), dtype=np.uint8)
            nodes = np.zeros(n, dtype=np.uint64)
            status = np.zeros(n, dtype=np.uint8)
        else:
            sol, nodes, status = out
        o = dq_batch_opts(node_budget, ENGINE[engine], task_nodes)
        st = dq_batch_stats()
        _check(lib().dq_solve_batch_cells(self._h, cells.ctypes.data, n, stride, C.byref(o), sol.ctypes.data,
                                          nodes.ctypes.data, status.ctypes.data, C.byref(st)))
        return BatchResult(sol, nodes, status, st.n_sat, st.n_unsat, st.n_budget, st.total_nodes, st.kernel_ms,
                           st.kernel_launches, st.h2d_bytes, st.d2h_bytes)

    def count_batch_cells(self, cells: np.ndarray, solution_limit: int = 0, node_budget: int = 0,
                          engine: str = "auto") -> CountResult:
        """dq_count_batch_cells: each instance's solutions, up to `solution_limit` (0 = all) and within `node_budget`
        (0 = none).  cells: uint8[n, stride] host array (0 = keep template domain)."""
        assert cells.dtype == np.uint8 and cells.ndim == 2 and cells.flags.c_contiguous
        n, stride = cells.shape
        sols = np.zeros(n, dtype=np.uint64)
        first = np.zeros((n, stride), dtype=np.uint8)
        nodes = np.zeros(n, dtype=np.uint64)
        status = np.zeros(n, dtype=np.uint8)
        o = dq_count_opts(node_budget, solution_limit, ENGINE[engine] if isinstance(engine, str) else int(engine))
        st = dq_batch_stats()
        _check(lib().dq_count_batch_cells(self._h, cells.ctypes.data, n, stride, C.byref(o), sols.ctypes.data,
                                          first.ctypes.data, nodes.ctypes.data, status.ctypes.data, C.byref(st)))
        return _count_result(sols, first, nodes, status, st)

    def solve_batch_cells_ptr(self, cells_ptr: int, n: int, stride: int, sol_ptr: int, nodes_ptr: int, status_ptr: int,
                              node_budget: int = 0, engine: str = "auto", device: bool = False, task_nodes: int = 0):
        """Raw-pointer form (pinned host buffers or, with device=True, HBM-resident buffers)."""
        o = dq_batch_opts(node_budget, ENGINE[engine], task_nodes)
        st = dq_batch_stats()
        fn = lib().dq_solve_batch_cells_dev if device else lib().dq_solve_batch_cells
        _check(fn(self._h, cells_ptr, n, stride, C.byref(o), sol_ptr, nodes_ptr, status_ptr, C.byref(st)))
        return st


@dataclass
class ModelsResult:
    """Per model, in list order, what `Model.solve_tree(mode)` reports: status, solutions, nodes, first."""
    status: List[str]
    solutions: List[int]
    nodes: List[int]
    first: List[Optional[List[int]]]
    n_split: int
    kernel_ms: float
    launches: int


def solve_models(models, mode: str = "first", engine: str = "auto") -> ModelsResult:
    """dq_solve_models: many independent compiled models in one call.  `models` is a sequence of `Model` (the same one
    may appear more than once; None passes a NULL handle)."""
    n = len(models)
    hs = (C.c_void_p * max(n, 1))(*[m._h.value if m is not None and m._h else None for m in models])
    nvs = [m.n_vars if m is not None else 0 for m in models]
    off = np.concatenate([[0], np.cumsum(nvs, dtype=np.int64)])
    outcome = np.zeros(max(n, 1), dtype=np.int32)
    sols = np.zeros(max(n, 1), dtype=np.uint64)
    nodes = np.zeros(max(n, 1), dtype=np.uint64)
    first = np.zeros(max(int(off[-1]), 1), dtype=np.int32)
    n_split = C.c_int64()
    o = dq_tree_opts(DQ_MODE_COUNT_ALL if mode == "count" else DQ_MODE_FIRST, 0, 0, 1, 0, ENGINE[engine], 0)
    st = dq_batch_stats()
    i32 = C.POINTER(C.c_int32)
    _check(lib().dq_solve_models(hs, n, C.byref(o), outcome.ctypes.data_as(i32), sols.ctypes.data, nodes.ctypes.data,
                                 first.ctypes.data_as(i32), C.byref(n_split), C.byref(st)))
    firsts = []
    for i in range(n):
        f = first[off[i]:off[i + 1]].tolist()
        firsts.append(f if sols[i] and (nvs[i] == 0 or f[0] != UNASSIGNED) else None)
    return ModelsResult([OUTCOME[int(x)] for x in outcome[:n]], [int(x) for x in sols[:n]], [int(x) for x in nodes[:n]],
                        firsts, n_split.value, st.kernel_ms, st.kernel_launches)


def solve_batch_graphs(n_vertices: int, k: int, edge_off: np.ndarray, edges: np.ndarray, node_budget: int = 0,
                       engine: str = "auto") -> BatchResult:
    assert edge_off.dtype == np.int64 and edges.dtype == np.uint8
    edges = np.ascontiguousarray(edges)
    n = len(edge_off) - 1
    col = np.zeros((n, n_vertices), dtype=np.uint8)
    nodes = np.zeros(n, dtype=np.uint64)
    status = np.zeros(n, dtype=np.uint8)
    o = dq_batch_opts(node_budget, ENGINE[engine], 0)
    st = dq_batch_stats()
    _check(lib().dq_solve_batch_graphs(n_vertices, k, edge_off.ctypes.data, edges.ctypes.data, n, C.byref(o),
                                       col.ctypes.data, nodes.ctypes.data, status.ctypes.data, C.byref(st)))
    return BatchResult(col, nodes, status, st.n_sat, st.n_unsat, st.n_budget, st.total_nodes, st.kernel_ms,
                       st.kernel_launches, st.h2d_bytes, st.d2h_bytes, st.search_kernel_ms)


def count_batch_graphs(n_vertices: int, k: int, edge_off: np.ndarray, edges: np.ndarray, solution_limit: int = 0,
                       node_budget: int = 0, engine: str = "auto") -> CountResult:
    """dq_count_batch_graphs: each graph's k-colourings, up to `solution_limit` (0 = all) and within `node_budget`
    (0 = none); `first` holds the DFS-first colouring (0xFF where none)."""
    assert edge_off.dtype == np.int64 and edges.dtype == np.uint8
    edges = np.ascontiguousarray(edges)
    n = len(edge_off) - 1
    sols = np.zeros(n, dtype=np.uint64)
    col = np.zeros((n, n_vertices), dtype=np.uint8)
    nodes = np.zeros(n, dtype=np.uint64)
    status = np.zeros(n, dtype=np.uint8)
    o = dq_count_opts(node_budget, solution_limit, ENGINE[engine] if isinstance(engine, str) else int(engine))
    st = dq_batch_stats()
    _check(lib().dq_count_batch_graphs(n_vertices, k, edge_off.ctypes.data, edges.ctypes.data, n, C.byref(o),
                                       sols.ctypes.data, col.ctypes.data, nodes.ctypes.data, status.ctypes.data,
                                       C.byref(st)))
    return _count_result(sols, col, nodes, status, st)


def solve_batch_graphs_ptr(n_vertices: int, k: int, edge_off: np.ndarray, edge_off_dev: int, edges_ptr: int, col_ptr: int,
                           nodes_ptr: int, status_ptr: int, node_budget: int = 0, engine: str = "auto", device: bool = True):
    """Raw-pointer form: device=True -> dq_solve_batch_graphs_dev (HBM-resident edge lists and outputs; `edge_off` is the
    host copy of the offsets), device=False -> dq_solve_batch_graphs on (pinned) host buffers."""
    assert edge_off.dtype == np.int64
    n = len(edge_off) - 1
    o = dq_batch_opts(node_budget, ENGINE[engine], 0)
    st = dq_batch_stats()
    if device:
        _check(lib().dq_solve_batch_graphs_dev(n_vertices, k, edge_off.ctypes.data, edge_off_dev, edges_ptr, n, C.byref(o),
                                               col_ptr, nodes_ptr, status_ptr, C.byref(st)))
    else:
        _check(lib().dq_solve_batch_graphs(n_vertices, k, edge_off.ctypes.data, edges_ptr, n, C.byref(o),
                                           col_ptr, nodes_ptr, status_ptr, C.byref(st)))
    return st


def parse_sudoku_lines(text: str) -> np.ndarray:
    """81-character lines -> uint8[n, 81] (0 = blank), the input layout of `Model.solve_batch_cells`."""
    raw = text.encode()
    cap = raw.count(b"\n") + 1
    cells = np.zeros((cap, 81), dtype=np.uint8)
    n = C.c_int64()
    _check(lib().dq_parse_sudoku_lines(raw, len(raw), cells.ctypes.data, cap, C.byref(n)))
    return np.ascontiguousarray(cells[:n.value])


def parse_dimacs_col(text: str):
    """DIMACS .col -> (n_vertices, uint8[m, 2] edges, 0-based), the per-instance input of `solve_batch_graphs`."""
    raw = text.encode()
    cap = raw.count(b"\ne ") + raw.startswith(b"e ") + 1
    edges = np.zeros((cap, 2), dtype=np.uint8)
    nv, m = C.c_int32(), C.c_int64()
    _check(lib().dq_parse_dimacs_col(raw, len(raw), C.byref(nv), edges.ctypes.data, cap, C.byref(m)))
    return nv.value, np.ascontiguousarray(edges[:m.value])
