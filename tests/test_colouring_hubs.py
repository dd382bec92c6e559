"""Colouring batches on graphs with hub vertices, against the CPU oracle, on every engine.

The lane-per-instance engine (dq_group_graphs.cuh) keeps eight later neighbours of each vertex in its row; a vertex
with more has a marker byte in its last slot and the rest of its neighbours in an overflow list sorted by vertex.  The
marker holds the vertex's start in the list as 255 - min(start, 254 - nv) (a start that does not fit is clamped and
the walk skips forward), the header holds the pair count as a u16, and a lane keeps only the first `over_smem` pairs
in shared memory: the rest are read from the record.  Sparse random graphs numbered in maximum-cardinality order reach
little of this, so the families here are built around hubs (vertices adjacent to a large share of the later ones):

- hubs over a sparse core: G(nv, c/(nv-1)) in maximum-cardinality order, a hub at vertex 0, one at nv/3 (its list
  starts deep, clamped once the lists before it are long) and, in every other instance, a third one before it;
- stars: K_(a, nv-a) with the small side first, a in {1, 2, 4}, some with a few edges or a K_k inside the large side.

Expected answers: oracle_lib.solve(colouring(...), "first", budget), status, node count and colours, bit for bit;
counting batches against dqo_count_limit (test_count_batches.py)."""
import functools

import numpy as np
import pytest

import oracle_lib as O
from dequan_b200 import api
from dequan_b200 import generators as G
from dequan_b200.model import colouring
from test_count_batches import check as check_count, oracle_count

STATUS = {"unsat": 0, "sat": 1, "budget": 2}
SIZES = (40, 120, 200, 230, 250, 254)
DQ_ERR_INVALID = -1
LAUNCHES = {"lane": 3, "reg": 1, "warp": 2, "auto": 1}      # (auto: fewer than 4096 instances go to the register engine)


# ---- the lane engine's layout, restated -------------------------------------------------------------------------------

def lane_share(nv: int, k: int) -> int:
    """Overflow pairs a lane keeps in shared memory when the batch's lists are at least that long: run_graphs_lane in
    dequan_b200/csrc/dq_api.cu (as many as cost no CTA per SM), with graphs_lane_warp_bytes (dq_group_graphs.cuh) for
    the state of one warp.  Up to three colours the PACKED layout, four the K4 layout."""
    nvp = (nv + 16) & ~15
    base = (nv + 1) * 128 + (((nv + 15) // 16) * 128 if k <= 3 else nvp * 64) + 16
    ctas = min(228 * 1024 // (base + 1024), 32)
    return (228 * 1024 // ctas - 1024 - base) // 64


def overflow(nv: int, e: np.ndarray):
    """(pairs in the overflow list, starts of the vertices that have some) of k_graphs_adjacency's record: a vertex with
    more than eight later neighbours keeps seven in its row and the others, the eighth included, go to the list."""
    cnt = np.bincount(np.minimum(e[:, 0], e[:, 1]).astype(np.int64), minlength=nv)
    per = np.where(cnt > 8, cnt - 7, 0)
    start = np.cumsum(per) - per
    return int(per.sum()), start[per > 0]


# ---- families ---------------------------------------------------------------------------------------------------------

CORE_C = {2: (0.0, 0.5), 3: (1.0, 2.5), 4: (2.5, 7.5)}     # average degree of the core: a mix of all three outcomes


def _edge_list(rng, adj: np.ndarray) -> np.ndarray:
    """The edges of a boolean adjacency matrix, in random order, each with its endpoints in random order."""
    u, v = np.nonzero(np.triu(adj | adj.T, 1))
    e = np.stack([u, v], axis=1)
    swap = rng.random(len(e)) < 0.5
    e[swap] = e[swap][:, ::-1]
    return np.ascontiguousarray(e[rng.permutation(len(e))], dtype=np.uint8)


def _hub_graph(rng, nv: int, k: int, i: int) -> np.ndarray:
    adj = np.zeros((nv, nv), dtype=bool)
    iu, ju = np.triu_indices(nv, 1)
    sel = rng.random(iu.size) < rng.uniform(*CORE_C[k]) / (nv - 1)
    if sel.any():
        nid = G.max_cardinality_order(nv, np.stack([iu[sel], ju[sel]], axis=1))
        adj[nid[iu[sel]], nid[ju[sel]]] = True
    for h in [0, nv // 3] + ([int(rng.integers(1, nv // 3))] if i % 2 else []):
        adj[h, h + 1:] |= rng.random(nv - h - 1) < rng.uniform(0.3, 1.0)
    if i % 8 == 6:                                # a K_(k+1) on vertex 0 and k of the ten after it
        q = np.concatenate([[0], 1 + rng.choice(10, size=k, replace=False)])
        adj[np.ix_(q, q)] = True
        adj[q, q] = False
    return adj


def _star(rng, nv: int, k: int, i: int) -> np.ndarray:
    a = (1, 2, 4)[i % 3]
    adj = np.zeros((nv, nv), dtype=bool)
    adj[:a, a:] = True
    variant = (i // 3) % 4
    if variant == 1:                              # a few edges inside the large side
        for _ in range(int(rng.integers(1, 6))):
            u, v = rng.choice(np.arange(a, nv), size=2, replace=False)
            adj[u, v] = True
    elif variant >= 2:                            # a K_k there (k - 1 colours left): first in line, or deep
        q = a + np.arange(k) if variant == 2 else rng.choice(np.arange(nv // 2, nv), size=k, replace=False)
        adj[np.ix_(q, q)] = True
        adj[q, q] = False
    return adj


FAMILIES = [f"hubs-{nv}-{k}" for k in (2, 3, 4) for nv in SIZES] + [f"stars-{nv}-{k}" for k in (3, 4) for nv in SIZES]


@functools.lru_cache(maxsize=None)
def family(name: str):
    """(nv, k, node budget, edge_off, edges): 64 to 100 instances, every eleventh one an empty graph."""
    kind, nv, k = name.split("-")
    nv, k = int(nv), int(k)
    j = FAMILIES.index(name)
    rng = np.random.default_rng([20261022, j])
    count = (77, 64, 100, 96)[j % 4]
    make = _hub_graph if kind == "hubs" else _star
    lists = [_edge_list(rng, make(rng, nv, k, i)) if i % 11 != 5 else np.zeros((0, 2), dtype=np.uint8)
             for i in range(count)]
    off = np.zeros(count + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(e) for e in lists])
    budget = 500 if nv == 40 else 30_000           # (searches on 40 vertices rarely run longer)
    return nv, k, budget, off, np.ascontiguousarray(np.concatenate(lists))


def instances(name: str):
    nv, _, _, off, edges = family(name)
    return [edges[off[i]:off[i + 1]] for i in range(len(off) - 1)]


@functools.lru_cache(maxsize=None)
def expected(name: str):
    """(status, nodes, colours with 0xFF where none) per instance, from the oracle under the family's budget."""
    nv, k, budget, _, _ = family(name)
    outs = [O.solve(colouring(nv, k, e), "first", budget) for e in instances(name)]
    col = np.full((len(outs), nv), 0xFF, dtype=np.uint8)
    for i, o in enumerate(outs):
        if o.first is not None:
            col[i] = o.first
    return (np.array([STATUS[o.status] for o in outs], dtype=np.uint8), np.array([o.nodes for o in outs], dtype=np.uint64),
            col)


# ---- CPU: what the families reach --------------------------------------------------------------------------------------

def test_families_reach_the_overflow_paths():
    """In both layouts, from the edge lists alone: instances with more overflow pairs than a lane's shared-memory share
    (the rest read from the record), lists longer than 255 pairs (the header's high byte), clamped starts where
    254 - nv > 0 (the walk skips forward); and a count that is not a multiple of 32."""
    reach = {layout: {"beyond_share": 0, "over_255": 0, "clamped": 0} for layout in ("packed", "k4")}
    counts = set()
    for name in FAMILIES:
        nv, k, _, off, _ = family(name)
        counts.add(len(off) - 1)
        r = reach["packed" if k <= 3 else "k4"]
        share = lane_share(nv, k)
        for e in instances(name):
            assert len(e) == 0 or (int(e.max()) < nv and (e[:, 0] != e[:, 1]).all()), name
            pairs, starts = overflow(nv, e)
            r["beyond_share"] += pairs > share
            r["over_255"] += pairs > 255
            r["clamped"] += int((starts > 254 - nv).sum()) if nv < 254 else 0
    for layout, r in reach.items():
        assert all(v >= 4 for v in r.values()), (layout, r)
    assert any(c % 32 for c in counts)


def test_lane_share_matches_the_layout_table():
    """The restatement above at the sizes the families use (PACKED / K4 pairs per lane)."""
    assert [lane_share(nv, 3) for nv in SIZES] == [9, 6, 11, 12, 57, 49]
    assert [lane_share(nv, 4) for nv in SIZES] == [5, 19, 103, 11, 137, 129]


def test_families_are_not_vacuous():
    """(CPU) Every family ends with satisfiable, unsatisfiable and budget-bound instances under its budget."""
    for name in FAMILIES:
        st = expected(name)[0]
        assert all((st == s).sum() >= 2 for s in STATUS.values()), (name, np.bincount(st, minlength=3).tolist())


def test_graph_entry_points_refuse_more_than_254_vertices(product_lib):
    """Vertex ids are bytes and 255 marks the padding: 255 and 256 vertices are refused before any device work."""
    L = api.lib()
    off = np.array([0, 1], dtype=np.int64)
    edges = np.array([[0, 1]], dtype=np.uint8)
    col, nodes, status = np.zeros(256, dtype=np.uint8), np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint8)
    outs = (col.ctypes.data, nodes.ctypes.data, status.ctypes.data)
    for nv in (0, 255, 256):
        assert L.dq_solve_batch_graphs(nv, 3, off.ctypes.data, edges.ctypes.data, 1, None, *outs, None) == DQ_ERR_INVALID, nv
        # (the host buffers stand in for device ones: the size is checked before any of them is used)
        assert L.dq_solve_batch_graphs_dev(nv, 3, off.ctypes.data, off.ctypes.data, edges.ctypes.data, 1, None, *outs,
                                           None) == DQ_ERR_INVALID, nv
        assert "bad argument" in L.dq_last_error().decode()


# ---- GPU: every engine against the oracle ------------------------------------------------------------------------------

def _check(r, want, what):
    st, nodes, col = want
    bad = np.nonzero((r.status != st) | (r.nodes != nodes) | (r.solution != col).any(axis=1))[0]
    assert len(bad) == 0, (what, f"{len(bad)} of {len(st)} differ",
                           [(int(i), int(r.status[i]), int(st[i]), int(r.nodes[i]), int(nodes[i])) for i in bad[:5]])
    assert (r.n_sat, r.n_unsat, r.n_budget) == (int((st == 1).sum()), int((st == 0).sum()), int((st == 2).sum())), what
    assert r.total_nodes == int(nodes.sum()), what


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAMILIES)
def test_engines_vs_oracle(product_lib, name):
    nv, k, budget, off, edges = family(name)
    want = expected(name)
    for engine, launches in LAUNCHES.items():
        r = api.solve_batch_graphs(nv, k, off, edges, node_budget=budget, engine=engine)
        _check(r, want, (name, engine))
        assert r.launches == launches, (name, engine)
    # budgets on the boundary, one instance at a time: solved with B = nodes, BUDGET at exactly B + 1 with B = nodes - 1;
    # instances with the longest lists first (the record path of a lane)
    st, nodes, col = want
    lists = instances(name)
    solved = [i for i in np.nonzero(st != 2)[0] if nodes[i] > 1]
    for i in sorted(solved, key=lambda i: -overflow(nv, lists[i])[0])[:3]:
        one = (np.array([0, len(lists[i])], dtype=np.int64), lists[i])
        need = int(nodes[i])
        for engine in LAUNCHES:
            a = api.solve_batch_graphs(nv, k, *one, node_budget=need, engine=engine)
            assert (int(a.status[0]), int(a.nodes[0]), a.solution[0].tobytes()) == (int(st[i]), need, col[i].tobytes()), \
                (name, engine, int(i))
            b = api.solve_batch_graphs(nv, k, *one, node_budget=need - 1, engine=engine)
            assert (int(b.status[0]), int(b.nodes[0])) == (2, need) and (b.solution[0] == 0xFF).all(), (name, engine, int(i))


# ---- GPU: AUTO falls back to the register engine when the lane state does not fit --------------------------------------

@pytest.mark.gpu
def test_auto_falls_back_on_a_dense_instance(product_lib):
    """4 096 instances (enough for AUTO to try the lane engine): 4 095 sparse graphs and K_254, whose edge list does not
    fit the lane engine's shared memory.  AUTO serves the batch with the register engine; the lane engine, asked by
    name or through the device-buffer entry point (which has no engine that trusts the lists), refuses it."""
    import torch
    nv, k, n, dense = 254, 3, 4096, 2741
    off_s, edges_s = G.colouring_batch(n - 1, nv, 2.0, seed=77)
    iu, ju = np.triu_indices(nv, 1)
    full = np.stack([iu, ju], axis=1).astype(np.uint8)
    lists = [edges_s[off_s[i]:off_s[i + 1]] for i in range(n - 1)]
    lists.insert(dense, full)
    off = np.zeros(n + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(e) for e in lists])
    edges = np.ascontiguousarray(np.concatenate(lists))
    a = api.solve_batch_graphs(nv, k, off, edges, node_budget=30_000)
    assert a.launches == 1
    w = api.solve_batch_graphs(nv, k, off, edges, node_budget=30_000, engine="warp")
    assert w.launches == 2
    assert (a.status == w.status).all() and (a.nodes == w.nodes).all() and (a.solution == w.solution).all()
    assert (a.n_sat, a.n_unsat, a.n_budget, a.total_nodes) == (w.n_sat, w.n_unsat, w.n_budget, w.total_nodes)
    o = O.solve(colouring(nv, k, full), "first", 30_000)
    assert (int(a.status[dense]), int(a.nodes[dense])) == (STATUS[o.status], o.nodes) and o.status == "unsat"
    assert (a.solution[dense] == 0xFF).all()
    with pytest.raises(api.DequanError):
        api.solve_batch_graphs(nv, k, off, edges, node_budget=30_000, engine="lane")
    dev = torch.device("cuda", 0)
    flat = edges.reshape(-1)
    d_edges = torch.from_numpy(np.concatenate([flat, np.zeros((-flat.size) % 16, dtype=np.uint8)])).to(dev)
    d_off = torch.from_numpy(off).to(dev)
    d_col = torch.zeros((n, nv), dtype=torch.uint8, device=dev)
    d_nodes = torch.zeros(n, dtype=torch.int64, device=dev)
    d_status = torch.zeros(n, dtype=torch.uint8, device=dev)
    with pytest.raises(api.DequanError):
        api.solve_batch_graphs_ptr(nv, k, off, d_off.data_ptr(), d_edges.data_ptr(), d_col.data_ptr(), d_nodes.data_ptr(),
                                   d_status.data_ptr(), node_budget=30_000, device=True)
    torch.cuda.synchronize()


# ---- GPU: counting on the hub families ---------------------------------------------------------------------------------

COUNT_FAMILIES = ["hubs-200-2", "hubs-230-3", "hubs-120-4"]


@functools.lru_cache(maxsize=None)
def count_expected(name: str, limit: int):
    nv, k, budget, _, _ = family(name)
    outs = [oracle_count(colouring(nv, k, e), limit, budget) for e in instances(name)]
    first = np.full((len(outs), nv), 0xFF, dtype=np.uint8)
    for i, o in enumerate(outs):
        if o[3] is not None:
            first[i] = o[3]
    return (np.array([STATUS[o[0]] for o in outs], dtype=np.uint8), np.array([o[1] for o in outs], dtype=np.uint64),
            np.array([o[2] for o in outs], dtype=np.uint64), first)


@pytest.mark.gpu
@pytest.mark.parametrize("name", COUNT_FAMILIES)
def test_count_hub_families(product_lib, name):
    nv, k, budget, off, edges = family(name)
    for limit in (0, 2):
        r = api.count_batch_graphs(nv, k, off, edges, solution_limit=limit, node_budget=budget)
        assert r.launches == 2
        check_count(r, count_expected(name, limit), (name, limit))
