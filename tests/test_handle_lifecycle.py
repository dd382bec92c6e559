"""GPU: a closed handle gives back every device block it held.  Blocks go back to the library's block cache and the next
handle takes them from there, so repeating compile -> solve -> close on one entry point reaches a steady state in which
the device's free memory no longer changes.  A block that a handle keeps after dq_free is allocated anew in every round;
the driver hands out memory in 2 MiB pages, so a handle with small tables needs tens of rounds before its leak shows."""
import pytest

from dequan_b200 import api
from dequan_b200 import generators as G
from dequan_b200.model import nqueens, sudoku_template

pytestmark = pytest.mark.gpu

WARMUP_ROUNDS, ROUNDS = 3, 100


def _queens_count():
    m = api.Model(nqueens(12))
    # call by call, then captured as a CUDA graph, then replayed: close() also destroys the graph
    out = [(r.solutions, r.nodes) for r in (m.solve_tree("count") for _ in range(3))]
    m.close()
    return out


def _queens_first():
    m = api.Model(nqueens(12))
    out = m.solve_tree("first").first
    m.close()
    return out


def _generic():
    # head slab, frontier levels, subtree search, enumeration, and the node count up to the first solution
    m = api.Model(nqueens(8))
    sols, r = m.enumerate_solutions(92)
    f = m.solve_tree("first", split_depth=2)
    m.close()
    return r.solutions, r.nodes, sols.tobytes(), f.nodes, f.first


def _sudoku(cells):
    m = api.Model(sudoku_template())
    r = m.solve_batch_cells(cells)
    m.close()
    return r.total_nodes, r.solution.tobytes(), r.status.tobytes()


def _colouring(graphs):
    # no handle: the batch owns its buffers for the duration of the call
    return [(r.total_nodes, r.solution.tobytes())
            for r in (api.solve_batch_graphs(30, 3, *graphs, node_budget=20_000, engine=e) for e in ("lane", "reg", "warp"))]


def test_closed_handles_give_back_every_block(product_lib):
    import torch
    cells = G.sudoku_batch(512, givens=30, seed=5)
    cells[0, 0], cells[0, 1] = 5, 5                       # clashing givens: the generic batch engine after the lane pipeline
    graphs = G.colouring_batch(4096, 30, 3.0, seed=9)
    # one entry point at a time: rounds that mix them settle only after several rounds, as the cache's best fit sorts out
    # which block serves which request
    for name, solve in [("queens count", _queens_count), ("queens first", _queens_first), ("generic tree", _generic),
                        ("sudoku batch", lambda: _sudoku(cells)), ("colouring batches", lambda: _colouring(graphs))]:
        want = solve()
        for _ in range(WARMUP_ROUNDS - 1):
            assert solve() == want, name
        free = torch.cuda.mem_get_info(0)[0]
        for _ in range(ROUNDS):
            assert solve() == want, name
        assert torch.cuda.mem_get_info(0)[0] == free, f"{name}: device memory not given back"
