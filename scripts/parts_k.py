"""N-Queens: per-partition kernel time by split depth, partitions emulated one after the other on one GPU.
usage: parts_k.py [n] [worlds,..] [ks,..]"""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dequan_b200 import api
from dequan_b200.model import nqueens
n = int(sys.argv[1]) if len(sys.argv) > 1 else 17
worlds = tuple(int(x) for x in sys.argv[2].split(",")) if len(sys.argv) > 2 else (1, 8)
ks = tuple(int(x) for x in sys.argv[3].split(",")) if len(sys.argv) > 3 else (7, 8, 9)
m = api.Model(nqueens(n))
for k in ks:
    for world in worlds:
        tot_s = tot_n = 0; times = []; srch = []
        for r in range(world):
            m.solve_tree("count", part_rank=r, part_count=world, split_depth=k)
            x = m.solve_tree("count", part_rank=r, part_count=world, split_depth=k, time_kernels=True)
            tot_s += x.solutions; tot_n += x.nodes; times.append(x.kernel_ms); srch.append(x.search_kernel_ms)
        print(f"K={k} used={x.split_depth} parts={world} sols={tot_s} nodes={tot_n} max_ms={max(times):.3f} mean_ms={sum(times)/world:.3f} "
              f"search_max={max(srch):.3f} search_mean={sum(srch)/world:.3f} records={x.n_prefixes}", flush=True)
