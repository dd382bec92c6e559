// dq_kernels.cuh — kernels around the generic warp engine: frontier (prefix) expansion,
// the persistent subtree DFS, and the batched-instance kernels.
#pragma once
#include "dq_warp_engine.cuh"

namespace dq {

constexpr int kWarpsPerCta = 4;
constexpr unsigned long long KEY_NONE = 0xFFFFFFFFFFFFFFFFull;

template <typename W>
struct TreeModelDevT {
    DevTablesT<W> T;
    const W* __restrict__ dom0;          // [nv] by var id
    const uint16_t* __restrict__ order;  // [nv]
    const uint16_t* __restrict__ pos;    // [nv]
    int trail;                           // trail capacity per warp
    // the state k_expand_head left at the end of the forced chain (domains / fails-validation words by var id): prefixes
    // are replayed from there instead of from the root.  base_depth == 0: no chain.
    const W* base_D = nullptr;
    const W* base_F = nullptr;
    int base_depth = 0;
};
typedef TreeModelDevT<uint32_t> TreeModelDev;

template <typename W>
__device__ __forceinline__ void load_root_state(const TreeModelDevT<W>& M, const WarpStateT<W>& S, int lane) {
    for (int v = lane; v < M.T.nv; v += 32) {
        S.D[v] = M.base_depth ? __ldg(M.base_D + v) : __ldg(M.dom0 + v);
        S.F[v] = M.base_depth ? __ldg(M.base_F + v) : W(0);
        S.order[v] = __ldg(M.order + v);
        S.pos[v] = __ldg(M.pos + v);
    }
    __syncwarp();
}

// Re-apply a prefix (value indices for depths 0..depth-1) to the root state.
// (COHERENT: the prefix was written by this very launch — k_expand_head — so no read-only cache path)
template <bool HAS_F, bool HAS_TABLE, typename W, bool COHERENT = false>
__device__ __forceinline__ void replay_prefix(const TreeModelDevT<W>& M, const WarpStateT<W>& S, const uint8_t* __restrict__ prefix,
                                              int depth, int lane) {
    load_root_state(M, S, lane);
    int top = 0;
    for (int i = 0; i < depth; i++) {
        const int b = COHERENT ? (int)*(const volatile uint8_t*)(prefix + i) : (int)__ldg(prefix + i);
        if (lane == 0) S.val[i] = (uint8_t)b;
        if (i < M.base_depth) continue;               // (the forced chain is already in the base state)
        fc_apply<HAS_F, HAS_TABLE>(M.T, S, S.order[i], b, i, top, lane);
        top = 0;                                      // nothing above the split depth is ever undone
    }
    __syncwarp();
}

// ---- frontier expansion, one level: warp per parent state --------------------------------------
// dmask[i] = current domain of the next variable (each bit is one node, dequan.h:416-423)
// surv[i]  = values whose validation and forward check succeed (children states)
template <bool HAS_F, bool HAS_TABLE, typename W = uint32_t>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_expand(TreeModelDevT<W> M, const uint8_t* __restrict__ prefixes, int depth, int n_states,
         W* __restrict__ dmask, W* __restrict__ surv) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int i = blockIdx.x * (blockDim.x >> 5) + wib;       // (large models run fewer warps per CTA)
    if (i >= n_states) return;
    WarpStateT<W> S = carve_warp_state_t<W>(smem + (size_t)wib * warp_state_bytes(M.T.nv, M.trail, sizeof(W)), M.T.nv, M.trail);
    replay_prefix<HAS_F, HAS_TABLE>(M, S, prefixes + (size_t)i * depth, depth, lane);
    const int x = S.order[depth];
    const W dm = S.D[x];
    W c = HAS_F ? (dm & ~S.F[x]) : dm, sv = 0;
    while (c) {
        const int b = dq_ffs(c) - 1;
        c &= c - 1;
        int top = 0;
        const bool wiped = fc_apply<HAS_F, HAS_TABLE>(M.T, S, x, b, depth, top, lane);
        trail_undo<HAS_F>(S, 0, top, lane);
        if (!wiped) sv |= W(1) << b;
    }
    if (lane == 0) { dmask[i] = dm; surv[i] = sv; }
}

// Single-CTA exclusive scans of popc(surv) -> child_off and popc(dmask) -> node_off; totals in tot[0..1].
template <typename W>
__global__ void __launch_bounds__(1024)
k_scan_level(const W* __restrict__ dmask, const W* __restrict__ surv, int n,
             uint32_t* __restrict__ child_off, unsigned long long* __restrict__ node_off,
             unsigned long long* __restrict__ tot) {
    __shared__ unsigned long long wsum_c[32], wsum_n[32];
    __shared__ unsigned long long carry_c, carry_n;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) { carry_c = 0; carry_n = 0; }
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        unsigned long long c = i < n ? dq_popc(surv[i]) : 0, nd = i < n ? dq_popc(dmask[i]) : 0;
        unsigned long long ic = c, in = nd;
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long tc = __shfl_up_sync(FULL, ic, o), tn = __shfl_up_sync(FULL, in, o);
            if (lane >= o) { ic += tc; in += tn; }
        }
        if (lane == 31) { wsum_c[w] = ic; wsum_n[w] = in; }
        __syncthreads();
        if (w == 0) {
            unsigned long long sc = wsum_c[lane], sn = wsum_n[lane];
            for (int o = 1; o < 32; o <<= 1) {
                unsigned long long tc = __shfl_up_sync(FULL, sc, o), tn = __shfl_up_sync(FULL, sn, o);
                if (lane >= o) { sc += tc; sn += tn; }
            }
            wsum_c[lane] = sc; wsum_n[lane] = sn;
        }
        __syncthreads();
        const unsigned long long pc = carry_c + (w ? wsum_c[w - 1] : 0), pn = carry_n + (w ? wsum_n[w - 1] : 0);
        if (i < n) { child_off[i] = (uint32_t)(pc + ic - c); node_off[i] = pn + in - nd; }
        __syncthreads();
        if (threadIdx.x == 1023) { carry_c = pc + ic; carry_n = pn + in; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { tot[0] = carry_c; tot[1] = carry_n; }
}

// Children prefixes in DFS (lexicographic) order: thread per parent.
template <typename W>
__global__ void k_write_children(const uint8_t* __restrict__ prefixes, int depth, int n_states,
                                 const W* __restrict__ surv, const uint32_t* __restrict__ child_off,
                                 uint8_t* __restrict__ out, uint32_t* __restrict__ parent_of) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_states) return;
    W sv = surv[i];
    size_t o = child_off[i];
    while (sv) {
        const int b = dq_ffs(sv) - 1;
        sv &= sv - 1;
        uint8_t* dst = out + o * (size_t)(depth + 1);
        for (int j = 0; j < depth; j++) dst[j] = prefixes[(size_t)i * depth + j];
        dst[depth] = (uint8_t)b;
        parent_of[o] = (uint32_t)i;
        ++o;
    }
}

// ---- the forced head of the tree in ONE launch -------------------------------------------------------------------
// Givens and other singleton domains at the head of the static order (Assignment::Reset puts them first, dequan.h:384-394),
// and every level where forward checking leaves a single passing value, keep the frontier at ONE prefix — often for
// dozens of levels (the reference's SudokuTest: 32 givens) — and each such level is a microsecond of work behind three
// launches and a host round trip.  One warp walks that chain: per level exactly what k_expand / k_scan_level /
// k_write_children produce (domain mask, surviving values, offsets, the child prefix, its parent), with the state
// carried along instead of replayed, until a level has no child or more than one; the host carries on from there.
template <typename W>
struct HeadLevel {
    uint8_t* prefixes;                 // [1][level]
    W* dmask;                          // [1]
    W* surv;                           // [1]
    uint32_t* child_off;               // [1]
    unsigned long long* node_off;      // [1]
    uint32_t* parent_of;               // [1] index into the previous level
};
// out[0] = levels completed (the frontier at that depth is materialised), out[1] = nodes of those levels,
// out[2] = 1 if the frontier died out, out[4 + l] = frontier size at depth l
template <bool HAS_F, bool HAS_TABLE, typename W = uint32_t>
__global__ void __launch_bounds__(32)
k_expand_head(TreeModelDevT<W> M, const HeadLevel<W>* __restrict__ lv, int max_levels, W* __restrict__ base_D, W* __restrict__ base_F,
              unsigned long long* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x;
    WarpStateT<W> S = carve_warp_state_t<W>(smem, M.T.nv, M.trail);
    load_root_state(M, S, lane);
    int done = 0, top = 0;
    unsigned long long nodes = 0;
    bool died = false;
    if (lane == 0) out[4] = 1;
    for (int l = 0; l < max_levels; l++) {
        const HeadLevel<W> L = lv[l];
        const int x = S.order[l];
        const W dm = S.D[x];
        W c = HAS_F ? (dm & ~S.F[x]) : dm, sv = 0;
        while (c) {
            const int b = dq_ffs(c) - 1;
            c &= c - 1;
            const bool wiped = fc_apply<HAS_F, HAS_TABLE>(M.T, S, x, b, l, top, lane);
            trail_undo<HAS_F>(S, 0, top, lane);
            if (!wiped) sv |= W(1) << b;
        }
        const int kids = dq_popc(sv);
        if (kids > 1) break;                                         // the tree fans out: this level is the host's
        if (lane == 0) { L.dmask[0] = dm; L.surv[0] = sv; L.child_off[0] = 0; L.node_off[0] = 0; out[4 + l + 1] = (unsigned long long)kids; }
        nodes += dq_popc(dm);
        done = l + 1;
        if (kids == 0) { died = true; break; }
        const int b = dq_ffs(sv) - 1;
        if (lane == 0) S.val[l] = (uint8_t)b;
        __syncwarp();
        const HeadLevel<W> C = lv[l + 1];
        for (int j = lane; j <= l; j += 32) C.prefixes[j] = S.val[j];
        if (lane == 0) C.parent_of[0] = 0;
        fc_apply<HAS_F, HAS_TABLE>(M.T, S, x, b, l, top, lane);      // for good: nothing above the split is ever undone
        top = 0;
    }
    __syncwarp();
    for (int v = lane; v < M.T.nv; v += 32) { base_D[v] = S.D[v]; base_F[v] = S.F[v]; }      // the state after `done` levels
    if (lane == 0) { out[0] = (unsigned long long)done; out[1] = nodes; out[2] = died ? 1ull : 0ull; }
}

// ---- persistent subtree DFS: warps pull prefix indices from an atomic cursor -------------------
struct TreeDfsArgs {
    const uint8_t* prefixes;            // [n_prefix][depth]
    int depth;
    unsigned long long n_prefix;
    int part_rank, part_count;
    int count_all;
    unsigned long long* cursor;         // work counter
    unsigned long long* totals;         // [0]=solutions [1]=nodes   (COUNT_ALL)
    unsigned long long* best_key;       // lowest prefix index holding a solution
    unsigned long long* sub_nodes;      // [n_prefix] nodes per subtree (this partition's)
    unsigned long long* sol_key;        // [n_warps] key of the solution each warp recorded
    uint8_t* sol;                       // [n_warps][nv] value index per var id
    unsigned long long node_budget;     // root probe only: give up past this many nodes (0 = none) ...
    unsigned long long* gave_up;        // ... and say so here
    // dq_enumerate_solutions (COUNT_ALL): every solution is appended here, tagged with its place in the DFS order
    uint8_t* enum_out;                  // [enum_cap][nv] value index per var id (null: not enumerating)
    unsigned long long* enum_prefix;    // [enum_cap] prefix index of the subtree that holds the solution
    unsigned long long* enum_seq;       // [enum_cap] rank of the solution inside that subtree
    unsigned long long* enum_count;     // solutions appended (may exceed enum_cap: the host reports the overflow)
    unsigned long long enum_cap;
};

// Append the solutions formed by the current assignment of depths 0..nv-2 (value index per depth in `val`, depth ->
// var id in `order`) and each value of `valid` for the last variable; the first one has rank `seq` in its subtree.
template <class ValT, class OrdT, typename W>
__device__ __forceinline__ void enum_append(const TreeDfsArgs& A, unsigned long long prefix_idx, int nv, const ValT* val,
                                            const OrdT* order, W valid, unsigned long long seq, int lane) {
    while (valid) {
        const int b = dq_ffs(valid) - 1;
        valid &= valid - 1;
        unsigned long long slot = 0;
        if (lane == 0) slot = atomicAdd(A.enum_count, 1ull);
        slot = __shfl_sync(FULL, slot, 0);
        if (slot < A.enum_cap) {
            uint8_t* dst = A.enum_out + slot * (size_t)nv;
            for (int i = lane; i < nv - 1; i += 32) dst[order[i]] = (uint8_t)val[i];
            if (lane == 0) { dst[order[nv - 1]] = (uint8_t)b; A.enum_prefix[slot] = prefix_idx; A.enum_seq[slot] = seq; }
        }
        ++seq;
    }
}

struct RecordFirst {
    const TreeDfsArgs& A;
    unsigned long long key;
    int gw, nv, lane;
    template <typename W>
    __device__ void operator()(const WarpStateT<W>& S) const {
        unsigned long long old = 0;
        if (lane == 0) old = atomicMin(A.best_key, key);
        old = __shfl_sync(FULL, old, 0);
        if (key < old) {
            for (int i = lane; i < nv; i += 32) A.sol[(size_t)gw * nv + S.order[i]] = S.val[i];
            if (lane == 0) A.sol_key[gw] = key;
        }
    }
    // COUNT_ALL, last variable: `valid` are its solution values (warp_dfs calls this for every such node)
    template <typename W>
    __device__ void solutions(const WarpStateT<W>& S, W valid, unsigned long long seq) const {
        if (A.enum_out) enum_append(A, key, nv, S.val, S.order, valid, seq, lane);
    }
};

template <bool HAS_F, bool HAS_TABLE, typename W = uint32_t>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_tree_dfs(TreeModelDevT<W> M, TreeDfsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int gw = blockIdx.x * (blockDim.x >> 5) + wib;
    const int nv = M.T.nv;
    WarpStateT<W> S = carve_warp_state_t<W>(smem + (size_t)wib * warp_state_bytes(nv, M.trail, sizeof(W)), nv, M.trail);
    unsigned long long acc_nodes = 0, acc_sols = 0;
    for (;;) {
        unsigned long long j = 0;
        if (lane == 0) j = atomicAdd(A.cursor, 1ull);
        j = __shfl_sync(FULL, j, 0);
        const unsigned long long idx = j * (unsigned long long)A.part_count + (unsigned long long)A.part_rank;
        if (idx >= A.n_prefix) break;
        if (!A.count_all && *(volatile unsigned long long*)A.best_key < idx) break;   // later prefixes cannot win
        replay_prefix<HAS_F, HAS_TABLE>(M, S, A.prefixes + idx * (size_t)A.depth, A.depth, lane);
        RecordFirst rec{A, idx, gw, nv, lane};
        DfsResult R = warp_dfs<HAS_F, HAS_TABLE>(M.T, S, A.depth, A.count_all != 0, A.node_budget,
                                                 A.count_all ? nullptr : A.best_key, idx, lane, rec);
        if (R.outcome == 3) continue;                                                 // overtaken by an earlier prefix
        if (R.outcome == 2) { if (lane == 0) *A.gave_up = 1ull; break; }              // root probe over budget: the host runs the split search
        if (lane == 0) A.sub_nodes[idx] = R.nodes;
        if (A.count_all) { acc_nodes += R.nodes; acc_sols += R.sols; }
        else if (R.have_first) rec(S);
    }
    if (A.count_all && lane == 0) {
        atomicAdd(A.totals + 0, acc_sols);
        atomicAdd(A.totals + 1, acc_nodes);
    }
}

// ---- batch: one template graph, per-instance initial domains ("cells") -------------------------
struct BatchCellsArgs {
    const uint8_t* cells;       // [n][stride]
    long long n;
    int stride;
    const uint8_t* cell_lut;    // [nv][256] byte -> value index (0xFF = not in the template domain)
    const int32_t* values;      // [nv][32] value index -> value
    const int32_t* sizes;       // distinct domain sizes after overrides, ascending
    int n_sizes;
    int caller_order;           // the template's assign_order came from the caller: every instance searches in it
    unsigned long long budget;
    unsigned long long* cursor;
    uint8_t* solution;          // [n][stride]
    unsigned long long* nodes;  // [n]
    uint8_t* status;            // [n]
    unsigned long long* totals; // [0]=sat [1]=unsat [2]=budget [3]=nodes
    const int* idx_list;        // optional: the n instance ids to solve (null = 0..n-1)
    // counting batches (k_count_batch_cells) only
    unsigned long long limit = 0;               // solution limit per instance (0 = every solution)
    unsigned long long* n_solutions = nullptr;  // [n]
};

struct NoFirst {
    __device__ void operator()(const WarpState&) const {}
    __device__ void solutions(const WarpState&, uint32_t, unsigned long long) const {}
};

// Counting batches: the DFS-first solution goes to the instance's output row when it is found (the count searches on
// and changes val[]), as bytes: values[v][index] for cell batches, the value index itself (the colour) when values is
// null.
struct FirstBytes {
    uint8_t* out;
    const int32_t* values;
    int nv, lane;
    __device__ void operator()(const WarpState& S) const {
        for (int i = lane; i < nv; i += 32) {
            const int v = S.order[i], b = S.val[i];
            out[v] = values ? (uint8_t)__ldg(values + v * 32 + b) : (uint8_t)b;
        }
    }
    __device__ void solutions(const WarpState&, uint32_t, unsigned long long) const {}
};

// One warp per instance, in turn.  COUNT: count its solutions up to A.limit (warp_dfs's LIMITED path) and write the
// DFS-first one; else its FIRST-mode solve.  (The kernels pass in their shared memory and lane: so the FIRST-mode
// kernels compile to the same code as when this body was theirs.)
template <bool HAS_F, bool HAS_TABLE, bool COUNT>
__device__ __forceinline__ void batch_cells(TreeModelDev M, BatchCellsArgs A, unsigned char* smem, int lane, int wib) {
    const int nv = M.T.nv;
    const uint32_t lt = (1u << lane) - 1u;
    WarpState S = carve_warp_state(smem + (size_t)wib * warp_state_bytes(nv, M.trail), nv, M.trail);
    unsigned long long t_sat = 0, t_unsat = 0, t_budget = 0, t_nodes = 0;
    for (;;) {
        long long i = 0;
        if (lane == 0) i = (long long)atomicAdd(A.cursor, 1ull);
        i = __shfl_sync(FULL, i, 0);
        if (i >= A.n) break;
        if (A.idx_list) i = A.idx_list[i];
        const uint8_t* cell = A.cells + (size_t)i * A.stride;
        // initial domains: template domain, or the singleton of the given (AddFixedVar, dequan.h:467-471)
        bool bad = false;
        for (int v = lane; v < nv; v += 32) {
            const uint32_t c = cell[v];
            uint32_t dm = __ldg(M.dom0 + v);
            if (c) {
                const uint32_t bi = __ldg(A.cell_lut + v * 256 + c);
                if (bi == 0xFF) bad = true; else dm = 1u << bi;
            }
            S.D[v] = dm;
            S.F[v] = 0;
        }
        bad = __any_sync(FULL, bad);
        __syncwarp();
        if (A.caller_order) {
            // a caller-supplied assign_order replaces Reset's sort (dequan.h:316), givens or not
            for (int v = lane; v < nv; v += 32) { S.order[v] = __ldg(M.order + v); S.pos[v] = __ldg(M.pos + v); }
        } else {
            // static order for THIS instance: (domain size asc, id asc) — Assignment::Reset, dequan.h:384-394
            int base = 0;
            for (int s = 0; s < A.n_sizes; s++) {
                const int sz = __ldg(A.sizes + s);
                for (int v0 = 0; v0 < nv; v0 += 32) {
                    const int v = v0 + lane;
                    const bool hit = v < nv && __popc(S.D[v]) == sz;
                    const uint32_t m = __ballot_sync(FULL, hit);
                    if (hit) { const int p = base + __popc(m & lt); S.order[p] = (uint16_t)v; S.pos[v] = (uint16_t)p; }
                    base += __popc(m);
                }
            }
        }
        __syncwarp();
        DfsResult R;
        if (bad) { R.nodes = 0; R.sols = 0; R.outcome = 0; R.have_first = false; }
        else if constexpr (COUNT)
            R = warp_dfs<HAS_F, HAS_TABLE, true>(M.T, S, 0, true, A.budget, nullptr, 0ull, lane,
                                                 FirstBytes{A.solution + (size_t)i * A.stride, A.values, nv, lane}, A.limit);
        else R = warp_dfs<HAS_F, HAS_TABLE>(M.T, S, 0, false, A.budget, nullptr, 0ull, lane, NoFirst());
        uint8_t* out = A.solution + (size_t)i * A.stride;
        if constexpr (COUNT) {
            if (!R.sols) for (int v = lane; v < nv; v += 32) out[v] = 0;
            if (lane == 0) A.n_solutions[i] = R.sols;
        } else {
            for (int v = lane; v < nv; v += 32)
                out[v] = R.outcome == 1 ? (uint8_t)__ldg(A.values + v * 32 + S.val[S.pos[v]]) : (uint8_t)0;
        }
        if (lane == 0) { A.nodes[i] = R.nodes; A.status[i] = bad ? (uint8_t)3 : (uint8_t)R.outcome; }
        t_nodes += R.nodes;
        t_sat += R.outcome == 1; t_unsat += R.outcome == 0; t_budget += R.outcome == 2;
        __syncwarp();
    }
    if (lane == 0) {
        atomicAdd(A.totals + 0, t_sat); atomicAdd(A.totals + 1, t_unsat);
        atomicAdd(A.totals + 2, t_budget); atomicAdd(A.totals + 3, t_nodes);
    }
}

template <bool HAS_F, bool HAS_TABLE>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_batch_cells(TreeModelDev M, BatchCellsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    batch_cells<HAS_F, HAS_TABLE, false>(M, A, smem, threadIdx.x & 31, threadIdx.x >> 5);
}

template <bool HAS_F, bool HAS_TABLE>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_count_batch_cells(TreeModelDev M, BatchCellsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    batch_cells<HAS_F, HAS_TABLE, true>(M, A, smem, threadIdx.x & 31, threadIdx.x >> 5);
}

// ---- batch: one graph per instance (k-colouring) ------------------------------------------------
// Pass 1 builds each instance's entry table in HBM (CSR adjacency in var-id space, both directions);
// pass 2 runs the generic engine with per-instance tables.
struct BatchGraphsArgs {
    int nv, k;
    const long long* edge_off;  // [n+1]
    const uint8_t* edges;       // [total][2]
    long long n;
    uint32_t* ent_off;          // [n][nv+1]
    uint32_t* ent;              // [2*total]
    unsigned long long budget;
    unsigned long long* cursor;
    uint8_t* colours;           // [n][nv]
    unsigned long long* nodes;
    uint8_t* status;
    unsigned long long* totals;
    int trail;
    // counting batches (k_count_batch_graphs) only
    unsigned long long limit = 0;               // solution limit per instance (0 = every solution)
    unsigned long long* n_solutions = nullptr;  // [n]
};

// k_graphs_build's shared memory per warp: deg[nv + 1] and an nv x nv adjacency bit matrix
__host__ __device__ inline size_t graphs_build_warp_bytes(int nv) { return ((size_t)(nv + 1) + (size_t)nv * ((nv + 31) / 32)) * 4; }

__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_graphs_build(BatchGraphsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long i = (long long)blockIdx.x * kWarpsPerCta + wib;
    if (i >= A.n) return;
    const int nw = (A.nv + 31) / 32;
    uint32_t* deg = (uint32_t*)(smem + (size_t)wib * graphs_build_warp_bytes(A.nv));
    uint32_t* adj = deg + A.nv + 1;                   // row v: the neighbours of v
    const long long e0 = A.edge_off[i], e1 = A.edge_off[i + 1];
    for (int v = lane; v <= A.nv; v += 32) deg[v] = 0;
    for (int w = lane; w < A.nv * nw; w += 32) adj[w] = 0;
    __syncwarp();
    // A repeated or reversed edge is one neighbour: fc_apply trails every entry that changes a domain word, and two
    // entries on the same neighbour in one 32-lane pass would both be trailed, past the trail's nv * k + 32 bound.
    for (long long e = e0 + lane; e < e1; e += 32) {
        const int u = A.edges[2 * e], v = A.edges[2 * e + 1];
        atomicOr(&adj[u * nw + (v >> 5)], 1u << (v & 31));
        atomicOr(&adj[v * nw + (u >> 5)], 1u << (u & 31));
    }
    __syncwarp();
    for (int v = lane; v < A.nv; v += 32) {
        uint32_t d = 0;
        for (int w = 0; w < nw; w++) d += __popc(adj[v * nw + w]);
        deg[v] = d;
    }
    __syncwarp();
    // exclusive scan of deg[0..nv) by the warp, 32 at a time
    uint32_t carry = 0;
    uint32_t* off = A.ent_off + (size_t)i * (A.nv + 1);
    for (int v0 = 0; v0 < A.nv; v0 += 32) {
        const int v = v0 + lane;
        const uint32_t dv = v < A.nv ? deg[v] : 0;
        uint32_t inc = dv;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += t; }
        if (v < A.nv) { off[v] = carry + inc - dv; deg[v] = carry + inc - dv; }
        carry += __shfl_sync(FULL, inc, 31);
    }
    if (lane == 0) off[A.nv] = carry;
    __syncwarp();
    uint32_t* ent = A.ent + 2 * e0;
    // each adjacency list in ascending neighbour id (deterministic; the order of a variable's entries changes no result)
    for (int v = lane; v < A.nv; v += 32) {
        uint32_t o = deg[v];
        for (int w = 0; w < nw; w++)
            for (uint32_t b = adj[v * nw + w]; b; b &= b - 1)
                ent[o++] = (uint32_t)(w * 32 + __ffs((int)b) - 1) | (D_K_NE_SAME << D_KIND_SHIFT);
    }
}

// As batch_cells, with the instance's adjacency from k_graphs_build.
template <bool COUNT>
__device__ __forceinline__ void batch_graphs(BatchGraphsArgs A, unsigned char* smem, int lane, int wib) {
    const int nv = A.nv;
    WarpState S = carve_warp_state(smem + (size_t)wib * warp_state_bytes(nv, A.trail), nv, A.trail);
    const uint32_t full = A.k >= 32 ? FULL : ((1u << A.k) - 1u);
    unsigned long long t_sat = 0, t_unsat = 0, t_budget = 0, t_nodes = 0;
    for (;;) {
        long long i = 0;
        if (lane == 0) i = (long long)atomicAdd(A.cursor, 1ull);
        i = __shfl_sync(FULL, i, 0);
        if (i >= A.n) break;
        DevTables T;
        T.nv = nv;
        T.ent_off = A.ent_off + (size_t)i * (nv + 1);
        T.ent = A.ent + 2 * A.edge_off[i];
        T.ent_moff = nullptr;
        T.masks = nullptr;
        for (int v = lane; v < nv; v += 32) { S.D[v] = full; S.F[v] = 0; S.order[v] = (uint16_t)v; S.pos[v] = (uint16_t)v; }
        __syncwarp();
        DfsResult R;
        if constexpr (COUNT)
            R = warp_dfs<false, false, true>(T, S, 0, true, A.budget, nullptr, 0ull, lane,
                                             FirstBytes{A.colours + (size_t)i * nv, nullptr, nv, lane}, A.limit);
        else R = warp_dfs<false, false>(T, S, 0, false, A.budget, nullptr, 0ull, lane, NoFirst());
        uint8_t* out = A.colours + (size_t)i * nv;
        if constexpr (COUNT) {
            if (!R.sols) for (int v = lane; v < nv; v += 32) out[v] = 0xFF;
            if (lane == 0) A.n_solutions[i] = R.sols;
        } else {
            for (int v = lane; v < nv; v += 32) out[v] = R.outcome == 1 ? S.val[v] : (uint8_t)0xFF;
        }
        if (lane == 0) { A.nodes[i] = R.nodes; A.status[i] = (uint8_t)R.outcome; }
        t_nodes += R.nodes;
        t_sat += R.outcome == 1; t_unsat += R.outcome == 0; t_budget += R.outcome == 2;
        __syncwarp();
    }
    if (lane == 0) {
        atomicAdd(A.totals + 0, t_sat); atomicAdd(A.totals + 1, t_unsat);
        atomicAdd(A.totals + 2, t_budget); atomicAdd(A.totals + 3, t_nodes);
    }
}

__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_batch_graphs(BatchGraphsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    batch_graphs<false>(A, smem, threadIdx.x & 31, threadIdx.x >> 5);
}

__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_count_batch_graphs(BatchGraphsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    batch_graphs<true>(A, smem, threadIdx.x & 31, threadIdx.x >> 5);
}

// ---- many independent models (dq_solve_models): one warp owns one model's whole tree -----------------------------
// Node budget of one model inside the batch: a tree that is not finished by then is marked split and solved afterwards
// by the single-model path.  Not yet measured: scripts/models_budget_sweep.py is the sweep that is to choose it
// (DESIGN.md §4.1f).
constexpr unsigned long long kModelWarpNodes = 1ull << 14;

// Where one model's tables sit in the packed block (byte offsets from `base`; ent_off at `base` itself) and its slice of
// the output value-index bytes.
struct ModelSlot {
    unsigned long long base;
    uint32_t o_ent, o_ent_moff, o_masks, o_dom0, o_order, o_pos;
    int nv, trail;
    unsigned long long sol;
};
struct ModelOut {
    unsigned long long nodes, sols;
    int outcome;            // dq_outcome; DQ_BUDGET = split
    int pad;
};
struct ModelsArgs {
    const ModelSlot* slots;         // this launch's slots
    long long n;
    const uint8_t* tables;          // the packed block
    size_t warp_bytes;              // shared memory per warp: the largest state of this launch
    int count_all;
    unsigned long long* cursor;
    ModelOut* out;                  // [n] this launch's results
    uint8_t* sol;                   // value index per var id, every model's slice
};

// The first solution of one model into its slice, value indices by var id.  Only this warp writes the slice.
struct FirstToSlice {
    uint8_t* dst;
    int nv, lane;
    template <typename W>
    __device__ void operator()(const WarpStateT<W>& S) const {
        for (int i = lane; i < nv; i += 32) dst[S.order[i]] = S.val[i];
    }
    template <typename W>
    __device__ void solutions(const WarpStateT<W>&, W, unsigned long long) const {}
};

template <bool HAS_F, bool HAS_TABLE, typename W>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_models_dfs(ModelsArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned char* region = smem + (size_t)wib * A.warp_bytes;
    for (;;) {
        long long j = 0;
        if (lane == 0) j = (long long)atomicAdd(A.cursor, 1ull);
        j = __shfl_sync(FULL, j, 0);
        if (j >= A.n) break;
        const ModelSlot s = A.slots[j];
        const uint8_t* b = A.tables + s.base;
        TreeModelDevT<W> M;
        M.T.nv = s.nv;
        M.T.ent_off = reinterpret_cast<const uint32_t*>(b);
        M.T.ent = reinterpret_cast<const uint32_t*>(b + s.o_ent);
        M.T.ent_moff = reinterpret_cast<const uint32_t*>(b + s.o_ent_moff);
        M.T.masks = reinterpret_cast<const W*>(b + s.o_masks);
        M.dom0 = reinterpret_cast<const W*>(b + s.o_dom0);
        M.order = reinterpret_cast<const uint16_t*>(b + s.o_order);
        M.pos = reinterpret_cast<const uint16_t*>(b + s.o_pos);
        M.trail = s.trail;
        const WarpStateT<W> S = carve_warp_state_t<W>(region, s.nv, s.trail);
        load_root_state(M, S, lane);
        const FirstToSlice rec{A.sol + s.sol, s.nv, lane};
        const DfsResult R = warp_dfs<HAS_F, HAS_TABLE>(M.T, S, 0, A.count_all != 0, kModelWarpNodes, nullptr, 0ull, lane, rec);
        if (!A.count_all && R.have_first) rec(S);
        if (lane == 0) { A.out[j].nodes = R.nodes; A.out[j].sols = R.sols; A.out[j].outcome = R.outcome; }
        __syncwarp();
    }
}

// ---- integer-pipe peak: 8 independent lop3.b32 chains per lane, one LOP3 per statement ------------
#define DQ_LOP3(d, a, b) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(d) : "r"(a), "r"(b))
__global__ void __launch_bounds__(1024) k_int_peak(uint32_t* out, int iters) {
    uint32_t a0 = threadIdx.x, a1 = a0 * 3 + 1, a2 = a0 * 5 + 2, a3 = a0 * 7 + 3, a4 = a0 * 11 + 4, a5 = a0 * 13 + 5,
             a6 = a0 * 17 + 6, a7 = a0 * 19 + 7;
    const uint32_t k0 = blockIdx.x * 2654435761u + 1;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            DQ_LOP3(a0, a1, k0); DQ_LOP3(a1, a2, k0); DQ_LOP3(a2, a3, k0); DQ_LOP3(a3, a4, k0);
            DQ_LOP3(a4, a5, k0); DQ_LOP3(a5, a6, k0); DQ_LOP3(a6, a7, k0); DQ_LOP3(a7, a0, k0);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

// FIRST-mode node accounting above the split (dq_tree_nodes_upto): one thread walks the parent chain of prefix `key`
// from the split depth to the root and adds, per level, the nodes the reference visits there up to the value that leads
// on (node_off of the parent + the values of its domain up to that one).  One launch and one 8-byte read-back instead
// of three synchronous copies per level.
struct LevelPtrs {
    const uint32_t* parent_of;           // [n of level l+1] -> index in level l   (stored with level l+1's entry)
    const unsigned long long* node_off;  // [n of level l]
    const void* dmask;                   // [n of level l], 32- or 64-bit words
};
__global__ void k_nodes_upto(const LevelPtrs* __restrict__ lv, int depth, unsigned long long key, const uint8_t* __restrict__ prefix,
                             int wide, unsigned long long* __restrict__ out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    unsigned long long total = 0, idx = key;
    for (int l = depth - 1; l >= 0; l--) {
        const uint32_t par = lv[l + 1].parent_of[idx];
        const unsigned long long dm = wide ? reinterpret_cast<const unsigned long long*>(lv[l].dmask)[par]
                                           : (unsigned long long)reinterpret_cast<const uint32_t*>(lv[l].dmask)[par];
        const int v = prefix[l];
        const unsigned long long upto_bit = v >= 63 ? ~0ull : (2ull << v) - 1ull;
        total += lv[l].node_off[par] + (unsigned long long)__popcll(dm & upto_bit);
        idx = par;
    }
    *out = total;
}

}  // namespace dq
