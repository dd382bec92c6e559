// dq_lane_queens.cuh — forward-checking search for the N-Queens model class
// (CLASS_QUEENS: N variables on [0,N), NotEqual with offsets {0, +-(j-i)} for every pair —
// exactly /root/reference/test/main-test.cpp:36-49, recognised by the model compiler).
//
// The search state of a node is three bit masks:
//   a      values taken by the assigned variables
//   l, r   the two diagonal masks, shifted one bit per depth, so that the current domain of the
//          variable at distance j+1 is   full & ~(a | l<<j | r>>j)
//          — the closed form of what OpConstraint::AplyArcConsistency + Domain::Exclude
//          (dequan.h:631-694, 985-1031) leave in current_domains[d+1+j].
// Forward checking of a candidate = test every later variable's domain for emptiness
// (dequan.h:514-518, 663-668).  Node accounting is the reference's: one node per AssignVar call
// (dequan.h:416-423), i.e. per value of the current filtered domain of the next variable, whether
// or not its check then succeeds.
//
// A queue of kernels with no host round trip in between:
//   k_queens_level      : one launch per level above the split depth k.  The frontier is a record list
//                         in HBM {key, a, l, r}; key is the base-N number formed by the prefix values,
//                         i.e. the DFS order of the prefix.  One lane per (record, value) pair: a value
//                         of the current domain is a node; a surviving child is appended to the next
//                         frontier with a CTA-aggregated atomic.
//   k_queens_bucket_t   : the search below the depth-k records: per-warp pools of open frames
//                         {a, l, r, untried} in shared memory, bucketed by depth, 64 nodes of ONE depth
//                         per trip; compiled per bucket count (up to 8), levels as static control flow, the
//                         records in registers and the last variable in the lane (see the comments above
//                         the kernel).  DEFAULT.
//   k_queens_bucket     : the same search with the bucket count at run time, for splits that leave more
//                         than eight buckets.
//   k_queens_first_warp : one warp, on a side stream, walks the tree in the reference's order to the
//                         DFS-first solution of this partition (solution bookkeeping stays out of the
//                         counting kernel).
// Prefixes are dealt to partitions (multi-GPU) by key at depth min(k, 5): partition r owns keys = r (mod parts);
// the levels above that depth are expanded by every partition and counted by partition 0 only, the levels below
// it by the owner alone.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "dq_group_graphs.cuh"     // bulk-copy / mbarrier primitives

namespace dq {

struct QueensLaneArgs {
    int n, k;                         // board size; split depth
    int part_rank, part_count;
    int part_level;                   // children of this level are dealt to the partitions by key (multi-GPU); -1: the root
    uint4* records;                   // [record_cap] {key, a, l, r}: one FC-surviving prefix = one subtree
    unsigned long long record_cap;
    unsigned long long* n_records;    // depth-k records found (may exceed record_cap: then the host grows and reruns)
    unsigned long long* cursor;       // next record to search
    unsigned long long* totals;       // [0] solutions, [1] nodes counted by the frontier (level) kernels
    unsigned long long* dfs_nodes;    // nodes counted by the subtree DFS kernel
    unsigned long long* best_key;     // lowest item index that holds a solution
    uint8_t* first_out;               // [32] DFS-first solution, values by variable
};

constexpr int kQueensBlock = 256;
constexpr int kQueensMaxN = 31;       // one spare bit so that ~(a|l|r) of a full board is still distinguishable

// Phase A, one launch per level above the split: every lane takes one (record, value) pair of the
// current frontier, and if the value is in the record's current domain it is a node (AssignVar);
// if its forward check leaves no later domain empty the child record is appended (warp-aggregated
// atomic) to the next frontier.  The launches are queued back to back: the frontier sizes never
// come back to the host.  On the last level only the children this partition owns are kept.
template <bool IN_IS_READ_ONLY>
__device__ __forceinline__ void queens_level_body(const QueensLaneArgs& A, int level, const uint4* __restrict__ in, unsigned long long n_found,
                                                  uint4* __restrict__ out, unsigned long long* __restrict__ n_out_ptr, int count_nodes,
                                                  int filter_partition, uint32_t* s_cnt, unsigned long long* s_base_p) {
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const int N = A.n;
    const uint32_t full = (1u << N) - 1u;
    const unsigned long long n_in = min(n_found, A.record_cap);
    const unsigned long long pairs = n_in * (unsigned long long)N;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long tot_nodes = 0;
    unsigned long long& s_base = *s_base_p;
    const unsigned long long first = (unsigned long long)blockIdx.x * blockDim.x;
    for (unsigned long long tile = first; tile < pairs; tile += stride) {      // CTA-uniform trip count
        const unsigned long long base = tile + (threadIdx.x & ~31);
        const unsigned long long p = base + lane;
        bool valid = p < pairs;
        uint32_t key = 0, a = 0, l = 0, r = 0;
        if (valid) {
            const unsigned long long rix = p / (unsigned long long)N;          // (the host caps the list at 2^29 records: pairs may pass 2^32)
            const uint32_t v = (uint32_t)(p - rix * N);
            // (the fused head kernel reads records it wrote itself one level earlier: no read-only cache path there)
            const uint4 rec = IN_IS_READ_ONLY ? __ldg(in + rix) : __ldcg(in + rix);
            const uint32_t bit = 1u << v;
            valid = (full & ~(rec.y | rec.z | rec.w) & bit) != 0;               // value in the current domain
            if (valid) {
                ++tot_nodes;
                key = rec.x * N + v;
                a = rec.y | bit;
                l = (rec.z | bit) << 1;
                r = (rec.w | bit) >> 1;
                const uint32_t ah = a | ~full;
                for (int j = 0; j <= N - 2 - level; j++)
                    if ((ah | (l << j) | (r >> j)) == 0xFFFFFFFFu) { valid = false; break; }   // wipe-out
                if (valid && filter_partition) valid = (key % (uint32_t)A.part_count) == (uint32_t)A.part_rank;
            }
        }
        // one atomic per CTA and tile (all warps of the CTA run the same number of tiles): the shared counter sees
        // 8x fewer same-address atomics than with warp-level aggregation
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, valid);
        const int wib = threadIdx.x >> 5;
        if (lane == 0) s_cnt[wib] = __popc(m);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
#pragma unroll
            for (int w = 0; w < kQueensBlock / 32; w++) { const uint32_t c = s_cnt[w]; s_cnt[w] = tot; tot += c; }
            s_base = tot ? atomicAdd(n_out_ptr, (unsigned long long)tot) : 0ull;
        }
        __syncthreads();
        if (valid) {
            const unsigned long long slot = s_base + s_cnt[wib] + __popc(m & lt);
            if (slot < A.record_cap) out[slot] = make_uint4(key, a, l, r);
        }
        __syncthreads();
    }
    if (count_nodes) {
        for (int o = 16; o > 0; o >>= 1) tot_nodes += __shfl_down_sync(0xFFFFFFFFu, tot_nodes, o);
        if (lane == 0 && tot_nodes) atomicAdd(A.totals + 1, tot_nodes);
    }
}

__global__ void __launch_bounds__(kQueensBlock)
k_queens_level(QueensLaneArgs A, int level, const uint4* __restrict__ in, const unsigned long long* __restrict__ n_in_ptr,
               uint4* __restrict__ out, unsigned long long* __restrict__ n_out_ptr, int count_nodes, int filter_partition) {
    __shared__ uint32_t s_cnt[kQueensBlock / 32];
    __shared__ unsigned long long s_base;
    queens_level_body<true>(A, level, in, *n_in_ptr, out, n_out_ptr, count_nodes, filter_partition, s_cnt, &s_base);
}

// The same level step for WIDE frontiers (tens of thousands of records and more): one lane per RECORD instead of one
// per (record, value) pair — with N = 17 only about three of a record's seventeen values are in its domain, so the
// pair layout idles four lanes in five.  Pass 1 forward-checks the record's candidate values one per trip (the trip
// count is the warp's largest domain) and keeps the survivors as a bit mask; the CTA then reserves its output range
// with ONE atomic; pass 2 writes the children trip-major, so that each trip's stores are contiguous.
__global__ void __launch_bounds__(kQueensBlock)
k_queens_level_wide(QueensLaneArgs A, int level, const uint4* __restrict__ in, const unsigned long long* __restrict__ n_in_ptr,
                    uint4* __restrict__ out, unsigned long long* __restrict__ n_out_ptr, int count_nodes, int filter_partition) {
    __shared__ uint32_t s_cnt[kQueensBlock / 32];
    __shared__ unsigned long long s_base;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int N = A.n;
    const uint32_t full = (1u << N) - 1u;
    const int last = N - 2 - level;
    const unsigned long long n_in = min(*n_in_ptr, A.record_cap);
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long tot_nodes = 0;
    for (unsigned long long tile = (unsigned long long)blockIdx.x * blockDim.x; tile < n_in; tile += stride) {   // CTA-uniform trip count
        const unsigned long long rix = tile + threadIdx.x;
        uint4 rec = make_uint4(0u, 0xFFFFFFFFu, 0u, 0u);
        if (rix < n_in) rec = __ldg(in + rix);
        const uint32_t ah = rec.y | ~full;
        uint32_t cand = ~(ah | rec.z | rec.w);
        tot_nodes += __popc(cand);                                          // every value of the domain is a node
        uint32_t surv = 0;
        while (__any_sync(0xFFFFFFFFu, cand != 0u)) {
            const uint32_t bit = cand & (0u - cand);
            cand ^= bit;
            const uint32_t na = ah | bit, nl = (rec.z | bit) << 1, nr = (rec.w | bit) >> 1;
            uint32_t worst = 0;
            for (int j = 0; j <= last; j++) worst = max(worst, na | (nl << j) | (nr >> j));
            bool ok = bit != 0u && worst != 0xFFFFFFFFu;
            if (ok && filter_partition)
                ok = ((rec.x * (uint32_t)N + ((uint32_t)__ffs((int)bit) - 1u)) % (uint32_t)A.part_count) == (uint32_t)A.part_rank;
            if (ok) surv |= bit;
        }
        // one atomic per CTA and tile
        uint32_t mine = __popc(surv), incl = mine;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) s_cnt[wib] = incl;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
#pragma unroll
            for (int w = 0; w < kQueensBlock / 32; w++) { const uint32_t c = s_cnt[w]; s_cnt[w] = tot; tot += c; }
            s_base = tot ? atomicAdd(n_out_ptr, (unsigned long long)tot) : 0ull;
        }
        __syncthreads();
        unsigned long long slot0 = s_base + s_cnt[wib];
        while (__any_sync(0xFFFFFFFFu, surv != 0u)) {
            const uint32_t bit = surv & (0u - surv);
            surv ^= bit;
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, bit != 0u);
            if (bit) {
                const unsigned long long slot = slot0 + __popc(m & lt);
                if (slot < A.record_cap)
                    out[slot] = make_uint4(rec.x * (uint32_t)N + ((uint32_t)__ffs((int)bit) - 1u), rec.y | bit, (rec.z | bit) << 1, (rec.w | bit) >> 1);
            }
            slot0 += __popc(m);
        }
        __syncthreads();
    }
    if (count_nodes) {
        for (int o = 16; o > 0; o >>= 1) tot_nodes += __shfl_down_sync(0xFFFFFFFFu, tot_nodes, o);
        if (lane == 0 && tot_nodes) atomicAdd(A.totals + 1, tot_nodes);
    }
}

// The first levels hold a handful of records (1, N, about N^2 / 1.2): ONE CTA walks levels 0 .. n_levels-1 back to back
// instead of one launch each (a launch costs more than these levels' work).  buf0 / buf1 alternate as in the host loop,
// sizes[l] is the frontier size at depth l.
__global__ void __launch_bounds__(kQueensBlock)
k_queens_levels_head(QueensLaneArgs A, int n_levels, uint4* __restrict__ buf0, uint4* __restrict__ buf1,
                     unsigned long long* __restrict__ sizes, int count_nodes) {
    __shared__ uint32_t s_cnt[kQueensBlock / 32];
    __shared__ unsigned long long s_base;
    for (int l = 0; l < n_levels; l++) {
        const unsigned long long n_in = *(volatile unsigned long long*)(sizes + l);
        queens_level_body<false>(A, l, (l & 1) ? buf1 : buf0, n_in, (l & 1) ? buf0 : buf1, sizes + l + 1, count_nodes, 0, s_cnt, &s_base);
        __threadfence();
        __syncthreads();                                 // the children and their count are visible to the whole CTA
    }
}

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
// PTX shifts clamp the amount (>= 32 gives 0), unlike C++ where it is undefined.
__device__ __forceinline__ uint32_t shl_clamp(uint32_t x, uint32_t n) { uint32_t r; asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n)); return r; }
__device__ __forceinline__ uint32_t shr_clamp(uint32_t x, uint32_t n) { uint32_t r; asm("shr.u32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n)); return r; }

// ---------------------------------------------------------------------------------------------------------------
// Depth-bucketed warp search (COUNT_ALL).  A lane-per-subtree search (round 1's first engine: explicit stack per lane;
// profiles/r1_ncu_queens17_lane_old.txt) pays for SIMT twice: its forward-check loop runs to the row count of the
// SHALLOWEST lane of the warp (about 9 rows per trip when a node needs 4.3 on average, N=17), and lanes idle while
// their mates finish a subtree.  Here a warp owns a pool of open frames
// {a, l, r, untried} in shared memory, bucketed by depth, and every trip takes up to 64 frames of ONE depth, two per
// lane:
//   * the row count of the forward check is warp-uniform and exact (no max over lanes, uniform shift amounts);
//   * each lane tries the lowest untried value of each of its two frames (one node each, dequan.h:416-423); frames
//     that still hold untried values go back to the bucket, surviving children go to the next bucket, both
//     compacted with ballots; the bucket choice, the counts and the loop are paid once per 64 nodes and the two
//     dependency chains interleave;
//   * the bucket is chosen deepest-first among those holding 64 frames, which bounds every bucket below 128 frames
//     (a bucket is only fed, by at most 64, while it holds fewer than 64); with no full bucket the warp pulls 64
//     more records from the frontier list, and once that is empty widens from the shallowest bucket.
// Node and solution counts do not depend on the visiting order; the DFS-first solution is found separately by
// queens_first_owned.  Bucket sizes live in registers, lane i holding the size of bucket i.
constexpr int kQueensBucketMaxWarps = 12;             // warps per CTA: the host picks what packs an SM's shared memory best
constexpr int kQueensBucketCap = 128;

// DFS-first solution of the part of the tree this partition owns, and the depth-k key of its prefix
// (ForwardCheckingStep's own order, dequan.h:494-571).  Run by one warp in a kernel of its own, on a second stream
// next to the level and bucket kernels (inside the bucket kernel the call costs the compiler its proof that the
// search loop is warp-uniform, and with it the uniform datapath: 18.0 -> 21.6 ms on 17-Queens).  The search state is
// warp-uniform, lane j tests the domain of the j-th later variable (one vote per
// node), and lane d keeps the frame of depth d in its registers (a pop is four shuffles, nothing touches memory).
// (Measured and dropped: a whole level per step — lane v forward-checks value v in a row loop of its own, one ballot per
// level.  Fewer steps but three times the instructions, and this warp shares its SM quarter with the bucket kernel's
// warps: the 14-Queens solve went from 0.179 to 0.238 ms.  And the two lowest untried values per vote, lanes 0-15 on the
// rows of the first and 16-31 on the rows of the second: the warp alone 152 -> 205 us on 14-Queens; both values on all
// lanes, two chains and two votes per step: 187 us — most values pass, so the second verdict is rarely the one needed.)
__device__ __forceinline__ void queens_first_owned(const QueensLaneArgs& A, int lane, unsigned long long* nodes_out = nullptr) {
    const int N = A.n, K = A.k;
    const uint32_t full = (1u << N) - 1u;
    const int own_depth = A.part_level + 1;              // prefixes of this depth are dealt to the partitions by key
    if (A.part_count > 1 && own_depth <= 0 && A.part_rank != 0) return;
    uint32_t fa = 0, fl = 0, fr = 0, fc = 0, fb = 0;     // lane d: the frame of depth d (state before its value, values left, the value's bit)
    uint32_t a = 0, l = 0, r = 0, cand = full;
    int d = 0;
    unsigned long long tries = 0;                        // values tried = AssignVar calls (dequan.h:416-423) on the way
    // Nothing in the loop needs a value's INDEX or the prefix key (a find-first-set and a 64-bit multiply-add per node
    // that the in-order issue would wait for): frames keep the value's bit, and keys are folded out of the frames
    // where they are used — at the level the partitions are dealt at, and once at the end.
    // base-N number of the values at depths 0 .. upto-1 (frames of lanes 0 .. upto-1), 64-bit: N^k outgrows 32 bits from k = 8 on
    auto key_of = [&](int upto) {
        unsigned long long key = 0;
        for (int i = 0; i < upto; i++) key = key * (unsigned long long)N + ((unsigned)__ffs((int)__shfl_sync(0xFFFFFFFFu, fb, i)) - 1u);
        return key;
    };
    for (;;) {
        if (cand == 0) {                                 // every value tried at this depth
            if (d == 0) { if (nodes_out && lane == 0) *nodes_out = tries; return; }   // no solution in this partition's share
            --d;
            a = __shfl_sync(0xFFFFFFFFu, fa, d); l = __shfl_sync(0xFFFFFFFFu, fl, d); r = __shfl_sync(0xFFFFFFFFu, fr, d);
            cand = __shfl_sync(0xFFFFFFFFu, fc, d);
            continue;
        }
        const uint32_t bit = cand & (0u - cand);
        cand ^= bit;
        ++tries;
        const uint32_t na = a | bit, nl = (l | bit) << 1, nr = (r | bit) >> 1;
        const bool wiped = lane < N - 1 - d && ((na | ~full) | (nl << lane) | (nr >> lane)) == 0xFFFFFFFFu;
        if (__any_sync(0xFFFFFFFFu, wiped)) continue;
        if (A.part_count > 1 && d + 1 == own_depth) {
            const unsigned long long kchild = key_of(d) * (unsigned long long)N + ((unsigned)__ffs((int)bit) - 1u);   // (own_depth <= k)
            if ((uint32_t)(kchild % (unsigned long long)A.part_count) != (uint32_t)A.part_rank) continue;
        }
        if (lane == d) { fa = a; fl = l; fr = r; fc = cand; fb = bit; }
        if (d == N - 2) {
            uint32_t fv = (uint32_t)__ffs((int)fb) - 1u;
            if (lane == N - 1) fv = (uint32_t)__ffs((int)(full & ~(na | nl | nr))) - 1u;
            if (lane < N) A.first_out[lane] = (uint8_t)fv;
            const unsigned long long key = key_of(K < N - 1 ? K : N - 1);       // the key stops growing at depth k
            if (lane == 0) *A.best_key = key;
            if (nodes_out && lane == 0) *nodes_out = tries + 1ull;      // ... and the last variable's first value completes the solution
            return;
        }
        a = na; l = nl; r = nr; cand = full & ~(na | nl | nr);
        ++d;
    }
}

// Unsigned max over the next ROWS variables of their occupied masks (all ones <=> that domain is empty).
template <int ROWS>
__device__ __forceinline__ uint32_t queens_rows_occupied(uint32_t na, uint32_t nl, uint32_t nr) {
    uint32_t m = 0;
#pragma unroll
    for (int j = 0; j < ROWS; j++) m = max(m, na | (nl << j) | (nr >> j));
    return m;
}

__global__ void __launch_bounds__(32) k_queens_first_warp(QueensLaneArgs A) { queens_first_owned(A, (int)threadIdx.x); }
// FIRST mode on the class (one partition): the same walk IS the reference's search up to its first solution — the values
// it tries are the nodes.
__global__ void __launch_bounds__(32) k_queens_first_nodes(QueensLaneArgs A, unsigned long long* nodes) { queens_first_owned(A, (int)threadIdx.x, nodes); }

__global__ void __launch_bounds__(kQueensBucketMaxWarps * 32)
k_queens_bucket(QueensLaneArgs A) {
    extern __shared__ uint4 qb_frames[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int N = A.n;
    const int L = N - 2 - A.k;                                   // buckets: depth k .. N-3 (frames of depth N-2 never reach a bucket: see below)
    const uint32_t hi = ~((1u << N) - 1u);
    const uint32_t per_warp = (uint32_t)L * kQueensBucketCap * 16u;
    const uint32_t bbase = (uint32_t)__cvta_generic_to_shared(qb_frames) + (uint32_t)wib * per_warp;
    uint32_t pf_n = 0;                                           // records prefetched into pf0 / pf1 (in flight or landed)
    uint4 pf0 = make_uint4(0u, 0u, 0u, 0u), pf1 = pf0;
    const unsigned long long n_found = *A.n_records;
    const unsigned long long n_rec = n_found < A.record_cap ? n_found : A.record_cap;   // overflow: the host grows the list and reruns
    const unsigned long long total_warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    const uint32_t fair_share = (uint32_t)min((n_rec + total_warps - 1) / total_warps, 64ull);


    uint32_t cnt = 0;                                            // lane i: frames in bucket i
    unsigned long long trip_nodes = 0;                           // warp-uniform: one node per frame taken (AssignVar of its next value)
    unsigned long long tot_sols = 0;                             // per lane: values of the last variable (a node and a solution each)
    unsigned long long tot_lane_nodes = 0;                       // per lane: values tried for variable N-2
    unsigned long long chunk_pos = 0, chunk_end = 0;
    bool exhausted = false;

    for (;;) {
        const uint32_t big = __ballot_sync(0xFFFFFFFFu, cnt >= 64u);
        int lvl;
        if (big) lvl = 31 - __clz((int)big);
        else {
            // claims the next chunk of the record list if need be and starts the loads of up to 64 records of it: they
            // stay in flight (two uint4 registers per lane) while the warp works through the records it has
            auto prefetch = [&]() {
                if (exhausted) return;
                if (chunk_pos >= chunk_end) {
                    unsigned long long base = 0;
                    uint32_t size = 0;
                    if (lane == 0) {
                        const unsigned long long cur = *(volatile unsigned long long*)A.cursor;
                        const unsigned long long remaining = cur < n_rec ? n_rec - cur : 0;
                        size = (uint32_t)min(max(remaining / (4ull * total_warps), (unsigned long long)max(fair_share, 1u)), 256ull);
                        base = atomicAdd(A.cursor, (unsigned long long)size);
                    }
                    base = __shfl_sync(0xFFFFFFFFu, base, 0);
                    size = __shfl_sync(0xFFFFFFFFu, size, 0);
                    chunk_pos = base;
                    chunk_end = min(base + size, n_rec);
                    if (base >= n_rec) { exhausted = true; chunk_end = chunk_pos; return; }
                }
                pf_n = (uint32_t)min(chunk_end - chunk_pos, 64ull);
                if ((uint32_t)lane < pf_n) pf0 = __ldg(A.records + chunk_pos + lane);
                if ((uint32_t)lane + 32u < pf_n) pf1 = __ldg(A.records + chunk_pos + lane + 32);
                chunk_pos += pf_n;
            };
            if (pf_n == 0u) prefetch();
            if (pf_n != 0u) {
                const uint32_t c0 = __shfl_sync(0xFFFFFFFFu, cnt, 0);
                if ((uint32_t)lane < pf_n) { const uint32_t a = pf0.y | hi; sts128(bbase + ((c0 + lane) << 4), a, pf0.z, pf0.w, ~(a | pf0.z | pf0.w)); }
                if ((uint32_t)lane + 32u < pf_n) { const uint32_t a = pf1.y | hi; sts128(bbase + ((c0 + lane + 32) << 4), a, pf1.z, pf1.w, ~(a | pf1.z | pf1.w)); }
                if (lane == 0) cnt = c0 + pf_n;
                pf_n = 0;
                __syncwarp();
                prefetch();
                continue;
            }
            const uint32_t any = __ballot_sync(0xFFFFFFFFu, cnt != 0u);
            if (!any) break;
            lvl = __ffs((int)any) - 1;
        }
        const uint32_t c = __shfl_sync(0xFFFFFFFFu, cnt, lvl);
        const uint32_t row = bbase + (uint32_t)lvl * (kQueensBucketCap * 16u);
        uint32_t keep_base = c - 64u;
        if (c < 64u) {
            // a short trip (the tail of the warp's work): pads the bucket to 64 with frames that hold no value — every
            // trip is then a full one, with no per-lane "is this slot in use" anywhere below
            if ((uint32_t)lane >= c) sts128(row + ((uint32_t)lane << 4), 0xFFFFFFFFu, 0u, 0u, 0u);
            if ((uint32_t)lane + 32u >= c) sts128(row + (((uint32_t)lane + 32u) << 4), 0xFFFFFFFFu, 0u, 0u, 0u);
            keep_base = 0u;
            __syncwarp();
        }
        trip_nodes += min(c, 64u);
        // two frames per lane and trip: the bucket choice, the counts and the loop are paid once for 64 nodes, and the two
        // dependency chains interleave
        const uint4 fA = lds128(row + ((keep_base + lane) << 4)), fB = lds128(row + ((keep_base + 32u + lane) << 4));
        const uint32_t aA = fA.x, lA = fA.y, rA = fA.z, aB = fB.x, lB = fB.y, rB = fB.z;
        const uint32_t bitA = fA.w & (0u - fA.w), bitB = fB.w & (0u - fB.w);      // (0 for a frame without values: its child below is "wiped")
        const uint32_t cA = fA.w ^ bitA, cB = fB.w ^ bitB;
        const uint32_t naA = aA | bitA, nlA = (lA | bitA) << 1, nrA = (rA | bitA) >> 1;
        const uint32_t naB = aB | bitB, nlB = (lB | bitB) << 1, nrB = (rB | bitB) >> 1;
        const int last = L - lvl;                                // later variables to check, minus one (>= 1)
        uint32_t occA = 0, occB = 0;                             // all ones <=> some later domain is empty
        switch (last) {
#define DQ_QROWS(J) case J: occA = queens_rows_occupied<J + 1>(naA, nlA, nrA); occB = queens_rows_occupied<J + 1>(naB, nlB, nrB); break;
            DQ_QROWS(0) DQ_QROWS(1) DQ_QROWS(2) DQ_QROWS(3) DQ_QROWS(4) DQ_QROWS(5) DQ_QROWS(6) DQ_QROWS(7) DQ_QROWS(8) DQ_QROWS(9)
            DQ_QROWS(10) DQ_QROWS(11) DQ_QROWS(12) DQ_QROWS(13) DQ_QROWS(14) DQ_QROWS(15) DQ_QROWS(16) DQ_QROWS(17) DQ_QROWS(18) DQ_QROWS(19)
            DQ_QROWS(20) DQ_QROWS(21) DQ_QROWS(22) DQ_QROWS(23) DQ_QROWS(24) DQ_QROWS(25) DQ_QROWS(26) DQ_QROWS(27) DQ_QROWS(28)
#undef DQ_QROWS
            default: occA = queens_rows_occupied<30>(naA, nlA, nrA); occB = queens_rows_occupied<30>(naB, nlB, nrB); break;
        }
        // (a padding frame has a = all ones: "wiped" whatever the rows say)
        const bool passA = occA != 0xFFFFFFFFu, passB = occB != 0xFFFFFFFFu;
        const uint32_t keepA = __ballot_sync(0xFFFFFFFFu, cA != 0u), keepB = __ballot_sync(0xFFFFFFFFu, cB != 0u);
        const uint32_t nkA = __popc(keepA);
        if (cA) sts128(row + ((keep_base + __popc(keepA & lt)) << 4), aA, lA, rA, cA);
        if (cB) sts128(row + ((keep_base + nkA + __popc(keepB & lt)) << 4), aB, lB, rB, cB);
        const uint32_t c_new = keep_base + nkA + __popc(keepB);
        const uint32_t dA = ~(naA | nlA | nrA), dB = ~(naB | nlB | nrB);
        if (last == 1) {
            // The children hold variable N-2.  Two columns are free there, so a child has at most two values: both are
            // tried right here instead of going through a bucket of their own.  Each value is a node; what it leaves
            // to the last variable (at most the other free column) is a node and a solution per value.
            const uint32_t eA = passA ? dA : 0u, eB = passB ? dB : 0u;
            const uint32_t bA1 = eA & (0u - eA), bA2 = eA ^ bA1, bB1 = eB & (0u - eB), bB2 = eB ^ bB1;
            const uint32_t fA1 = ~(naA | bA1 | ((nlA | bA1) << 1) | ((nrA | bA1) >> 1)), fA2 = ~(naA | bA2 | ((nlA | bA2) << 1) | ((nrA | bA2) >> 1));
            const uint32_t fB1 = ~(naB | bB1 | ((nlB | bB1) << 1) | ((nrB | bB1) >> 1)), fB2 = ~(naB | bB2 | ((nlB | bB2) << 1) | ((nrB | bB2) >> 1));
            const uint32_t s = (bA1 ? __popc(fA1) : 0) + (bA2 ? __popc(fA2) : 0) + (bB1 ? __popc(fB1) : 0) + (bB2 ? __popc(fB2) : 0);
            tot_sols += s;
            tot_lane_nodes += __popc(eA) + __popc(eB);
            if (lane == lvl) cnt = c_new;
        } else {
            const uint32_t kidsA = __ballot_sync(0xFFFFFFFFu, passA), kidsB = __ballot_sync(0xFFFFFFFFu, passB);
            const uint32_t c1 = __shfl_sync(0xFFFFFFFFu, cnt, lvl + 1);
            const uint32_t nA = __popc(kidsA);
            const uint32_t nrow = row + kQueensBucketCap * 16u;
            if (passA) sts128(nrow + ((c1 + __popc(kidsA & lt)) << 4), naA, nlA, nrA, dA);
            if (passB) sts128(nrow + ((c1 + nA + __popc(kidsB & lt)) << 4), naB, nlB, nrB, dB);
            if (lane == lvl) cnt = c_new;
            if (lane == lvl + 1) cnt = c1 + nA + __popc(kidsB);
        }
        __syncwarp();
    }
    for (int o = 16; o > 0; o >>= 1) {
        tot_sols += __shfl_down_sync(0xFFFFFFFFu, tot_sols, o);
        tot_lane_nodes += __shfl_down_sync(0xFFFFFFFFu, tot_lane_nodes, o);
    }
    if (lane == 0) {
        atomicAdd(A.totals + 0, tot_sols);
        atomicAdd(A.dfs_nodes, tot_sols + tot_lane_nodes + trip_nodes);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The same search with the number of buckets L (<= 8) a template parameter, which makes everything the kernel above
// finds out per trip a compile-time constant of the code that serves one level: the bucket's address, its count (a
// register of its own), the number of later variables to check (no dispatch on it).  The deepest-first rule becomes
// control flow: after a trip at level v only bucket v+1 can have reached 64 frames, so the code of level v falls
// into the code of level v+1 when it has, and repeats itself while its own bucket still holds 64 (queens_run_from) —
// no level choice, no jump table, no shuffle in the trip's dependency chain.
//
// The round-1 kernel was bound by the ALU pipe (LOP3 / SHF / ISETP / VIMNMX: 16 lanes per clock and SM quarter, the
// INT32 roofline of bench.py), with the FMA pipe's integer multiply-add (IMAD, another 16 lanes per clock) idle next to
// it.  So what can be a multiplication is one: left shifts, the rank of a lane in a ballot (popc(ballot * 2^(32-lane))),
// and unions of disjoint masks (sums).
struct QueensTripState {
    uint32_t cnt[8];                       // frames per bucket (warp-uniform)
    unsigned long long trip_nodes;         // warp-uniform: one node per frame taken (AssignVar of its next value)
    unsigned long long tot_sols;           // per lane: values of the last variable (a node and a solution each)
    unsigned long long tot_lane_nodes;     // per lane: values tried for variable N-2
};

__device__ __forceinline__ uint32_t nor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x01;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t mad_lo(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// The forward check with every row in its own shifted frame: row j (the variable j+1 places on) is full when
//     (na << j | 2^j - 1)  |  nl << 2j  |  nr        is all ones
// — the same test as na | nl << j | nr >> j moved j bits up, so that no operand shifts right: the two left shifts are
// multiplications, and the ALU pipe is left with one LOP3 per row and the maximum.  Exact while no board bit of
// nl << 2j leaves the word: N + 2j <= 32.  Rows 1 .. JUP take this form and the others the plain one; the host picks
// JUP = 5 (boards up to 22 queens), the mix that loads the two pipes equally (profiles/r2_queens_split_depth.txt), else 0.
// ls = l | value bit (nl before its shift).
// The powers of two and the low ones of the first product come in registers whose values the compiler cannot see
// (QueensRowConsts): knowing them it turns the multiply-add back into a shift-add (LEA) plus a LOP3 on the ALU pipe.
struct QueensRowConsts { uint32_t pow[10], ones[10]; };
template <int ROWS, int JUP>
__device__ __forceinline__ uint32_t queens_rows_occupied_up(uint32_t na, uint32_t ls, uint32_t nr, const QueensRowConsts& rc) {
    const uint32_t nl = ls * 2u;
    uint32_t m = na | nl | nr;
#pragma unroll
    for (int j = 1; j < ROWS; j++)
        m = max(m, j <= JUP ? (mad_lo(na, rc.pow[j], rc.ones[j]) | (ls * (2u << (2 * j))) | nr)      // rows whose shifted frame fits the word
                            : (na | (nl << j) | (nr >> j)));
    return m;
}

template <int L, int LVL, int JUP, bool FULL>
__device__ __forceinline__ void queens_trip(QueensTripState& S, const uint32_t bbase, const uint32_t lane, const uint32_t rank_mul, const QueensRowConsts& rc) {
    constexpr uint32_t kRow = (uint32_t)LVL * kQueensBucketCap * 16u;
    constexpr int ROWS = L - LVL + 1;                            // later variables to check
    const uint32_t c = S.cnt[LVL];
    const uint32_t row = bbase + kRow;
    uint32_t keep_base = c - 64u;
    if constexpr (FULL) S.trip_nodes += 64u;
    else {
        if (c < 64u) {
            // a short trip (the tail of the warp's work): pads the bucket to 64 with frames that hold no value — every
            // trip is then a full one, with no per-lane "is this slot in use" anywhere below
            if (lane >= c) sts128(row + (lane << 4), 0xFFFFFFFFu, 0u, 0u, 0u);
            if (lane + 32u >= c) sts128(row + ((lane + 32u) << 4), 0xFFFFFFFFu, 0u, 0u, 0u);
            keep_base = 0u;
            __syncwarp();
        }
        S.trip_nodes += min(c, 64u);
    }
    const uint32_t top = row + (keep_base << 4);
    const uint4 fA = lds128(top + (lane << 4)), fB = lds128(top + (lane << 4) + 512u);
    const uint32_t aA = fA.x, lA = fA.y, rA = fA.z, aB = fB.x, lB = fB.y, rB = fB.z;
    const uint32_t bitA = fA.w & (0u - fA.w), bitB = fB.w & (0u - fB.w);      // (0 for a frame without values: its child below is "wiped")
    // the value is in none of a, l, r (it came out of their complement): the unions are sums
    const uint32_t cA = fA.w - bitA, cB = fB.w - bitB;
    const uint32_t naA = aA + bitA, lsA = lA + bitA, nrA = (rA + bitA) >> 1;
    const uint32_t naB = aB + bitB, lsB = lB + bitB, nrB = (rB + bitB) >> 1;
    const uint32_t nlA = lsA * 2u, nlB = lsB * 2u;
    // all ones <=> some later domain is empty (a padding frame has a = all ones)
    const bool passA = queens_rows_occupied_up<ROWS, JUP>(naA, lsA, nrA, rc) != 0xFFFFFFFFu;
    const bool passB = queens_rows_occupied_up<ROWS, JUP>(naB, lsB, nrB, rc) != 0xFFFFFFFFu;
    const uint32_t keepA = __ballot_sync(0xFFFFFFFFu, cA != 0u), keepB = __ballot_sync(0xFFFFFFFFu, cB != 0u);
    const uint32_t nkA = __popc(keepA);
    if (cA) sts128(top + (__popc(keepA * rank_mul) << 4), aA, lA, rA, cA);
    if (cB) sts128(top + (nkA << 4) + (__popc(keepB * rank_mul) << 4), aB, lB, rB, cB);
    S.cnt[LVL] = keep_base + nkA + __popc(keepB);
    const uint32_t dA = nor3(naA, nlA, nrA), dB = nor3(naB, nlB, nrB);
    if constexpr (LVL == L - 1) {
        // The children hold variable N-2.  Two columns are free there, so a child has at most two values: both are
        // tried right here instead of going through a bucket of their own.  Each value is a node; what it leaves
        // to the last variable (at most the other free column) is a node and a solution per value.
        const uint32_t eA = passA ? dA : 0u, eB = passB ? dB : 0u;
        const uint32_t bA1 = eA & (0u - eA), bA2 = eA - bA1, bB1 = eB & (0u - eB), bB2 = eB - bB1;
        const uint32_t fA1 = nor3(naA + bA1, (nlA + bA1) * 2u, (nrA + bA1) >> 1), fA2 = nor3(naA + bA2, (nlA + bA2) * 2u, (nrA + bA2) >> 1);
        const uint32_t fB1 = nor3(naB + bB1, (nlB + bB1) * 2u, (nrB + bB1) >> 1), fB2 = nor3(naB + bB2, (nlB + bB2) * 2u, (nrB + bB2) >> 1);
        S.tot_sols += (bA1 ? __popc(fA1) : 0) + (bA2 ? __popc(fA2) : 0) + (bB1 ? __popc(fB1) : 0) + (bB2 ? __popc(fB2) : 0);
        S.tot_lane_nodes += __popc(eA) + __popc(eB);
    } else {
        const uint32_t kidsA = __ballot_sync(0xFFFFFFFFu, passA), kidsB = __ballot_sync(0xFFFFFFFFu, passB);
        const uint32_t c1 = S.cnt[LVL + 1];
        const uint32_t nA = __popc(kidsA);
        const uint32_t ntop = row + kQueensBucketCap * 16u + (c1 << 4);
        if (passA) sts128(ntop + (__popc(kidsA * rank_mul) << 4), naA, nlA, nrA, dA);
        if (passB) sts128(ntop + (nA << 4) + (__popc(kidsB * rank_mul) << 4), naB, nlB, nrB, dB);
        S.cnt[LVL + 1] = c1 + nA + __popc(kidsB);
    }
    __syncwarp();
}

// The records themselves (depth k, variable k) never enter a bucket: a lane holds two of them in registers and tries
// one value of each per trip until the warp's 64 are spent — no load, nothing to put back, children to bucket 0.
// A spent record has no value bit: its "child" is nobody's.  (The nodes of this level are counted when the records
// are taken: every value of a record's domain is tried exactly once.)
struct QueensRecordRegs { uint32_t aA, lA, rA, cA, aB, lB, rB, cB; };

template <int L, int JUP>
__device__ __forceinline__ void queens_record_trip(QueensTripState& S, QueensRecordRegs& R, const uint32_t bbase, const uint32_t rank_mul, const QueensRowConsts& rc) {
    constexpr int ROWS = L + 2;                                  // later variables to check
    const uint32_t bitA = R.cA & (0u - R.cA), bitB = R.cB & (0u - R.cB);
    R.cA -= bitA; R.cB -= bitB;
    const uint32_t naA = R.aA + bitA, lsA = R.lA + bitA, nrA = (R.rA + bitA) >> 1;
    const uint32_t naB = R.aB + bitB, lsB = R.lB + bitB, nrB = (R.rB + bitB) >> 1;
    const uint32_t nlA = lsA * 2u, nlB = lsB * 2u;
    const bool passA = bitA != 0u && queens_rows_occupied_up<ROWS, JUP>(naA, lsA, nrA, rc) != 0xFFFFFFFFu;
    const bool passB = bitB != 0u && queens_rows_occupied_up<ROWS, JUP>(naB, lsB, nrB, rc) != 0xFFFFFFFFu;
    const uint32_t kidsA = __ballot_sync(0xFFFFFFFFu, passA), kidsB = __ballot_sync(0xFFFFFFFFu, passB);
    const uint32_t c0 = S.cnt[0];
    const uint32_t nA = __popc(kidsA);
    const uint32_t ntop = bbase + (c0 << 4);
    if (passA) sts128(ntop + (__popc(kidsA * rank_mul) << 4), naA, nlA, nrA, nor3(naA, nlA, nrA));
    if (passB) sts128(ntop + (nA << 4) + (__popc(kidsB * rank_mul) << 4), naB, nlB, nrB, nor3(naB, nlB, nrB));
    S.cnt[0] = c0 + nA + __popc(kidsB);
    __syncwarp();
}

// Entered with 64 frames or more in bucket LVL and fewer in every deeper one; returns once no bucket from LVL down
// holds 64.
template <int L, int LVL, int JUP>
__device__ __forceinline__ void queens_run_from(QueensTripState& S, const uint32_t bbase, const uint32_t lane, const uint32_t rank_mul, const QueensRowConsts& rc) {
    do {
        queens_trip<L, LVL, JUP, true>(S, bbase, lane, rank_mul, rc);
        if constexpr (LVL + 1 < L) {
            if (S.cnt[LVL + 1] >= 64u) queens_run_from<L, LVL + 1, JUP>(S, bbase, lane, rank_mul, rc);
        }
    } while (S.cnt[LVL] >= 64u);
}

template <int L, int JUP>
__global__ void __launch_bounds__(kQueensBucketMaxWarps * 32)
k_queens_bucket_t(QueensLaneArgs A) {
    static_assert(L >= 1 && L <= 8, "one count register per bucket");
    extern __shared__ uint4 qb_frames[];
    const uint32_t lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t rank_mul = lane ? 1u << (32u - lane) : 0u;
    const uint32_t hi = ~((1u << A.n) - 1u);
    constexpr uint32_t per_warp = (uint32_t)L * kQueensBucketCap * 16u;
    const uint32_t bbase = (uint32_t)__cvta_generic_to_shared(qb_frames) + wib * per_warp;
    uint32_t pf_n = 0;                                           // records prefetched into pf0 / pf1 (in flight or landed)
    uint4 pf0 = make_uint4(0u, 0u, 0u, 0u), pf1 = pf0;
    const unsigned long long n_found = *A.n_records;
    const unsigned long long n_rec = n_found < A.record_cap ? n_found : A.record_cap;   // overflow: the host grows the list and reruns
    const unsigned long long total_warps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    const uint32_t fair_share = (uint32_t)min((n_rec + total_warps - 1) / total_warps, 64ull);
    QueensTripState S;
#pragma unroll
    for (int i = 0; i < 8; i++) S.cnt[i] = 0u;
    S.trip_nodes = 0ull; S.tot_sols = 0ull; S.tot_lane_nodes = 0ull;
    QueensRowConsts rc;
    const uint32_t zero = (uint32_t)A.n >> 8;                    // 0, but not to the compiler
#pragma unroll
    for (int j = 0; j < 10; j++) { rc.pow[j] = (1u << j) + zero; rc.ones[j] = rc.pow[j] - 1u; }
    unsigned long long chunk_pos = 0, chunk_end = 0;
    bool exhausted = false;

    QueensRecordRegs R = {0xFFFFFFFFu, 0u, 0u, 0u, 0xFFFFFFFFu, 0u, 0u, 0u};
    // claims the next chunk of the record list if need be and starts the loads of up to 64 records of it: they
    // stay in flight (two uint4 registers per lane) while the warp works through the records it has
    auto prefetch = [&]() {
        if (exhausted) return;
        if (chunk_pos >= chunk_end) {
            unsigned long long base = 0;
            uint32_t size = 0;
            if (lane == 0) {
                const unsigned long long cur = *(volatile unsigned long long*)A.cursor;
                const unsigned long long remaining = cur < n_rec ? n_rec - cur : 0;
                size = (uint32_t)min(max(remaining / (4ull * total_warps), (unsigned long long)max(fair_share, 1u)), 256ull);
                base = atomicAdd(A.cursor, (unsigned long long)size);
            }
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            size = __shfl_sync(0xFFFFFFFFu, size, 0);
            chunk_pos = base;
            chunk_end = min(base + size, n_rec);
            if (base >= n_rec) { exhausted = true; chunk_end = chunk_pos; return; }
        }
        pf_n = (uint32_t)min(chunk_end - chunk_pos, 64ull);
        if (lane < pf_n) pf0 = __ldg(A.records + chunk_pos + lane);
        if (lane + 32u < pf_n) pf1 = __ldg(A.records + chunk_pos + lane + 32);
        chunk_pos += pf_n;
    };
    prefetch();
    for (;;) {
        // (here no bucket holds 64 frames)
        if (!__any_sync(0xFFFFFFFFu, (R.cA | R.cB) != 0u)) {
            // the warp's records are spent: the next 64 (already loaded), and the loads of the 64 after them
            if (pf_n == 0u) prefetch();
            if (pf_n == 0u) break;                               // the list is spent as well
            R.aA = 0xFFFFFFFFu; R.cA = 0u; R.aB = 0xFFFFFFFFu; R.cB = 0u;
            if (lane < pf_n) { R.aA = pf0.y | hi; R.lA = pf0.z; R.rA = pf0.w; R.cA = ~(R.aA | R.lA | R.rA); }
            if (lane + 32u < pf_n) { R.aB = pf1.y | hi; R.lB = pf1.z; R.rB = pf1.w; R.cB = ~(R.aB | R.lB | R.rB); }
            S.tot_lane_nodes += __popc(R.cA) + __popc(R.cB);
            pf_n = 0;
            prefetch();
            continue;
        }
        queens_record_trip<L, JUP>(S, R, bbase, rank_mul, rc);
        if (S.cnt[0] >= 64u) queens_run_from<L, 0, JUP>(S, bbase, lane, rank_mul, rc);
    }
    for (;;) {
        // The record list is spent: the deepest bucket that holds 64 frames, else the shallowest that holds anything
        // (short trips; this is the tail of the warp's work).
        int lvl = -1;
#pragma unroll
        for (int v = L - 1; v >= 0; v--) if (lvl < 0 && S.cnt[v] >= 64u) lvl = v;
        if (lvl < 0) {
#pragma unroll
            for (int v = 0; v < L; v++) if (lvl < 0 && S.cnt[v] != 0u) lvl = v;
        }
        if (lvl < 0) break;
        switch (lvl) {
#define DQ_QTRIP(V) case V: if constexpr (V < L) queens_trip<L, V, JUP, false>(S, bbase, lane, rank_mul, rc); break;
            DQ_QTRIP(0) DQ_QTRIP(1) DQ_QTRIP(2) DQ_QTRIP(3) DQ_QTRIP(4) DQ_QTRIP(5) DQ_QTRIP(6) DQ_QTRIP(7)
#undef DQ_QTRIP
            default: break;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        S.tot_sols += __shfl_down_sync(0xFFFFFFFFu, S.tot_sols, o);
        S.tot_lane_nodes += __shfl_down_sync(0xFFFFFFFFu, S.tot_lane_nodes, o);
    }
    if (lane == 0) {
        atomicAdd(A.totals + 0, S.tot_sols);
        atomicAdd(A.dfs_nodes, S.tot_sols + S.tot_lane_nodes + S.trip_nodes);
    }
}

}  // namespace dq
