// dq_warp_engine.cuh — generic warp-cooperative forward-checking DFS (sm_100a).
//
// One warp owns one search tree (a prefix subtree of a single model, or one instance of a
// batch).  It replaces, for that tree, the reference's recursive
//   CSP::ForwardCheckingStep (dequan.h:494-571)  -> explicit stack: cand[]/mark[]/val[] per depth
//   OpConstraint/AllDifferent/Equality::AplyArcConsistency (631-694, 915-939, 710-743)
//                                                -> fc_apply(): each lane filters ONE neighbour's
//                                                   domain word with AND/ANDNOT masks; wipe-out is a
//                                                   warp vote
//   Domain::Exclude/Intersect/ExcludeInf/Sup (957-1172) -> bit masks on a 32-bit domain word
//   EnsureSavedDomain / RestoreSavedDomainStep (431-452) -> warp-appended trail in shared memory
//   ValidateVarConstraints (573-587)             -> the F ("fails validation") word per variable
//
// A node is one AssignVar call (dequan.h:416-423): every value of the current domain of the
// next variable, including values whose validation or forward check then fails.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace dq {

// entry word layout — keep in sync with dq_model.hpp
constexpr uint32_t D_K_NE_SAME = 0, D_K_AND = 1, D_K_WEQ = 2, D_K_CHK = 3;
constexpr uint32_t D_Q_MASK = 0xFFFFu;
constexpr int D_KIND_SHIFT = 16;
constexpr uint32_t D_FORCE_D = 1u << 18, D_FORCE_F = 1u << 19, D_NOTRAIL_D = 1u << 20, D_NOTRAIL_F = 1u << 21,
                   D_SKIP = 1u << 22, D_FIRST = 1u << 23;
constexpr uint32_t FULL = 0xFFFFFFFFu;
constexpr uint32_t TRAIL_F = 0x8000;  // trail entry refers to F[q], not D[q]

// Domain word: 32 bits, or 64 for models whose largest domain has 33..64 values (single-tree solves only).
__device__ __forceinline__ int dq_ffs(uint32_t x) { return __ffs((int)x); }
__device__ __forceinline__ int dq_ffs(unsigned long long x) { return __ffsll((long long)x); }
__device__ __forceinline__ int dq_popc(uint32_t x) { return __popc(x); }
__device__ __forceinline__ int dq_popc(unsigned long long x) { return __popcll(x); }

// Read-only model tables (HBM, read through L1 with ld.global.nc)
template <typename W>
struct DevTablesT {
    int nv;
    const uint32_t* __restrict__ ent_off;   // [nv+1]
    const uint32_t* __restrict__ ent;       // [n_ent]
    const uint32_t* __restrict__ ent_moff;  // [n_ent]
    const W* __restrict__ masks;
};
typedef DevTablesT<uint32_t> DevTables;

// Per-warp mutable state, all in shared memory
template <typename W>
struct WarpStateT {
    W* D;             // [nv] current domain bits            (Assignment::current_domains)
    W* F;             // [nv] values that will fail Evaluate (only if HAS_F)
    W* cand;          // [nv] untried values per depth
    W* told;          // [trail] saved words                 (Assignment::saved_domains)
    uint16_t* tq;     // [trail] which word
    uint16_t* mark;   // [nv] trail height per depth
    uint8_t* val;     // [nv] chosen value index per depth   (Assignment::inst_vars)
    uint16_t* order;  // [nv] depth -> var                   (Assignment::assign_order)
    uint16_t* pos;    // [nv] var -> depth
};
typedef WarpStateT<uint32_t> WarpState;

__host__ __device__ inline size_t warp_state_bytes(int nv, int trail, int word_bytes = 4) {
    size_t nvp = (size_t)((nv + 3) & ~3);
    size_t tp = (size_t)((trail + 3) & ~3);
    return (nvp * word_bytes * 3 + tp * word_bytes + tp * 2 + nvp * 2 + nvp * 5 + 15) & ~(size_t)15;   // the next warp's block stays 16-byte aligned
}

template <typename W>
__device__ inline WarpStateT<W> carve_warp_state_t(unsigned char* base, int nv, int trail) {
    size_t nvp = (size_t)((nv + 3) & ~3);
    size_t tp = (size_t)((trail + 3) & ~3);
    WarpStateT<W> s;
    s.D = (W*)base;                  base += nvp * sizeof(W);
    s.F = (W*)base;                  base += nvp * sizeof(W);
    s.cand = (W*)base;               base += nvp * sizeof(W);
    s.told = (W*)base;               base += tp * sizeof(W);
    s.tq = (uint16_t*)base;          base += tp * 2;
    s.mark = (uint16_t*)base;        base += nvp * 2;
    s.order = (uint16_t*)base;       base += nvp * 2;
    s.pos = (uint16_t*)base;         base += nvp * 2;
    s.val = base;
    return s;
}
__device__ inline WarpState carve_warp_state(unsigned char* base, int nv, int trail) { return carve_warp_state_t<uint32_t>(base, nv, trail); }

struct DfsResult {
    unsigned long long nodes;
    unsigned long long sols;
    int outcome;        // dq_outcome
    bool have_first;    // val[0..nv) holds a solution (value indices by depth)
};

// Undo the trail down to `mk` (RestoreSavedDomainStep, dequan.h:431-440).
template <bool HAS_F, typename W>
__device__ __forceinline__ void trail_undo(const WarpStateT<W>& S, int mk, int& top, int lane) {
    for (int i = mk + lane; i < top; i += 32) {
        uint32_t t = S.tq[i];
        if (HAS_F && (t & TRAIL_F)) S.F[t & 0x7FFF] = S.told[i];
        else S.D[t] = S.told[i];
    }
    top = mk;
    __syncwarp();
}

// Forward-check the assignment x = value index b made at depth d.  Returns true on a domain
// wipe-out of some unassigned neighbour.  Domain changes are trailed above `top`.
template <bool HAS_F, bool HAS_TABLE, typename W>
__device__ __forceinline__ bool fc_apply(const DevTablesT<W>& T, const WarpStateT<W>& S, int x, int b, int d, int& top, int lane) {
    const int e0 = (int)__ldg(T.ent_off + x), e1 = (int)__ldg(T.ent_off + x + 1);
    const uint32_t lt = (1u << lane) - 1u;
    bool wiped = false;
    for (int base = e0; base < e1; base += 32) {
        const int e = base + lane;
        uint32_t w = e < e1 ? __ldg(T.ent + e) : D_SKIP;
        const int q = (int)(w & D_Q_MASK);
        bool act = !(w & D_SKIP);
        if (act) act = S.pos[q] > d;                      // only unassigned neighbours are filtered
        W oldD = 0, newD = 0, oldF = 0, newF = 0;
        if (act) {
            oldD = S.D[q];
            newD = oldD;
            if (HAS_F) { oldF = S.F[q]; newF = oldF; }
            const uint32_t kind = (w >> D_KIND_SHIFT) & 3;
            if (!HAS_TABLE || kind == D_K_NE_SAME) newD = oldD & ~(W(1) << b);
            else {
                const W m = __ldg(T.masks + __ldg(T.ent_moff + e) + b);
                if (kind == D_K_AND) {
                    if (w & D_FIRST) { const W t = oldD & m; newD = oldD & ~(t & (W(0) - t)); }   // erase the first match only (duplicate values)
                    else newD = oldD & m;
                } else if (HAS_F) {
                    // Domain::Intersect(val) leaves ONE copy of val (dequan.h:957-984), or the domain alone if val is absent
                    if (kind == D_K_WEQ) { const W t = oldD & m; if (t) newD = t & (W(0) - t); else newF = ~W(0); }
                    else newF = oldF | m;
                }
            }
        }
        const bool tD = act && (newD != oldD || (w & D_FORCE_D)) && !(w & D_NOTRAIL_D);
        const uint32_t mD = __ballot_sync(FULL, tD);
        if (tD) { const int i = top + __popc(mD & lt); S.tq[i] = (uint16_t)q; S.told[i] = oldD; }
        top += __popc(mD);
        if (act && newD != oldD) S.D[q] = newD;
        if (HAS_F) {
            const bool tF = act && (newF != oldF || (w & D_FORCE_F)) && !(w & D_NOTRAIL_F);
            const uint32_t mF = __ballot_sync(FULL, tF);
            if (tF) { const int i = top + __popc(mF & lt); S.tq[i] = (uint16_t)(q | TRAIL_F); S.told[i] = oldF; }
            top += __popc(mF);
            if (act && newF != oldF) S.F[q] = newF;
        }
        wiped |= act && newD == 0;
        __syncwarp();
    }
    return __any_sync(FULL, wiped);
}

// Bit index of the n-th (1-based) set bit of x, which has at least n.
template <typename W>
__device__ __forceinline__ int dq_nth_bit(W x, int n) {
    for (; n > 1; --n) x &= x - 1;
    return dq_ffs(x) - 1;
}

// Explicit-stack DFS from depth d0 (domains already reflect the d0 assignments above it).
//   count_all : walk the whole subtree (solutions + nodes); else stop at the DFS-first solution.
//   budget    : stop once more than `budget` nodes have been counted (0 = none), outcome DQ_BUDGET.
//   abort_key / my_key : FIRST-mode prefix search — give up when another warp has recorded a solution
//                in an earlier prefix (abort_key may be null).
//   LIMITED (count_all only): the counting constraint passes the `limit`-th solution (0 = none), so the search stops
//                there with outcome DQ_SAT; the node count stops at that value or at node budget + 1 also inside the
//                last level, where the plain count adds the whole level before it tests the budget.
template <bool HAS_F, bool HAS_TABLE, bool LIMITED = false, typename W, class OnFirst>
__device__ DfsResult warp_dfs(const DevTablesT<W>& T, const WarpStateT<W>& S, int d0, bool count_all,
                              unsigned long long budget, const unsigned long long* abort_key,
                              unsigned long long my_key, int lane, OnFirst on_first, unsigned long long limit = 0) {
    const int nv = T.nv;
    DfsResult R;
    R.nodes = 0; R.sols = 0; R.outcome = 0; R.have_first = false;
    if (d0 >= nv) { R.sols = 1; R.outcome = 1; R.have_first = true; return R; }   // IsComplete, dequan.h:496-499
    int top = 0, d = d0;
    int x = S.order[d];
    W c = S.D[x];
    unsigned poll = 0;
    for (;;) {
        if (c == 0) {                                     // every value tried: return false (dequan.h:569-570)
            if (d == d0) break;
            --d;
            x = S.order[d];
            trail_undo<HAS_F>(S, S.mark[d], top, lane);
            c = S.cand[d];
            continue;
        }
        if (abort_key && ((++poll & 63u) == 0) && *(volatile const unsigned long long*)abort_key < my_key) { R.outcome = 3; break; }
        if (d == nv - 1) {
            // last variable: each remaining value is a node; valid ones are solutions, no filtering left to do
            const W valid = HAS_F ? (c & ~S.F[x]) : c;
            if (LIMITED) {
                W reach = c;                              // the values of this level the search visits
                if (limit && (unsigned long long)dq_popc(valid) >= limit - R.sols) {
                    const int b = dq_nth_bit(valid, (int)(limit - R.sols));
                    reach = c & ((W(2) << b) - W(1));     // ... up to the one that completes the limit-th solution
                }
                if (budget && R.nodes + dq_popc(reach) > budget) {
                    const int b = dq_nth_bit(c, (int)(budget - R.nodes) + 1);
                    reach = c & ((W(1) << b) - W(1));     // ... before node budget + 1
                    R.outcome = 2;
                }
                const W got = valid & reach;
                R.nodes = R.outcome == 2 ? budget + 1 : R.nodes + dq_popc(reach);
                if (got) on_first.solutions(S, got, R.sols);
                if (got && !R.have_first) {
                    R.have_first = true;
                    if (lane == 0) S.val[d] = (uint8_t)(dq_ffs(got) - 1);
                    __syncwarp();
                    on_first(S);
                }
                R.sols += dq_popc(got);
                if (R.outcome == 2) break;
                if (limit && R.sols == limit) { R.outcome = 1; break; }
                c = 0;
                continue;
            }
            if (count_all) {
                R.nodes += dq_popc(c);
                if (budget && R.nodes > budget) { R.outcome = 2; break; }
                if (valid) on_first.solutions(S, valid, R.sols);
                R.sols += dq_popc(valid);
                if (valid && !R.have_first) {
                    // first solution of this tree: val[] is the assignment right now (count_all keeps searching)
                    R.have_first = true;
                    if (lane == 0) S.val[d] = (uint8_t)(dq_ffs(valid) - 1);
                    __syncwarp();
                    on_first(S);
                }
                c = 0;
                continue;
            }
            if (valid) {
                const int b = dq_ffs(valid) - 1;
                unsigned long long n = dq_popc(c & ((W(2) << b) - W(1)));
                if (budget && R.nodes + n > budget) {
                    R.nodes = budget + 1; R.outcome = 2; break;
                }
                R.nodes += n;
                if (lane == 0) S.val[d] = (uint8_t)b;
                __syncwarp();
                R.sols = 1; R.outcome = 1; R.have_first = true;
                break;
            }
            if (budget && R.nodes + dq_popc(c) > budget) { R.nodes = budget + 1; R.outcome = 2; break; }
            R.nodes += dq_popc(c);
            c = 0;
            continue;
        }
        const int b = dq_ffs(c) - 1;
        c &= c - 1;
        ++R.nodes;                                        // AssignVar, dequan.h:416-423
        if (budget && R.nodes > budget) { R.outcome = 2; break; }
        if (HAS_F && ((S.F[x] >> b) & 1u)) continue;      // ValidateVarConstraints fails, dequan.h:535-538
        const int mk = top;
        if (fc_apply<HAS_F, HAS_TABLE>(T, S, x, b, d, top, lane)) { trail_undo<HAS_F>(S, mk, top, lane); continue; }
        if (lane == 0) { S.mark[d] = (uint16_t)mk; S.cand[d] = c; S.val[d] = (uint8_t)b; }
        ++d;
        __syncwarp();
        x = S.order[d];
        c = S.D[x];
    }
    if (count_all && R.outcome != 2) R.outcome = R.sols ? 1 : 0;
    return R;
}

}  // namespace dq
