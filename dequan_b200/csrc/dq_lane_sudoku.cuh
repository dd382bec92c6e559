// dq_lane_sudoku.cuh — batches of 9x9 Sudoku on B200 (CLASS_SUDOKU9: 81 variables on 1..9,
// NotEqual/AllDifferent over the 27 rows, columns and boxes — BASELINE config C3, recognised by
// the model compiler whatever mix of binary != and AllDifferent rows produced it).
//
// What the reference does per node (CSP::ForwardCheckingStep dequan.h:494-571 with
// OpConstraint/AllDifferent::AplyArcConsistency 631-694, 915-939 and Domain::Exclude 985-1031)
// collapses, for this model class, to a closed form: the current domain of an unassigned cell is
//     {1..9} minus the values assigned in its row, its column and its box
// so the whole search state of one instance is 27 nine-bit "used" masks.  Undo on backtrack
// (RestoreSavedDomainStep, dequan.h:431-440) is clearing one bit in three masks; there is no trail.
//
// Static order (Assignment::Reset, dequan.h:376-394): givens first (domain size 1) by id, then the
// blanks by id.  A node is an AssignVar call (dequan.h:416-423): one per given, then one per value
// tried at a blank.  Assigning value v at cell p passes its forward check unless some LATER blank
// peer q is left with no value, i.e. unless dom(q) == {v}.  Cells are packed three to a word
// (10-bit fields, one word per (row, stack) = one box-row), so "which values of p are forbidden by
// a later peer" is a handful of packed-field operations per peer word (sk_singletons).
//
// Lane engine: every lane owns one search; its masks, blank-field masks and DFS stack live in
// shared memory as [word][thread], bank-conflict-free whatever each lane indexes.  A level is
// entered once (domain + forbidden values in one pass); failing values are never stepped through,
// only counted when the search moves past them.
//
// Pipeline for a batch (all on one stream, no host round trip in between):
//   k_sudoku_digest  one thread per instance: working tables of the givens, coalesced.
//   k_sudoku_first   lane per instance: the reference's search, up to `first_budget` nodes.  Node
//                    counts are heavy-tailed (30 givens: median 363, max > 1e6) and a lane is slow,
//                    so an instance that is not done by then is put on the HARD list instead.
//   k_sudoku_strong  warp per hard instance: finds the solution the reference would return — the
//                    lexicographically first one in (blank order, ascending values), SURVEY.md §9
//                    S5 — by the same static-order DFS with naked-single propagation to a fixed
//                    point.  Sound extra pruning never changes WHICH solution is first, only how
//                    many nodes it takes to get there (a few hundred instead of up to 1e6).
//   k_sudoku_walk    lane per hard instance: walks the solution path and counts what the
//                    reference's plain forward-checking search visits on the way: at every path
//                    level the values tried up to the solution's (nodes), and for each of those
//                    that passes its forward check a ROOT TASK = "count the whole subtree below it".
//   k_sudoku_count   lanes take root tasks from a queue and count their subtrees exhaustively.
//                    Every one of those nodes is a node of the reference's search, so there is no
//                    speculative work; lanes that run dry raise a hunger count and busy lanes hand
//                    over their shallowest stack level with untried values (the largest subtree
//                    they own) as a new task.  Sums go to nodes[instance] with atomicAdd.
//   k_sudoku_finish  API node budget on the exact totals, batch totals.
// Instances with clashing givens or foreign bytes are handed to the generic warp engine.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "dq_group_graphs.cuh"     // bulk-copy / mbarrier primitives

namespace dq {

constexpr int kSudokuBlock = 128;               // threads per CTA
constexpr uint32_t SK_ONES = 0x00100401u;       // 1 in each of the three 10-bit fields
constexpr uint32_t SK_SPARE = 0x20080200u;      // bit 9 of each field
constexpr uint32_t SK_FULL3 = 0x1FF7FDFFu;      // 0x1FF in each field
constexpr uint8_t SK_STATUS_HARD = 0xFD;        // interim: on the hard list
constexpr uint8_t SK_STATUS_DEFER = 0xFE;       // interim: handed to the generic warp engine

// Per-instance record written by k_sudoku_digest and copied into shared memory by the lane that
// takes the instance: everything the search needs, already in its working layout (18 x uint4).
//   w[0..2]   blank bitmap by cell id (81 bits, row-major)
//   w[3]      bit 31 = deferred to the generic engine; low byte = number of blanks
//   w[4..6]   rows' used masks, one band per word, one row per 10-bit field
//   w[7..9]   columns' used masks, one stack per word, one column per field
//   w[10..18] boxes' used masks, replicated in the three fields
//   w[19..45] per (row, stack): 0x1FF in the fields of blank cells
//   w[46..66] the blank cells' ids in search order, one byte per level
//   w[67..69] blank bitmap transposed (bit 9*column + row)
constexpr int kDigestVec = 18;
constexpr int kTableWords = 63;                 // w[4..66]: copied verbatim into the lane's shared-memory tables
struct SudokuDigest { uint4 v[kDigestVec]; };

// One unit of counting work (16 bytes).
//   root task : count the subtree below "path values at levels < level, then `value` at `level`"
//   piece     : a range of stack levels [lo, hi] of a donor's snapshot
// `info` is written LAST by whoever publishes the task; 0 = not published yet.
struct SudokuTask {
    uint32_t puzzle;
    uint32_t snap_id;          // piece: which stack snapshot it resumes from
    uint32_t info;             // bit 31 valid | bit 30 root | bit 29 null | bit 28 top ; root: level | value << 8 ; piece: lo | hi << 8
                               // (top: hi is the level the snapshot's search stood on; its untried sets are entries hi, hi+1)
    uint32_t pad;
};
constexpr uint32_t SKT_VALID = 0x80000000u, SKT_ROOT = 0x40000000u, SKT_NULL = 0x20000000u, SKT_TOP = 0x10000000u;
constexpr int kSnapWords = 12;                  // uint4 per stack snapshot: 96 u16 entries (passing untried | value << 9) per level

// Control block (unsigned long long words)
enum SkCtrl { SKC_FRESH = 0,        // k_sudoku_first: next fresh instance
              SKC_HARD = 1,         // instances on the hard list
              SKC_HARD_CUR = 2,     // k_sudoku_strong / k_sudoku_walk cursors over the hard list
              SKC_WALK_CUR = 3,
              SKC_RESERVE = 4,      // tasks reserved (root tasks by the walker, pieces by donors)
              SKC_SNAP = 5,         // snapshots reserved
              SKC_HEAD = 6,         // tickets drawn by consumers (may run ahead of SKC_RESERVE: lanes waiting for work)
              SKC_OUTSTANDING = 7,  // tasks published and not finished yet
              SKC_MAX_BLANK = 8,    // k_sudoku_digest: the most blanks any instance of the batch has (sizes the lanes' stacks)
              SKC_ERROR = 9,        // bit 0: a warp gave up waiting; bit 1: task pool overflow; bit 2: a counted subtree held a solution
              SKC_TOTALS = 12 };    // [12..15] sat, unsat, budget, nodes

struct SudokuArgs {
    const SudokuDigest* digest;
    long long n;                           // instances
    int stride;
    const uint8_t* cells;                  // [n][stride] givens
    uint8_t* solution;                     // [n][stride]
    unsigned long long* nodes;             // [n]
    uint8_t* status;                       // [n]
    uint32_t* hard;                        // [n][2] instances k_sudoku_first did not finish: {id, snapshot slot | stack level << 24}
    SudokuTask* tasks;    unsigned long long task_cap;
    uint4* snaps;         unsigned long long snap_cap;       // kSnapWords x uint4 per snapshot
    uint32_t* snap_state;                  // [snap_cap] 1 while a snapshot is waiting for the task that resumes from it (the pool is a ring)
    unsigned long long* ctrl;              // control block, see SkCtrl
    unsigned long long user_budget;        // per-instance node budget of the API (0 = none)
    unsigned first_budget;                 // nodes k_sudoku_first spends on an instance before calling it hard
    int stack_levels;                      // the most blanks any instance of the batch has: levels of the lanes' (and k_sudoku_strong's) stacks
    unsigned force_donate;                 // test knob: donate whenever a task is this many nodes old, hungry lanes or not (0 = off)
};

// ---------------------------------------------------------------------------------------------
// Pass 0: one thread per instance, persistent CTAs over tiles of 128 instances.  The 81-byte cell rows of a tile are
// one contiguous 10 368-byte span: a single bulk copy (cp.async.bulk + mbarrier) brings it into shared memory while
// the previous tile is being digested (two staging buffers); the 128 finished 288-byte records are assembled in shared
// memory and leave with one 36 864-byte bulk store.  (A ragged last tile, a stride other than 81 or a misaligned
// batch go through plain loads and stores.)
constexpr int kDigestTile = 128;
constexpr int kDigestInBytes = kDigestTile * 81;                 // 16 x 648
constexpr int kDigestOutBytes = kDigestTile * kDigestVec * 16;   // 36 864
constexpr int kDigestSmem = 2 * kDigestInBytes + kDigestOutBytes + 16;

__global__ void __launch_bounds__(kDigestTile)
k_sudoku_digest(const uint8_t* __restrict__ cells, long long n, int stride, SudokuDigest* __restrict__ out, unsigned long long* __restrict__ max_blank) {
    extern __shared__ __align__(128) uint8_t dg_raw[];           // in[2][10368] | records[128][288] | two mbarriers
    uint8_t* recs = dg_raw + 2 * kDigestInBytes;
    const uint32_t in_s = smem_u32(dg_raw), recs_s = smem_u32(recs), mbar = recs_s + kDigestOutBytes;
    const long long tiles = (n + kDigestTile - 1) / kDigestTile;
    const bool bulk_ok = stride == 81 && ((size_t)cells & 15) == 0 && ((size_t)out & 15) == 0;
    if (threadIdx.x == 0) { mbar_init(mbar, 1); mbar_init(mbar + 8, 1); mbar_init_fence(); }
    __syncthreads();
    auto full = [&](long long t) { return bulk_ok && (t + 1) * kDigestTile <= n; };
    auto issue = [&](long long t, int b) {                       // (thread 0) the whole tile in one copy
        mbar_expect_tx(mbar + 8 * b, kDigestInBytes);
        bulk_g2s(in_s + b * kDigestInBytes, cells + t * kDigestInBytes, kDigestInBytes, mbar + 8 * b);
    };
    uint32_t parity = 0;
    int b = 0;
    int most_blanks = 0;
    long long t = blockIdx.x;
    if (t < tiles && full(t) && threadIdx.x == 0) issue(t, 0);
    bool store_in_flight = false;
    for (; t < tiles; t += gridDim.x, b ^= 1) {
        const long long nxt = t + gridDim.x;
        if (nxt < tiles && full(nxt) && threadIdx.x == 0) issue(nxt, b ^ 1);
        const long long first = t * kDigestTile;
        const int here = (int)min((long long)kDigestTile, n - first);
        uint8_t* stage = dg_raw + b * kDigestInBytes;
        if (full(t)) { mbar_wait(mbar + 8 * b, (parity >> b) & 1u); parity ^= 1u << b; }
        else {
            for (int i = threadIdx.x; i < here * 81; i += kDigestTile) stage[i] = cells[(first + i / 81) * stride + i % 81];
            __syncthreads();
        }
        if (store_in_flight) {                                   // the previous tile's records have left shared memory
            if (threadIdx.x == 0) bulk_wait_read0();
            __syncthreads();
            store_in_flight = false;
        }
        if ((int)threadIdx.x < here) {
            const uint8_t* g = stage + threadIdx.x * 81;
            uint32_t row[9], col[9], box[9], blank[3] = {0, 0, 0};
#pragma unroll
            for (int i = 0; i < 9; i++) { row[i] = 0; col[i] = 0; box[i] = 0; }
            bool defer = false;
#pragma unroll
            for (int r = 0; r < 9; r++)
#pragma unroll
                for (int c = 0; c < 9; c++) {
                    const int p = r * 9 + c;
                    const uint32_t v = g[p];
                    if (v == 0) { blank[p >> 5] |= 1u << (p & 31); continue; }
                    if (v > 9) { defer = true; continue; }           // not a value of the template domain
                    const uint32_t bit = 1u << (v - 1);
                    const int bx = (r / 3) * 3 + c / 3;
                    if ((row[r] | col[c] | box[bx]) & bit) defer = true;   // two givens clash: the exact node count is the generic engine's job
                    row[r] |= bit; col[c] |= bit; box[bx] |= bit;
                }
            uint32_t w[kDigestVec * 4];
#pragma unroll
            for (int i = 0; i < kDigestVec * 4; i++) w[i] = 0;
            int level = 0;
#pragma unroll
            for (int r = 0; r < 9; r++)
#pragma unroll
                for (int c = 0; c < 9; c++) {
                    const int p = r * 9 + c;
                    if (!((blank[p >> 5] >> (p & 31)) & 1u)) continue;
                    if ((row[r] | col[c] | box[(r / 3) * 3 + c / 3]) == 0x1FFu) defer = true;  // a blank wiped out by the givens
                    w[19 + r * 3 + c / 3] |= 0x1FFu << (10 * (c % 3));
                    w[67 + (c * 9 + r) / 32] |= 1u << ((c * 9 + r) % 32);
                    ++level;
                }
            w[0] = blank[0]; w[1] = blank[1]; w[2] = blank[2];
            w[3] = (uint32_t)level | (defer ? 0x80000000u : 0u);
            most_blanks = max(most_blanks, level);
#pragma unroll
            for (int i = 0; i < 9; i++) w[10 + i] = box[i] * SK_ONES;
#pragma unroll
            for (int i = 0; i < 3; i++) {
                w[4 + i] = row[3 * i] | (row[3 * i + 1] << 10) | (row[3 * i + 2] << 20);
                w[7 + i] = col[3 * i] | (col[3 * i + 1] << 10) | (col[3 * i + 2] << 20);
            }
            uint32_t* rw = reinterpret_cast<uint32_t*>(recs + threadIdx.x * (kDigestVec * 16));
#pragma unroll
            for (int i = 0; i < kDigestVec * 4; i++) rw[i] = w[i];           // (w[46..66] are zero here)
            // cell id of every search level, one byte per level: the set bits of the blank bitmap in ascending order,
            // written straight into the record (the 81 x __fns of the all-register version were most of this pass)
            uint8_t* tab = recs + threadIdx.x * (kDigestVec * 16) + 46 * 4;
            int L = 0;
#pragma unroll
            for (int k = 0; k < 3; k++)
                for (uint32_t bits = blank[k]; bits; bits &= bits - 1u) tab[L++] = (uint8_t)(32 * k + __ffs((int)bits) - 1);
        }
        if (full(t)) {
            fence_async_smem();
            __syncthreads();
            if (threadIdx.x == 0) { bulk_s2g(out + first, recs_s, kDigestOutBytes); bulk_commit(); }
            store_in_flight = true;
        } else {
            __syncthreads();
            const uint4* src = reinterpret_cast<const uint4*>(recs);
            uint4* dst = reinterpret_cast<uint4*>(out + first);
            for (int i = threadIdx.x; i < here * kDigestVec; i += kDigestTile) dst[i] = src[i];
            __syncthreads();
        }
    }
    if (store_in_flight && threadIdx.x == 0) bulk_wait_read0();
    most_blanks = __reduce_max_sync(0xFFFFFFFFu, most_blanks);
    if ((threadIdx.x & 31) == 0 && most_blanks) atomicMax(max_blank, (unsigned long long)most_blanks);
}

// ---------------------------------------------------------------------------------------------
// Per-lane shared-memory state, all arrays [word][thread].
struct SudokuSmem {
    uint32_t rowp[3][kSudokuBlock];     // row used masks of one band, one row per field
    uint32_t colp[3][kSudokuBlock];     // column used masks of one stack, one column per field
    uint32_t boxr[9][kSudokuBlock];     // box used mask, replicated
    uint32_t blk[27][kSudokuBlock];     // (row, stack) -> 0x1FF in the fields of blank cells
    uint32_t cellw[21][kSudokuBlock];   // blank cell ids in search order, four levels per word
    uint16_t stk[81][kSudokuBlock];     // per level: passing values not tried yet | chosen value index << 9
                                        // (LAST member: a batch whose instances have at most B blanks launches with B levels of it)
};

__device__ __forceinline__ uint32_t sk_rep(uint32_t x9) { return x9 * SK_ONES; }

struct SkCell { int r, s, f, band, box, rm; };    // row, stack, column in stack, band, box, row in band
__device__ __forceinline__ SkCell sk_decode(int p) {
    SkCell c;
    c.r = (p * 57) >> 9;                 // p / 9 for p < 81
    const int col = p - 9 * c.r;
    c.s = (col * 11) >> 5;               // col / 3 for col < 9
    c.f = col - 3 * c.s;
    c.band = (c.r * 11) >> 5;            // r / 3
    c.box = c.band * 3 + c.s;
    c.rm = c.r - 3 * c.band;
    return c;
}

// Packed fields x (three 9-bit sets): keeps the fields that hold exactly one value, clears the rest.
// A later blank peer whose domain is a single value forbids that value here: taking it would wipe
// the peer out (the wipe-out test of OpConstraint::AplyArcConsistency, dequan.h:663-668).
__device__ __forceinline__ uint32_t sk_singletons(uint32_t x) {
    const uint32_t y = x + (SK_SPARE - SK_ONES);            // per field x - 1, the spare bit absorbs the borrow of an empty field
    const uint32_t z = x & y;                               // x & (x - 1): zero iff the field holds at most one value
    const uint32_t tt = z + (SK_SPARE - SK_ONES);           // spare bit survives iff z != 0
    const uint32_t nz = ~tt & SK_SPARE;
    return x & (nz - (nz >> 9));                            // 0x1FF in the fields with z == 0
}

// ---------------------------------------------------------------------------------------------
// Per-lane search state (registers) and the three steps every lane kernel is built from.
struct SkLane {
    bool have, enter;
    uint32_t puzzle;
    int p;                      // current cell
    SkCell c;                   // ... decoded
    int sp, base_sp, nblank;    // stack level of the current cell; the task's root level; blanks in the instance
    uint32_t passrem;           // values of the current cell that pass the forward check and are not tried yet
    uint32_t dom_rem;           // values of the current cell not tried yet, passing or not
    uint32_t nodes;             // nodes counted by this task
    unsigned long long nodes_hi;
};

__device__ __forceinline__ int sk_cell_at(const SudokuSmem& S, int t, int l) { return (int)((S.cellw[l >> 2][t] >> ((l & 3) * 8)) & 0xFF); }
__device__ __forceinline__ uint32_t sk_used_at(const SudokuSmem& S, int t, const SkCell& k) {
    return ((S.rowp[k.band][t] >> (10 * k.rm)) | (S.colp[k.s][t] >> (10 * k.f)) | S.boxr[k.box][t]) & 0x1FF;
}
__device__ __forceinline__ void sk_commit(SudokuSmem& S, int t, const SkCell& k, uint32_t bit) {
    S.rowp[k.band][t] |= bit << (10 * k.rm);
    S.boxr[k.box][t] |= sk_rep(bit);
    S.colp[k.s][t] |= bit << (10 * k.f);
}

// words 4..66 of the digest record -> rowp, colp, boxr, blk, cellw (contiguous in S)
__device__ __forceinline__ void sk_load_tables(SudokuSmem& S, int t, const uint4* __restrict__ dg) {
    uint32_t* dst = &S.rowp[0][t];
#pragma unroll
    for (int q = 1; q < kDigestVec; q++) {
        const uint4 x = __ldg(dg + q);
        const int wbase = 4 * q - 4;
        if (wbase + 0 < kTableWords) dst[(wbase + 0) * kSudokuBlock] = x.x;
        if (wbase + 1 < kTableWords) dst[(wbase + 1) * kSudokuBlock] = x.y;
        if (wbase + 2 < kTableWords) dst[(wbase + 2) * kSudokuBlock] = x.z;
        if (wbase + 3 < kTableWords) dst[(wbase + 3) * kSudokuBlock] = x.w;
    }
}
// the transposed blank bitmap (w[67..69]) stays in registers
struct SkBlankT { uint32_t t0, t1, t2; };
__device__ __forceinline__ SkBlankT sk_load_blank_t(const uint4* __restrict__ dg) {
    const uint4 a = __ldg(dg + 16), b = __ldg(dg + 17);
    SkBlankT x; x.t0 = a.w; x.t1 = b.x; x.t2 = b.y;
    return x;
}

// Enter a level: the cell's current domain and the subset that passes the forward check, i.e. is
// not the only value left to some later blank peer.  Seven packed words cover every later peer, all
// straight-line code (a lane whose cell has fewer later peers runs the same instructions on empty
// selections): the rest of the row (own word above the cell's field + two stacks to the right), the
// box-rows below inside the band (two), and the column below the band as two TRANSPOSED words —
// three rows of one column each — built from the band-packed row masks.
__device__ __forceinline__ void sk_enter(const SudokuSmem& S, int t, const SkCell& c, const SkBlankT& bt, uint32_t& dom, uint32_t& pass) {
    const uint32_t rowband = S.rowp[c.band][t];
    const uint32_t colw = S.colp[c.s][t];
    const uint32_t boxv = S.boxr[c.box][t];
    const uint32_t rowv = sk_rep((rowband >> (10 * c.rm)) & 0x1FF);
    const uint32_t colv = (colw >> (10 * c.f)) & 0x1FF;
    dom = ~(rowv | colv | boxv) & 0x1FF;
    // own word: the fields above the cell's
    uint32_t kill3 = sk_singletons(~(rowv | colw | boxv) & S.blk[c.r * 3 + c.s][t] & (0xFFFFFFFFu << (10 * c.f + 10)) & SK_FULL3);
    // stacks to the right
    {
        const uint32_t* colp = &S.colp[c.s][t];
        const uint32_t* boxp = &S.boxr[c.box][t];
        const uint32_t* blkp = &S.blk[c.r * 3 + c.s][t];
#pragma unroll
        for (int k = 1; k <= 2; k++) {
            const bool on = c.s + k < 3;
            const uint32_t u = on ? (rowv | colp[k * kSudokuBlock] | boxp[k * kSudokuBlock]) : 0xFFFFFFFFu;
            const uint32_t b = on ? blkp[k * kSudokuBlock] : 0u;
            kill3 |= sk_singletons(~u & b);
        }
    }
    // box-rows below, inside the band
    {
        const uint32_t* blkp = &S.blk[c.r * 3 + c.s][t];
#pragma unroll
        for (int k = 1; k <= 2; k++) {
            const bool on = c.rm + k < 3;
            const uint32_t rv = sk_rep((rowband >> (on ? 10 * (c.rm + k) : 0)) & 0x1FF);
            const uint32_t b = on ? blkp[3 * k * kSudokuBlock] : 0u;
            kill3 |= sk_singletons(~(rv | colw | boxv) & b);
        }
    }
    // the column below the band: bands band+1, band+2, three rows per word
    {
        const uint32_t crep = sk_rep(colv);
        const uint32_t* rowp = &S.rowp[c.band][t];
        const uint32_t* boxp = &S.boxr[c.box][t];
        const int q0 = 9 * (3 * c.s + c.f) + 3 * c.band;            // transposed bit index of (row 3*band, this column)
#pragma unroll
        for (int k = 1; k <= 2; k++) {
            const bool on = c.band + k < 3;
            const int q = q0 + 3 * k;
            const uint32_t lo = q < 32 ? bt.t0 : (q < 64 ? bt.t1 : bt.t2);
            const uint32_t hi = q < 32 ? bt.t1 : (q < 64 ? bt.t2 : 0u);
            const uint32_t m3 = on ? (__funnelshift_r(lo, hi, q & 31) & 7u) : 0u;
            const uint32_t b = ((m3 * 0x00040201u) & SK_ONES) * 0x1FFu;           // 0x1FF in the fields of the blank rows
            const uint32_t u = on ? (crep | rowp[k * kSudokuBlock] | boxp[3 * k * kSudokuBlock]) : 0xFFFFFFFFu;
            kill3 |= sk_singletons(~u & b);
        }
    }
    const uint32_t kill = (kill3 | (kill3 >> 10) | (kill3 >> 20)) & 0x1FF;
    pass = dom & ~kill;
}

// Step back one level (RestoreSavedDomainStep, dequan.h:431-440).  Returns true when the task's
// own root level is exhausted — the caller closes the task.
__device__ __forceinline__ bool sk_pop(SudokuSmem& S, int t, SkLane& L) {
    L.nodes += __popc(L.dom_rem);            // the leftover values here all fail their check: tried, counted, gone
    if (L.sp == L.base_sp) return true;
    --L.sp;
    const uint32_t e = S.stk[L.sp][t];
    const uint32_t v = e >> 9, bit = 1u << v;
    L.p = sk_cell_at(S, t, L.sp);
    L.c = sk_decode(L.p);
    S.rowp[L.c.band][t] ^= bit << (10 * L.c.rm);
    S.boxr[L.c.box][t] ^= sk_rep(bit);
    S.colp[L.c.s][t] ^= bit << (10 * L.c.f);
    L.passrem = e & 0x1FF;
    L.dom_rem = ~sk_used_at(S, t, L.c) & 0x1FF & ~((2u << v) - 1u);
    return false;
}

// AssignVar(next passing value) (dequan.h:416-423).  Returns true when that was the last blank
// (a solution); otherwise the value is committed and the lane stands before the next level.
__device__ __forceinline__ bool sk_choose(SudokuSmem& S, int t, SkLane& L) {
    const uint32_t nxt = L.passrem & (0u - L.passrem);
    L.nodes += __popc(L.dom_rem & (nxt | (nxt - 1u)));          // the failing values skipped on the way, and this one
    L.passrem ^= nxt;
    const uint32_t v = __ffs(nxt) - 1;
    S.stk[L.sp][t] = (uint16_t)(L.passrem | (v << 9));
    if (L.sp == L.nblank - 1) return true;
    sk_commit(S, t, L.c, nxt);
    ++L.sp;
    L.p = sk_cell_at(S, t, L.sp);
    L.enter = true;
    return false;
}

// Stack snapshot in HBM: u16 per level (passing untried | value << 9), eight levels per uint4.
__device__ __forceinline__ uint32_t sk_snap_entry(const uint4* __restrict__ sb, int l) {
    const uint4 cur = __ldcg(sb + (l >> 3));
    const uint32_t word = (l & 4) ? ((l & 2) ? cur.w : cur.z) : ((l & 2) ? cur.y : cur.x);
    return (l & 1) ? (word >> 16) : (word & 0xFFFF);
}
// levels 0..upto-1 from the stack, then `extra0`, `extra1` as entries upto and upto+1
__device__ __forceinline__ void sk_snap_write(uint4* __restrict__ sb, const SudokuSmem& S, int t, int upto, uint32_t extra0, uint32_t extra1) {
    for (int q = 0; q * 8 <= upto + 1; q++) {
        uint32_t w4[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int l0 = q * 8 + 2 * i, l1 = l0 + 1;
            const uint32_t e0 = l0 < upto ? (uint32_t)S.stk[l0][t] : (l0 == upto ? extra0 : (l0 == upto + 1 ? extra1 : 0u));
            const uint32_t e1 = l1 < upto ? (uint32_t)S.stk[l1][t] : (l1 == upto ? extra0 : (l1 == upto + 1 ? extra1 : 0u));
            w4[i] = e0 | (e1 << 16);
        }
        __stcg(sb + q, make_uint4(w4[0], w4[1], w4[2], w4[3]));
    }
}

constexpr int kPopQuorum = 10;          // extra pop rounds run while at least this many lanes still stand on an exhausted level

// The warp writes the solutions of its finished lanes, one lane at a time, coalesced.
__device__ __forceinline__ void sk_store_solutions(const SudokuSmem& S, const SudokuArgs& A, int t, bool fin, uint32_t puzzle,
                                                   uint32_t b0, uint32_t b1, uint32_t b2) {
    const int lane = t & 31;
    const uint32_t lt = (1u << lane) - 1u;
    __syncwarp();
    uint32_t fm = __ballot_sync(0xFFFFFFFFu, fin);
    while (fm) {
        const int Ls = __ffs(fm) - 1;
        fm &= fm - 1;
        const uint32_t x0 = __shfl_sync(0xFFFFFFFFu, b0, Ls), x1 = __shfl_sync(0xFFFFFFFFu, b1, Ls), x2 = __shfl_sync(0xFFFFFFFFu, b2, Ls);
        const uint32_t pz = __shfl_sync(0xFFFFFFFFu, puzzle, Ls);
        uint8_t* out = A.solution + (size_t)pz * A.stride;
        const uint8_t* in = A.cells + (size_t)pz * A.stride;
        const int tL = (t & ~31) + Ls;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const int cell = lane + 32 * k;
            if (cell < 81) {
                const uint32_t bw = k == 0 ? x0 : (k == 1 ? x1 : x2);
                uint8_t val;
                if ((bw >> lane) & 1u) {
                    const int level = __popc(bw & lt) + (k > 0 ? __popc(x0) : 0) + (k > 1 ? __popc(x1) : 0);
                    val = (uint8_t)((S.stk[level][tL] >> 9) + 1);
                } else val = in[cell];
                out[cell] = val;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// k_sudoku_first: lane per instance, the reference's search as it is, up to first_budget nodes.
__global__ void __launch_bounds__(kSudokuBlock)
k_sudoku_first(SudokuArgs A) {
    extern __shared__ __align__(16) unsigned char sk_raw[];
    SudokuSmem& S = *reinterpret_cast<SudokuSmem*>(sk_raw);
    const int t = threadIdx.x;
    const int lane = t & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const unsigned long long total_warps = (unsigned long long)gridDim.x * (kSudokuBlock / 32);

    SkLane L = {};
    SkBlankT bt = {0, 0, 0};
    uint32_t b0 = 0, b1 = 0, b2 = 0;        // blank bitmap
    uint32_t limit = 0;
    bool limit_is_api = false, done = false;
    unsigned long long chunk_pos = 0, chunk_end = 0;
    bool exhausted = false;

    for (;;) {
        // ---------------- refill ----------------
        const uint32_t need = __ballot_sync(0xFFFFFFFFu, !L.have && !done);
        if (need) {
            const uint32_t n_need = __popc(need);
            if (chunk_pos >= chunk_end && !exhausted) {
                unsigned long long base = 0;
                uint32_t size = 0;
                if (lane == 0) {
                    const unsigned long long cur = *(volatile unsigned long long*)(A.ctrl + SKC_FRESH);
                    const unsigned long long remaining = cur < (unsigned long long)A.n ? (unsigned long long)A.n - cur : 0;
                    size = (uint32_t)min(max(remaining / (8ull * total_warps), (unsigned long long)n_need), 64ull);
                    base = atomicAdd(A.ctrl + SKC_FRESH, (unsigned long long)size);
                }
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                size = __shfl_sync(0xFFFFFFFFu, size, 0);
                chunk_pos = base;
                chunk_end = min(base + size, (unsigned long long)A.n);
                if (base >= (unsigned long long)A.n) { exhausted = true; chunk_end = chunk_pos; }
            }
            const unsigned long long avail = chunk_end - chunk_pos;
            if (!L.have && !done) {
                const uint32_t rank = __popc(need & lt);
                if (rank < avail) {
                    L.puzzle = (uint32_t)(chunk_pos + rank);
                    const uint4* dg = A.digest[L.puzzle].v;
                    const uint4 head = __ldg(dg);
                    b0 = head.x; b1 = head.y; b2 = head.z;
                    L.nblank = (int)(head.w & 0xFF);
                    L.nodes = 0; L.nodes_hi = 0;
                    limit = A.first_budget; limit_is_api = false;
                    bool skip = false;
                    if (head.w & 0x80000000u) { A.status[L.puzzle] = SK_STATUS_DEFER; skip = true; }
                    else if (A.user_budget) {
                        const unsigned long long givens = 81 - L.nblank;
                        if (A.user_budget < givens) {        // the budget runs out among the givens
                            A.nodes[L.puzzle] = A.user_budget + 1; A.status[L.puzzle] = 2; skip = true;
                            uint8_t* out = A.solution + (size_t)L.puzzle * A.stride;
                            for (int i = 0; i < 81; i++) out[i] = 0;
                        } else if (A.user_budget - givens + 1 <= (unsigned long long)limit) {
                            limit = (uint32_t)(A.user_budget - givens + 1);
                            limit_is_api = true;
                        }
                    }
                    if (!skip && L.nblank == 0) {
                        // nothing to search: the givens are the solution (81 nodes); k_sudoku_finish applies the budget
                        A.nodes[L.puzzle] = 81; A.status[L.puzzle] = 1;
                        uint8_t* out = A.solution + (size_t)L.puzzle * A.stride;
                        const uint8_t* in = A.cells + (size_t)L.puzzle * A.stride;
                        for (int i = 0; i < 81; i++) out[i] = in[i];
                        skip = true;
                    }
                    if (!skip) {
                        sk_load_tables(S, t, dg);
                        bt = sk_load_blank_t(dg);
                        L.sp = 0; L.base_sp = 0; L.passrem = 0; L.dom_rem = 0;
                        L.p = sk_cell_at(S, t, 0);
                        L.enter = true;
                        L.have = true;
                    }
                } else if (exhausted) done = true;
            }
            chunk_pos += min((unsigned long long)n_need, avail);
            if (__all_sync(0xFFFFFFFFu, done && !L.have)) break;
        }

        // ---------------- exhausted levels: step back ----------------
        for (int rep = 0;; rep++) {
            const bool popping = L.have && !L.enter && L.passrem == 0;
            const uint32_t pm = __ballot_sync(0xFFFFFFFFu, popping);
            if (pm == 0 || (rep > 0 && __popc(pm) < kPopQuorum)) break;
            if (popping && sk_pop(S, t, L)) {
                // the whole tree is exhausted: ForwardCheckingStep returns false
                A.nodes[L.puzzle] = (81 - L.nblank) + L.nodes_hi + L.nodes;
                A.status[L.puzzle] = 0;
                uint8_t* out = A.solution + (size_t)L.puzzle * A.stride;
                for (int i = 0; i < 81; i++) out[i] = 0;
                L.have = false;
            }
        }

        // ---------------- next passing value ----------------
        bool fin = false;
        if (L.have && !L.enter && L.passrem != 0 && sk_choose(S, t, L)) {
            A.nodes[L.puzzle] = (81 - L.nblank) + L.nodes_hi + L.nodes;
            A.status[L.puzzle] = 1;
            fin = true;
            L.have = false;
        }

        // ---------------- enter the next level ----------------
        if (L.have && L.enter) {
            L.c = sk_decode(L.p);
            uint32_t dom, pass;
            sk_enter(S, t, L.c, bt, dom, pass);
            L.dom_rem = dom; L.passrem = pass; L.enter = false;
        }

        // ---------------- node budgets ----------------
        if (L.have && L.nodes >= limit) {
            if (limit_is_api) {
                A.nodes[L.puzzle] = A.user_budget + 1; A.status[L.puzzle] = 2;
                uint8_t* out = A.solution + (size_t)L.puzzle * A.stride;
                for (int i = 0; i < 81; i++) out[i] = 0;
            } else {
                // not done within the budget: park the search (stack snapshot + nodes so far) on the hard list; the
                // counting pipeline picks it up exactly where it stands
                const unsigned long long sslot = atomicAdd(A.ctrl + SKC_SNAP, 1ull);
                const unsigned long long idx = atomicAdd(A.ctrl + SKC_HARD, 1ull);
                if (sslot < A.snap_cap) { sk_snap_write(A.snaps + (size_t)sslot * kSnapWords, S, t, L.sp, L.passrem, L.dom_rem); A.snap_state[sslot] = 1u; }
                else atomicOr(A.ctrl + SKC_ERROR, 2ull);
                A.hard[2 * idx] = L.puzzle;
                A.hard[2 * idx + 1] = (uint32_t)sslot | ((uint32_t)L.sp << 24);
                A.nodes[L.puzzle] = (81 - L.nblank) + L.nodes_hi + L.nodes;
                A.status[L.puzzle] = SK_STATUS_HARD;
            }
            L.have = false;
        }

        sk_store_solutions(S, A, t, fin, L.puzzle, b0, b1, b2);
    }
}

// ---------------------------------------------------------------------------------------------
// k_sudoku_strong: warp per hard instance.  Lane j holds cells j, j+32, j+64 in the three fields
// of one register: bits 0-8 the cell's domain, bit 9 "this cell's single value has been
// propagated to its peers".  Same static order, same ascending value order as the reference, plus
// naked-single propagation to a fixed point after every assignment, so the first solution it
// reaches is the reference's first solution.
constexpr unsigned kStrongHiddenAfter = 400;   // value tries after which an instance also gets hidden-single propagation

struct StrongSmem {
    uint32_t peer[81][32];               // peer[x][lane]: bit 10*f set iff cell lane+32f is a peer of x
    // followed, for `levels` = the most blanks of any instance in the batch (SudokuArgs::stack_levels), by
    //   uint32_t saved[4][levels][32]   per warp, per level: the registers before the level's first value
    //   uint16_t rest[4][levels]        per warp, per level: values still to try (0: forced level)
};
__host__ __device__ inline size_t sudoku_strong_smem(int levels) { return sizeof(StrongSmem) + (size_t)4 * levels * (32 * 4 + 2) + 16; }

// Hidden singles: a value that only one cell of a row, column or box can still take goes to that cell; a value no
// cell of the unit can take is a contradiction.  Lane u < 27 owns unit u (its three 32-bit cell masks u0..u2 in the
// lane/field numbering); per value, three ballots give the 81-bit "cells that can hold it" mask.
// Returns false on a contradiction; `changed` reports whether any domain was cut.
__device__ __forceinline__ bool sk_hidden_singles(uint32_t& D, int lane, uint32_t u0, uint32_t u1, uint32_t u2, bool& changed) {
    bool mine = false;
#pragma unroll 1
    for (int v = 0; v < 9; v++) {
        const uint32_t w0 = __ballot_sync(0xFFFFFFFFu, (D >> v) & 1u) & u0;
        const uint32_t w1 = __ballot_sync(0xFFFFFFFFu, (D >> (10 + v)) & 1u) & u1;
        const uint32_t w2 = __ballot_sync(0xFFFFFFFFu, (D >> (20 + v)) & 1u) & u2;
        const int cnt = __popc(w0) + __popc(w1) + __popc(w2);
        if (__any_sync(0xFFFFFFFFu, lane < 27 && cnt == 0)) return false;
        uint32_t hs = __ballot_sync(0xFFFFFFFFu, lane < 27 && cnt == 1);
        const int cell = w0 ? __ffs(w0) - 1 : (w1 ? 32 + __ffs(w1) - 1 : 64 + __ffs(w2) - 1);
        while (hs) {
            const int u = __ffs(hs) - 1;
            hs &= hs - 1;
            const int c = __shfl_sync(0xFFFFFFFFu, cell, u);
            if (lane == (c & 31)) {
                const int f = c >> 5;
                if (((D >> (10 * f)) & 0x1FF) != (1u << v)) {             // more than this value left: cut (flag stays clear)
                    D = (D & ~(0x3FFu << (10 * f))) | ((1u << v) << (10 * f));
                    mine = true;
                }
            }
        }
    }
    changed = __any_sync(0xFFFFFFFFu, mine);
    return true;
}

// Naked singles to a fixed point; with `hidden`, hidden singles as well.
__device__ __forceinline__ bool sk_propagate(uint32_t& D, const StrongSmem& M, int lane, uint32_t valid3,
                                             bool hidden, uint32_t u0, uint32_t u1, uint32_t u2) {
    for (;;) {
        const uint32_t x3 = D & SK_FULL3;
        const uint32_t zero = ~(x3 + (SK_SPARE - SK_ONES)) & SK_SPARE & (valid3 << 9);    // spare bit of the EMPTY fields
        if (__any_sync(0xFFFFFFFFu, zero != 0)) return false;
        const uint32_t unfl = ~D & SK_SPARE & (valid3 << 9);
        const uint32_t sing = sk_singletons(x3 & ((unfl >> 9) * 0x1FFu));
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, sing != 0);
        if (!b) {
            if (!hidden) return true;
            bool changed = false;
            if (!sk_hidden_singles(D, lane, u0, u1, u2, changed)) return false;
            if (!changed) return true;
            continue;
        }
        const int j = __ffs(b) - 1;
        const uint32_t sj = __shfl_sync(0xFFFFFFFFu, sing, j);
        const int f = (sj & 0x1FF) ? 0 : (((sj >> 10) & 0x1FF) ? 1 : 2);
        const uint32_t bit = (sj >> (10 * f)) & 0x1FF;
        if (lane == j) D |= 0x200u << (10 * f);
        D &= ~(M.peer[j + 32 * f][lane] * bit);
    }
}

__global__ void __launch_bounds__(128)
k_sudoku_strong(SudokuArgs A) {
    extern __shared__ __align__(16) unsigned char sk_raw[];
    StrongSmem& M = *reinterpret_cast<StrongSmem*>(sk_raw);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint32_t* const saved = reinterpret_cast<uint32_t*>(sk_raw + sizeof(StrongSmem)) + (size_t)wib * A.stack_levels * 32 + lane;   // [level * 32]
    uint16_t* const rest = reinterpret_cast<uint16_t*>(sk_raw + sizeof(StrongSmem) + (size_t)4 * A.stack_levels * 128) + wib * A.stack_levels;
    // peer table, once per CTA
    for (int i = threadIdx.x; i < 81 * 32; i += blockDim.x) {
        const int x = i >> 5, l = i & 31;
        const int xr = x / 9, xc = x % 9;
        uint32_t m = 0;
        for (int f = 0; f < 3; f++) {
            const int q = l + 32 * f;
            if (q >= 81 || q == x) continue;
            const int qr = q / 9, qc = q % 9;
            if (qr == xr || qc == xc || (qr / 3 == xr / 3 && qc / 3 == xc / 3)) m |= 1u << (10 * f);
        }
        M.peer[x][l] = m;
    }
    __syncthreads();
    const uint32_t valid3 = lane < 17 ? SK_ONES : 0x00000401u;      // lanes 17..31 hold two cells
    // lane u < 27 owns unit u (rows 0-8, columns 9-17, boxes 18-26): its cells as bit (cell & 31) of word (cell >> 5)
    uint32_t u0 = 0, u1 = 0, u2 = 0;
    if (lane < 27)
        for (int k = 0; k < 9; k++) {
            const int cell = lane < 9 ? lane * 9 + k : (lane < 18 ? k * 9 + (lane - 9)
                                                                  : ((lane - 18) / 3 * 3 + k / 3) * 9 + ((lane - 18) % 3 * 3 + k % 3));
            const uint32_t bit = 1u << (cell & 31);
            if (cell < 32) u0 |= bit; else if (cell < 64) u1 |= bit; else u2 |= bit;
        }
    const unsigned long long n_hard = A.ctrl[SKC_HARD];
    for (;;) {
        unsigned long long idx = 0;
        if (lane == 0) idx = atomicAdd(A.ctrl + SKC_HARD_CUR, 1ull);
        idx = __shfl_sync(0xFFFFFFFFu, idx, 0);
        if (idx >= n_hard) break;
        const uint32_t puzzle = A.hard[2 * idx];
        const uint8_t* in = A.cells + (size_t)puzzle * A.stride;
        const uint32_t* dw = reinterpret_cast<const uint32_t*>(A.digest[puzzle].v);
        const int nblank = (int)(__ldg(dw + 3) & 0xFF);
        const uint32_t cw = lane < 21 ? __ldg(dw + 46 + lane) : 0u;          // cell ids per level, four per word
        // initial domains from the digest's used masks; givens are singletons already propagated
        uint32_t D = 0;
#pragma unroll
        for (int f = 0; f < 3; f++) {
            const int q = lane + 32 * f;
            if (q < 81) {
                const uint32_t g = in[q];
                uint32_t field;
                if (g) field = (1u << (g - 1)) | 0x200u;
                else {
                    const SkCell k = sk_decode(q);
                    field = ~((__ldg(dw + 4 + k.band) >> (10 * k.rm)) | (__ldg(dw + 7 + k.s) >> (10 * k.f)) | __ldg(dw + 10 + k.box)) & 0x1FF;
                }
                D |= field << (10 * f);
            }
        }
        // explicit-stack DFS over the blank levels; `back` = the level was reached by stepping back
        // Instances that stay hard under naked singles alone (a few per thousand) switch hidden singles on as well: any
        // sound pruning leaves the first solution in DFS order where it is.
        unsigned tries = 0;
        int l = sk_propagate(D, M, lane, valid3, false, u0, u1, u2) ? 0 : -1;
        bool back = false;
        while (l >= 0 && l < nblank) {
            const int p = (int)((__shfl_sync(0xFFFFFFFFu, cw, l >> 2) >> ((l & 3) * 8)) & 0xFF);
            const int owner = p & 31, f = p >> 5;
            uint32_t d;
            if (!back) {
                const uint32_t w = __shfl_sync(0xFFFFFFFFu, D, owner) >> (10 * f);
                if (w & 0x200u) {                          // forced: its single value is already everywhere
                    if (lane == 0) rest[l] = 0;
                    __syncwarp();
                    ++l;
                    continue;
                }
                d = w & 0x1FF;
                saved[l * 32] = D;
            } else d = rest[l];
            bool ok = false;
            while (d) {                                    // the level's values in ascending order, each from the saved state
                const uint32_t v = d & (0u - d);
                d ^= v;
                D = saved[l * 32];
                if (lane == owner) D = (D & ~(0x3FFu << (10 * f))) | ((v | 0x200u) << (10 * f));
                D &= ~(M.peer[p][lane] * v);
                ++tries;
                if (sk_propagate(D, M, lane, valid3, tries > kStrongHiddenAfter, u0, u1, u2)) { ok = true; break; }
            }
            __syncwarp();
            if (lane == 0) rest[l] = (uint16_t)d;
            __syncwarp();
            if (ok) { ++l; back = false; }
            else {
                --l;
                while (l >= 0 && rest[l] == 0) --l;
                back = true;
            }
        }
        const bool sat = l == nblank;
        // result: the reference's first solution, or none
        uint8_t* out = A.solution + (size_t)puzzle * A.stride;
#pragma unroll
        for (int f = 0; f < 3; f++) {
            const int q = lane + 32 * f;
            if (q < 81) out[q] = sat ? (uint8_t)__ffs((D >> (10 * f)) & 0x1FF) : (uint8_t)0;
        }
        if (lane == 0) A.status[puzzle] = sat ? 1 : 0;
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// k_sudoku_walk: lane per hard instance.  k_sudoku_first parked the reference's search at some
// point P of its DFS (stack snapshot, nodes so far); k_sudoku_strong found the solution S the
// search ends at (or that there is none).  What the reference still visits between P and S:
//   * everything left on the parked stack BELOW the level d where P's path leaves S's path — one
//     task: "count the snapshot's levels (d, sp] exhaustively";
//   * at level d the values between the parked one and S's: nodes; the passing ones are root tasks
//     ("count the whole subtree under path-prefix + value");
//   * at every deeper path level the values up to S's: nodes, passing earlier ones root tasks.
// No solution: everything left on the parked stack, one task.
__global__ void __launch_bounds__(kSudokuBlock)
k_sudoku_walk(SudokuArgs A) {
    extern __shared__ __align__(16) unsigned char sk_raw[];
    SudokuSmem& S = *reinterpret_cast<SudokuSmem*>(sk_raw);
    const int t = threadIdx.x;
    const int lane = t & 31;
    const unsigned long long n_hard = A.ctrl[SKC_HARD];
    auto emit = [&](uint32_t puzzle, uint32_t snap, uint32_t info) {
        const unsigned long long slot = atomicAdd(A.ctrl + SKC_RESERVE, 1ull);
        if (slot >= A.task_cap) { atomicOr(A.ctrl + SKC_ERROR, 2ull); return; }
        atomicAdd(A.ctrl + SKC_OUTSTANDING, 1ull);
        *reinterpret_cast<uint4*>(A.tasks + slot) = make_uint4(puzzle, snap, SKT_VALID | info, 0u);
    };
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(A.ctrl + SKC_WALK_CUR, 32ull);
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (base >= n_hard) break;
        const bool active = base + lane < n_hard;
        const uint32_t puzzle = active ? A.hard[2 * (base + lane)] : 0u;
        const uint32_t hinfo = active ? A.hard[2 * (base + lane) + 1] : 0u;
        const uint32_t snap = hinfo & 0xFFFFFFu;
        const int psp = (int)(hinfo >> 24);                        // the level the parked search stands on
        const uint4* sb = A.snaps + (size_t)snap * kSnapWords;
        int nblank = 0;
        bool sat = false;
        SkBlankT bt = {0, 0, 0};
        if (active) {
            const uint4* dg = A.digest[puzzle].v;
            nblank = (int)(__ldg(dg).w & 0xFF);
            sk_load_tables(S, t, dg);
            bt = sk_load_blank_t(dg);
            sat = A.status[puzzle] == 1;
        }
        const uint8_t* sol = A.solution + (size_t)puzzle * A.stride;
        if (active && !sat) emit(puzzle, snap, SKT_TOP | 0u | ((uint32_t)psp << 8));      // the whole parked stack
        unsigned long long direct = 0;
        bool on_parked_path = true;                                 // levels so far: parked path == solution path
        const int levels = active && sat ? nblank : 0;
        const int max_levels = __reduce_max_sync(0xFFFFFFFFu, levels);
        for (int l = 0; l < max_levels; l++) {
            if (l < levels) {
                const int p = sk_cell_at(S, t, l);
                const SkCell c = sk_decode(p);
                const uint32_t bit = 1u << (sol[p] - 1);
                uint32_t dom_rem, passrem;                          // what the reference still tries at this level
                bool charge = true;
                if (on_parked_path && l < psp) {
                    const uint32_t e = sk_snap_entry(sb, l);
                    const uint32_t v = e >> 9;
                    if ((1u << v) == bit) charge = false;           // the parked search already stands on the solution's value here
                    else {
                        // d: the parked path leaves the solution path.  Below d the parked stack is solution-free
                        if ((1u << v) > bit) atomicOr(A.ctrl + SKC_ERROR, 8ull);
                        emit(puzzle, snap, SKT_TOP | (uint32_t)(l + 1) | ((uint32_t)psp << 8));
                        passrem = e & 0x1FF;
                        dom_rem = ~sk_used_at(S, t, c) & 0x1FF & ~((2u << v) - 1u);
                        on_parked_path = false;
                    }
                } else if (on_parked_path && l == psp) {
                    passrem = sk_snap_entry(sb, l) & 0x1FF;         // parked exactly on the solution path: its untried sets
                    dom_rem = sk_snap_entry(sb, l + 1) & 0x1FF;
                    on_parked_path = false;
                } else {
                    uint32_t dom, pass;
                    sk_enter(S, t, c, bt, dom, pass);
                    dom_rem = dom; passrem = pass;
                }
                if (charge) {
                    direct += __popc(dom_rem & (bit | (bit - 1u)));          // tried in ascending order up to the solution's value
                    if (!(passrem & bit)) atomicOr(A.ctrl + SKC_ERROR, 8ull);
                    uint32_t V = passrem & (bit - 1u);                       // earlier passing values: whole subtrees to count
                    while (V) {
                        const uint32_t v = __ffs(V) - 1;
                        V &= V - 1;
                        emit(puzzle, 0u, SKT_ROOT | (uint32_t)l | (v << 8));
                    }
                }
                sk_commit(S, t, c, bit);
            }
        }
        if (active && direct) atomicAdd(A.nodes + puzzle, direct);
    }
}

// ---------------------------------------------------------------------------------------------
// k_sudoku_count: ONE persistent launch.  Lanes take tasks from the queue and count their subtrees
// exhaustively; a warp leaves when no task is outstanding.  Load balance is demand driven: idle
// lanes draw tickets for queue slots that are not published yet; busy lanes look every
// kDonatePeriod steps and, while tickets are waiting, hand over the SHALLOWEST stack level that
// still has untried passing values as a new task (a "piece").  A piece owns stack levels [lo, hi] of the
// donor's snapshot; the donor keeps the deeper ones.  Every level is owned by exactly one task,
// which also counts the level's failing leftovers when it steps back through it.
constexpr int kDonatePeriod = 32;
constexpr uint32_t kDonateMinNodes = 48;    // a task younger than this keeps its stack to itself
constexpr uint32_t kDonateGap = 96;         // ... and so does one that gave a level away fewer nodes ago than this
constexpr int kDonateDepth = 5;             // ... and it gives away only levels at least this far above the current one (swept 1..12: flat optimum around 5)
constexpr uint32_t kSplitGap = 512;         // a task splits unasked every time it has counted this many nodes (1 M puzzles, count stage: 4096 -> 11.0 ms, 1024 -> 10.2, 512 -> 9.9, 256 -> 10.0, 128 -> 33.8)

__global__ void __launch_bounds__(kSudokuBlock)
k_sudoku_count(SudokuArgs A) {
    extern __shared__ __align__(16) unsigned char sk_raw[];
    SudokuSmem& S = *reinterpret_cast<SudokuSmem*>(sk_raw);
    const int t = threadIdx.x;
    const int lane = t & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const unsigned long long total_warps = (unsigned long long)gridDim.x * (kSudokuBlock / 32);
    volatile unsigned long long* vctrl = A.ctrl;

    SkLane L = {};
    SkBlankT bt = {0, 0, 0};
    uint32_t donate_at = 0;                 // node count from which the task may give a level away
    uint32_t split_at = 0;                  // node count from which it does so unasked
    bool waiting = false, poll_now = false; // holds a ticket for a queue slot that is not published yet
    unsigned long long ticket = 0;
    int iter = 0;
    unsigned spins = 0;

    for (;;) {
        // ---------------- refill from the task queue ----------------
        // An idle lane draws a TICKET (the next queue slot, atomicAdd — no contention window) and waits for that slot
        // to be published.  Slots already written (the walker's root tasks) are there at once; a ticket beyond the
        // published end is a standing order that the next donor fills: tickets drawn minus tasks reserved IS the
        // number of hungry lanes.
        {
            const uint32_t need = __ballot_sync(0xFFFFFFFFu, !L.have && !waiting);
            if (need) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(A.ctrl + SKC_HEAD, (unsigned long long)__popc(need));
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (!L.have && !waiting) { ticket = base + __popc(need & lt); waiting = true; poll_now = true; }
            }
        }
        unsigned closed_now = 0;                // tasks this lane took and closed on the spot
        uint32_t got_info = 0, got_snap = 0;    // the task this lane has just drawn (info != 0, not a null task)
        if (waiting && (poll_now || (iter & 7) == 0) && ticket < A.task_cap) {
            volatile uint32_t* rec = reinterpret_cast<volatile uint32_t*>(A.tasks + ticket);
            const uint32_t info = rec[2];       // the publisher writes `info` last
            if (info) {
                __threadfence();
                waiting = false;
                L.puzzle = rec[0];
                if (info & SKT_NULL) closed_now = 1;
                else { got_info = info; got_snap = rec[1]; }
            }
        }
        // A drawn task is set up by the WHOLE warp, one task after the other: the instance's tables into the lane's
        // columns (63 words, two per helper), then the path above the task — the solution's values (root task) or the
        // donor's (piece), one level per helper, OR-ed into the used masks with shared-memory atomics.  Done by the
        // lane alone this was a loop of ~40 instructions per level with one lane in 32 active: a third of the kernel.
        for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, got_info != 0u); todo; todo &= todo - 1u) {
            const int src = __ffs((int)todo) - 1;
            const uint32_t pz = __shfl_sync(0xFFFFFFFFu, L.puzzle, src), inf = __shfl_sync(0xFFFFFFFFu, got_info, src);
            const uint32_t sn = __shfl_sync(0xFFFFFFFFu, got_snap, src);
            const int ts = (t & ~31) + src;                                // the column of the lane that owns the task
            const uint32_t* dgw = reinterpret_cast<const uint32_t*>(A.digest[pz].v);
            uint32_t* tab = &S.rowp[0][0];
            for (int w = lane; w < kTableWords; w += 32) tab[w * kSudokuBlock + ts] = __ldg(dgw + 4 + w);
            __syncwarp();
            const bool root = (inf & SKT_ROOT) != 0u;
            const int lo = (int)(inf & 0xFF), hi = (int)((inf >> 8) & 0xFF);    // root: the task's level / value (low nibble of hi)
            const int n_replay = root ? lo + 1 : hi;
            const uint8_t* sol = A.solution + (size_t)pz * A.stride;
            const uint4* sb = A.snaps + (size_t)sn * kSnapWords;
            for (int l = lane; l < n_replay; l += 32) {
                const int q = sk_cell_at(S, ts, l);
                uint32_t v, entry;
                if (root) { v = l < lo ? (uint32_t)sol[q] - 1u : (uint32_t)(hi & 0xF); entry = v << 9; }
                else { const uint32_t e = sk_snap_entry(sb, l); v = e >> 9; entry = l >= lo ? e : (e & 0xFE00u); }
                const SkCell k = sk_decode(q);
                const uint32_t bit = 1u << v;
                atomicOr(&S.rowp[k.band][ts], bit << (10 * k.rm));
                atomicOr(&S.boxr[k.box][ts], sk_rep(bit));
                atomicOr(&S.colp[k.s][ts], bit << (10 * k.f));
                S.stk[l][ts] = (uint16_t)entry;
            }
            __syncwarp();
        }
        if (got_info) {
            const uint32_t info = got_info;
            const uint4* dg = A.digest[L.puzzle].v;
            L.nblank = (int)(__ldg(dg).w & 0xFF);
            bt = sk_load_blank_t(dg);
            L.nodes = 0; L.nodes_hi = 0;
            L.passrem = 0; L.dom_rem = 0;
            L.have = true;
            donate_at = A.force_donate ? A.force_donate : kDonateMinNodes;
            split_at = kSplitGap;
            if (info & SKT_ROOT) {
                // path values at the levels above, then the task's own value at its level: committed above
                const int l0 = (int)(info & 0xFF);
                L.sp = l0 + 1; L.base_sp = l0 + 1;
                if (L.sp >= L.nblank) { atomicOr(A.ctrl + SKC_ERROR, 4ull); L.have = false; closed_now = 1; }
                else { L.p = sk_cell_at(S, t, L.sp); L.enter = true; }
            } else {
                // resumed from the donor's snapshot: the values chosen at levels 0..hi-1 are committed above; the untried
                // values of levels [lo, hi] are this piece's, everything shallower belongs to other tasks
                const int lo = (int)(info & 0xFF), hi = (int)((info >> 8) & 0xFF);
                const uint4* sb = A.snaps + (size_t)got_snap * kSnapWords;
                L.sp = hi; L.base_sp = lo;
                L.p = sk_cell_at(S, t, hi);
                L.c = sk_decode(L.p);
                const uint32_t e = sk_snap_entry(sb, hi);
                L.passrem = e & 0x1FF;
                if (info & SKT_TOP) L.dom_rem = sk_snap_entry(sb, hi + 1) & 0x1FF;
                else L.dom_rem = ~sk_used_at(S, t, L.c) & 0x1FF & ~((2u << (e >> 9)) - 1u);   // the values above the one the donor took here
                L.enter = false;
                __threadfence();
                A.snap_state[got_snap] = 0u;                     // the snapshot has been read: its slot is free again
            }
        }
        poll_now = false;
        {
            const uint32_t cm = __ballot_sync(0xFFFFFFFFu, closed_now != 0);
            if (cm && lane == 0) atomicAdd(A.ctrl + SKC_OUTSTANDING, 0ull - (unsigned long long)__popc(cm));
            if (cm) continue;                   // the lanes that closed a task on the spot draw again
        }
        if (__ballot_sync(0xFFFFFFFFu, L.have) == 0) {
            // nobody in the warp has work: leave when nothing is outstanding anywhere, else wait on the tickets
            unsigned long long out = 0;
            if (lane == 0) out = vctrl[SKC_OUTSTANDING];
            out = __shfl_sync(0xFFFFFFFFu, out, 0);
            if (out == 0) break;
            __nanosleep(spins < 4096u ? 200u : 2000u);
            // (a guard against a hang, not a deadline: batches of hard puzzles keep a few lanes busy for seconds while
            // everybody else waits here — about four minutes of waiting before the warp gives up)
            if (++spins > 120000000u) { if (lane == 0) atomicOr(A.ctrl + SKC_ERROR, 1ull); break; }
            poll_now = true;
            continue;
        }
        spins = 0;
        ++iter;

        // ---------------- donate work while lanes elsewhere are hungry ----------------
        if ((iter & (kDonatePeriod - 1)) == 0) {
            long long demand = 0;
            if (lane == 0) {
                const unsigned long long h = vctrl[SKC_HEAD], r = vctrl[SKC_RESERVE];
                demand = h > r ? (long long)(h - r) : 0;                       // tickets waiting for a task to be published
                if (A.force_donate) demand = (long long)total_warps * 8;
            }
            demand = __shfl_sync(0xFFFFFFFFu, demand, 0);
            // eligible: an established task with an untried passing value on a level below the current one.  A task that
            // has grown large splits whether or not anybody is waiting, so that no giant subtree is left for the end.
            const bool want = L.have && !L.enter && (L.nodes >= split_at || (demand > 0 && L.nodes >= donate_at));
            if (__any_sync(0xFFFFFFFFu, want)) {
                int hl = -1;
                if (want) {
                    int l = L.base_sp;
                    while (l < L.sp && (S.stk[l][t] & 0x1FF) == 0) ++l;
                    if (l + kDonateDepth <= L.sp) hl = l;                               // a level close to the current one roots a tiny subtree
                    else if (L.nodes >= split_at) split_at = L.nodes + kSplitGap / 4;     // nothing to give right now: look again soon
                }
                const uint32_t elig = __ballot_sync(0xFFFFFFFFu, hl >= 0);
                const long long quota = min((long long)8, demand / (long long)total_warps + 1);
                if (hl >= 0 && (L.nodes >= split_at || (long long)__popc(elig & lt) < quota)) {
                    // a snapshot slot first (the pool is a ring: a slot is free again once the task that resumes from it has
                    // read it); none free at this position: no piece this time, the task offers again a little later
                    const unsigned long long sslot = atomicAdd(A.ctrl + SKC_SNAP, 1ull) % A.snap_cap;
                    if (atomicCAS(A.snap_state + sslot, 0u, 1u) != 0u) {
                        donate_at = L.nodes + kDonateGap; split_at = L.nodes + kSplitGap / 4;
                    } else {
                        atomicAdd(A.ctrl + SKC_OUTSTANDING, 1ull);             // the piece exists from here on
                        const unsigned long long slot = atomicAdd(A.ctrl + SKC_RESERVE, 1ull);
                        if (slot >= A.task_cap) {                              // task pool full: nobody will ever claim it
                            atomicAdd(A.ctrl + SKC_OUTSTANDING, 0ull - 1ull);
                            A.snap_state[sslot] = 0u;
                            donate_at = 0xFFFFFFFFu; split_at = 0xFFFFFFFFu;   // ... and this task stops offering
                        } else {
                            // stack snapshot, levels 0..hl
                            sk_snap_write(A.snaps + (size_t)sslot * kSnapWords, S, t, hl + 1, 0u, 0u);
                            volatile uint32_t* rec = reinterpret_cast<volatile uint32_t*>(A.tasks + slot);
                            rec[0] = L.puzzle; rec[1] = (uint32_t)sslot;
                            __threadfence();
                            rec[2] = SKT_VALID | (uint32_t)L.base_sp | ((uint32_t)hl << 8);
                            L.base_sp = hl + 1;                                  // this task keeps the deeper levels
                            donate_at = L.nodes + (A.force_donate ? A.force_donate : kDonateGap);
                            split_at = L.nodes + kSplitGap;
                        }
                    }
                }
            }
        }

        // ---------------- exhausted levels: step back ----------------
        unsigned closed = 0;
        for (int rep = 0;; rep++) {
            const bool popping = L.have && !L.enter && L.passrem == 0;
            const uint32_t pm = __ballot_sync(0xFFFFFFFFu, popping);
            if (pm == 0 || (rep > 0 && __popc(pm) < kPopQuorum)) break;
            if (popping && sk_pop(S, t, L)) {
                atomicAdd(A.nodes + L.puzzle, L.nodes_hi + L.nodes);             // every node of the subtree is a node of the reference
                L.have = false; closed = 1;
            }
        }

        // ---------------- next passing value ----------------
        if (L.have && !L.enter && L.passrem != 0 && sk_choose(S, t, L))
            atomicOr(A.ctrl + SKC_ERROR, 4ull);                                  // a subtree left of the first solution cannot hold one

        // ---------------- enter the next level ----------------
        if (L.have && L.enter) {
            L.c = sk_decode(L.p);
            uint32_t dom, pass;
            sk_enter(S, t, L.c, bt, dom, pass);
            L.dom_rem = dom; L.passrem = pass; L.enter = false;
        }
        if (L.nodes >= 0x80000000u) { L.nodes_hi += L.nodes; L.nodes = 0; donate_at = 0; split_at = kSplitGap; }

        // ---------------- closed tasks leave the outstanding count ----------------
        {
            const uint32_t cm = __ballot_sync(0xFFFFFFFFu, closed != 0);
            if (cm && lane == 0) atomicAdd(A.ctrl + SKC_OUTSTANDING, 0ull - (unsigned long long)__popc(cm));
        }
    }
}

// Last pass, one thread per instance: the API node budget applied to the exact totals; batch totals.
__global__ void k_sudoku_finish(SudokuArgs A, unsigned long long* totals) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned sat = 0, unsat = 0, budget = 0;
    unsigned long long nd = 0;
    if (i < A.n) {
        uint8_t st = A.status[i];
        if (st != SK_STATUS_DEFER) {
            if (A.user_budget && A.nodes[i] > A.user_budget && st != 2) {
                st = 2;
                A.nodes[i] = A.user_budget + 1;
                uint8_t* out = A.solution + (size_t)i * A.stride;
                for (int c = 0; c < 81; c++) out[c] = 0;
            }
            A.status[i] = st;
            nd = A.nodes[i];
            sat = st == 1; unsat = st == 0; budget = st == 2;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        sat += __shfl_down_sync(0xFFFFFFFFu, sat, o);
        unsat += __shfl_down_sync(0xFFFFFFFFu, unsat, o);
        budget += __shfl_down_sync(0xFFFFFFFFu, budget, o);
        nd += __shfl_down_sync(0xFFFFFFFFu, nd, o);
    }
    if ((threadIdx.x & 31) == 0 && (sat | unsat | budget | (nd != 0))) {
        if (sat) atomicAdd(totals + 0, (unsigned long long)sat);
        if (unsat) atomicAdd(totals + 1, (unsigned long long)unsat);
        if (budget) atomicAdd(totals + 2, (unsigned long long)budget);
        atomicAdd(totals + 3, nd);
    }
}

// Compacts the ids of the instances the digest deferred to the generic engine.
__global__ void k_sudoku_collect_deferred(const uint8_t* __restrict__ status, long long n, int* __restrict__ list,
                                          unsigned long long* __restrict__ count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && status[i] == SK_STATUS_DEFER) list[atomicAdd(count, 1ull)] = (int)i;
}

}  // namespace dq
