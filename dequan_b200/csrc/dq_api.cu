// dq_api.cu — the C ABI (include/dequan_b200.h) over the CUDA engines.
// Host orchestration only: table upload, frontier expansion loop, kernel launches, result
// gathering.  No search runs on the CPU; every solve needs a CUDA device.
#include <algorithm>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "dequan_b200.h"
#include "dq_kernels.cuh"
#include "dq_lane_queens.cuh"
#include "dq_lane_sudoku.cuh"
#include "dq_reg_graphs.cuh"
#include "dq_group_graphs.cuh"
#include "dq_small_tree.cuh"
#include "dq_lane_tree.cuh"
#include "dq_model.hpp"

namespace dq {

static thread_local std::string g_err;
void set_last_error(const std::string& s) { g_err = s; }

#define DQ_CUDA(call)                                                                       \
    do {                                                                                    \
        cudaError_t e__ = (call);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            g_err = std::string(#call) + ": " + cudaGetErrorString(e__);                    \
            return DQ_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

// Device memory comes from a per-thread cache of freed blocks: compiling and solving a fresh model per call (the
// drop-in header's pattern: one CSP, one ForwardCheckingStep) must not pay cudaMalloc/cudaFree (each a device-wide
// synchronisation) every time.  Blocks go back to the driver only through trim(): when more than 8 GiB are parked, when
// cudaMalloc fails, and when a dq_solve_tree_multi worker ends.  At thread exit they are left to the driver.
struct BlockCache {
    struct Block { void* p; size_t bytes; int dev; };
    std::vector<Block> free_blocks;
    size_t cached_bytes = 0;
    cudaError_t take(size_t bytes, void** out) {
        int dev = 0;
        cudaGetDevice(&dev);
        size_t best = free_blocks.size();
        for (size_t i = 0; i < free_blocks.size(); i++) {
            const Block& b = free_blocks[i];
            if (b.dev != dev || b.bytes < bytes || b.bytes > 2 * bytes + (1u << 20)) continue;
            if (best == free_blocks.size() || b.bytes < free_blocks[best].bytes) best = i;
        }
        if (best != free_blocks.size()) {
            *out = free_blocks[best].p;
            cached_bytes -= free_blocks[best].bytes;
            free_blocks.erase(free_blocks.begin() + best);
            return cudaSuccess;
        }
        cudaError_t e = cudaMalloc(out, bytes);
        if (e != cudaSuccess && !free_blocks.empty()) {          // make room and try once more
            trim();
            e = cudaMalloc(out, bytes);
        }
        return e;
    }
    void give(void* p, size_t bytes, int dev) {
        if (dev < 0) cudaGetDevice(&dev);
        free_blocks.push_back(Block{p, bytes, dev});
        cached_bytes += bytes;
        if (cached_bytes > (size_t)8 << 30) trim();               // keep at most 8 GiB parked
    }
    void trim() {
        for (const Block& b : free_blocks) cudaFree(b.p);
        free_blocks.clear();
        cached_bytes = 0;
    }
    ~BlockCache() { /* the context may already be gone at thread exit: leave the blocks to the driver */ }
};
static thread_local BlockCache g_cache;

// A device block from the cache, handed back to it when the buffer is destroyed (or re-reserved).  A view does not own
// what it points to.
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0, bytes = 0;
    int dev = -1;                                        // the device the block lives on
    bool view = false;                                   // points into somebody else's block (never handed to the cache)
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap), bytes(o.bytes), dev(o.dev), view(o.view) { o.p = nullptr; o.cap = 0; o.bytes = 0; o.view = false; }
    ~DevBuf() { release(); }
    void set_view(T* q, size_t n) { release(); p = q; cap = n; bytes = 0; view = true; }
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        release();
        const size_t want = std::max<size_t>(n, 1) * sizeof(T);
        cudaError_t e = g_cache.take(want, (void**)&p);
        if (e == cudaSuccess) { cap = n; bytes = want; cudaGetDevice(&dev); }
        else p = nullptr;
        return e;
    }
    void release() { if (p && !view) g_cache.give(p, bytes, dev); p = nullptr; cap = 0; bytes = 0; view = false; }
};

// The pinned host words that queued copies read from and write to: a pageable target would cost a staging copy, and
// an asynchronous copy into pageable memory holds the calling thread until it is done.  Each use has its own words.
struct PinnedWords {
    struct {                                   // solve_queens_first
        unsigned long long key_nodes[2];       // best key, nodes
        uint8_t solution[32];
    } queens_first;
    struct {                                   // solve_queens_lane: the captured CUDA graph copies to and from these
        unsigned long long init[32];           // initial control block
        uint4 root;                            // root record
        unsigned long long ctrl[32];           // control block read back
        uint8_t first[32];                     // first-solution bytes
    } queens_lane;
    unsigned long long level_totals[2];        // solve_tree_generic: children and nodes of one frontier level
    unsigned long long head[38];               // k_expand_head's output, as far as it fits
    unsigned long long sudoku_max_blank;       // run_batch_sudoku: most blanks of an instance
    unsigned long long graphs_over;            // run_graphs_lane: longest overflow list
    unsigned long long graphs_ctrl[8];         // run_batch_graphs: control block read back
};
static_assert(sizeof(PinnedWords) <= 1024, "the pinned control words outgrew 1 KB");

// Stream + timing events are per thread and device, shared by every handle.
struct DeviceCtx {
    int dev = -1, sm_count = 0;
    cudaStream_t stream = nullptr, stream2 = nullptr;          // stream2: side work that overlaps the main queue
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;          // ordering only (no timing)
    PinnedWords* pin = nullptr;
};
// Never destroyed, like the streams, events and pinned words they hold: a handle keeps a pointer to the context of its
// first solve, also after the thread that created the context has ended.
static thread_local std::vector<DeviceCtx*> g_ctx;
static cudaError_t device_ctx(DeviceCtx** out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    for (DeviceCtx* c : g_ctx) if (c->dev == dev) { *out = c; return cudaSuccess; }
    DeviceCtx c;
    c.dev = dev;
    if ((e = cudaDeviceGetAttribute(&c.sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&c.ev0)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&c.ev1)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&c.ev2)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&c.ev3)) != cudaSuccess) return e;
    if ((e = cudaStreamCreateWithFlags(&c.stream2, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if ((e = cudaEventCreateWithFlags(&c.ev_fork, cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = cudaEventCreateWithFlags(&c.ev_join, cudaEventDisableTiming)) != cudaSuccess) return e;
    if ((e = cudaHostAlloc((void**)&c.pin, sizeof(PinnedWords), cudaHostAllocDefault)) != cudaSuccess) return e;
    g_ctx.push_back(new DeviceCtx(c));
    *out = g_ctx.back();
    return cudaSuccess;
}

// Waits for the stream when it goes out of scope.  Declared after a call's stack buffers, so that it runs before their
// destructors: a block goes back to the cache only once the queue that uses it has drained.
struct StreamDrain {
    cudaStream_t s;
    ~StreamDrain() { cudaStreamSynchronize(s); }
};

struct LevelArrays {               // kept per expansion level for FIRST-mode node accounting
    int n = 0;
    DevBuf<uint32_t> dmask, surv, child_off, parent_of;   // parent_of indexes the PREVIOUS level
    DevBuf<unsigned long long> dmask64, surv64;           // dmask / surv of models with 64-bit domain words
    DevBuf<unsigned long long> node_off;
    DevBuf<uint8_t> prefixes;      // [n][depth]
    void release_views() {
        auto drop = [](auto& b) { if (b.view) b.release(); };
        drop(dmask); drop(surv); drop(child_off); drop(parent_of); drop(dmask64); drop(surv64); drop(node_off); drop(prefixes);
    }
};

}  // namespace dq

using namespace dq;

struct MultiCtx;
static void multi_destroy(MultiCtx* mc);

struct dq_model {
    CompiledModel cm;
    DeviceCtx* ctx = nullptr;                   // the device context of the first solve; null until the tables are uploaded
    // the queue of one N-Queens solve (copies, level kernels, search, first solution) as an instantiated CUDA graph
    cudaGraphExec_t q_exec = nullptr;
    unsigned long long q_exec_key[6] = {0, 0, 0, 0, 0, 0}, q_seen_key[6] = {0, 0, 0, 0, 0, 0};
    // model tables in HBM
    DevBuf<uint8_t> d_blob;                     // all tables, one block
    std::vector<uint8_t> h_blob;                // its host image (kept while the copy may be in flight)
    uint32_t *t_ent_off = nullptr, *t_ent_moff = nullptr, *t_masks = nullptr, *t_dom0 = nullptr;   // masks / dom0: 64-bit words when cm.wide()
    bool last_wide = false;
    uint8_t* early_sol_host = nullptr;             // dq_solve_batch_cells: host buffer the solutions may be copied to as soon as they are final
    bool early_sol_done = false;
    bool last_queens_first = false;                 // the last solve was solve_queens_first (dq_tree_nodes_upto answers from its count)
    unsigned long long last_queens_first_nodes = 0;
    uint32_t* t_ent = nullptr;
    uint16_t *t_order = nullptr, *t_pos = nullptr;
    uint8_t* t_cell_lut = nullptr;
    int32_t *t_values = nullptr, *t_sizes = nullptr;
    uint32_t *t_s_and = nullptr, *t_s_weq = nullptr, *t_s_weq_on = nullptr, *t_s_chk = nullptr, *t_s_dom0 = nullptr;
    int n_sizes = 0;
    // tree-solve scratch, retained until the next solve for dq_tree_nodes_upto()
    std::vector<LevelArrays> levels;
    DevBuf<unsigned long long> d_ctrl;          // cursor, totals[2], best_key, scan totals[2], misc
    DevBuf<unsigned long long> d_sub_nodes, d_sol_key;
    DevBuf<uint8_t> d_sol;
    DevBuf<uint8_t> d_lvl_ptrs;                 // dq_tree_nodes_upto: 8-byte result + the per-level array pointers
    DevBuf<uint8_t> d_head;                     // k_expand_head: the first levels' arrays (views in `levels`) + its pointer table
    int head_levels = 0;                        // levels whose arrays live in d_head
    DevBuf<uint8_t> e_out;                      // dq_enumerate_solutions: [cap][nv] value indices
    DevBuf<unsigned long long> e_prefix, e_seq; // ... and their place in the DFS order
    int last_depth = 0;
    unsigned long long last_n_prefix = 0;
    int last_part_rank = 0, last_part_count = 1;
    // lane engine scratch
    DevBuf<uint4> q_records, q_records2;
    DevBuf<uint8_t> q_first;
    // batch scratch
    DevBuf<uint8_t> b_cells, b_solution, b_status;
    DevBuf<unsigned long long> b_nodes;
    DevBuf<unsigned long long> b_nsol;          // dq_count_batch_cells: solutions per instance
    // sudoku lane engine scratch (task pool)
    DevBuf<SudokuDigest> s_digest;
    DevBuf<unsigned long long> s_ctrl;
    DevBuf<uint32_t> s_hard;
    DevBuf<SudokuTask> s_tasks;
    DevBuf<uint4> s_snaps;
    DevBuf<uint32_t> s_snap_state;
    DevBuf<int> s_deferred;
    unsigned long long s_tasks_used = 0;
    // dq_solve_tree_multi: one worker thread + one clone of the compiled model per device
    struct MultiCtx* multi = nullptr;
    ~dq_model() {
        if (multi) multi_destroy(multi);
        if (q_exec) cudaGraphExecDestroy(q_exec);
    }
};

namespace dq {

// A handle is bound to the device (and thread) of its first solve: its stream, events and cached blocks live there.
static int check_bound(const dq_model* m, int dev) {
    if (m->ctx && dev != m->ctx->dev) { g_err = "model handle is bound to CUDA device " + std::to_string(m->ctx->dev) + " (dq_set_device before the first solve)"; return DQ_ERR_INVALID; }
    return DQ_OK;
}

// Appends one table to a host image at the next multiple of `align` bytes (at least 4 bytes, zero-filled).
template <class V>
static size_t put_table(std::vector<uint8_t>& blob, const V& vec, size_t align) {
    const size_t off = (blob.size() + align - 1) & ~(align - 1);
    blob.resize(off + std::max<size_t>(vec.size() * sizeof(vec[0]), 4), 0);
    if (!vec.empty()) memcpy(blob.data() + off, vec.data(), vec.size() * sizeof(vec[0]));
    return off;
}

// The generic tree engine's tables of one model, in this order: ent_off, ent, ent_moff, masks and dom0 (32-bit words, or
// 64-bit when the model is wide), order and pos (16-bit).  upload() and dq_solve_models both pack them here.
struct TreeTableOffsets { size_t ent_off, ent, ent_moff, masks, dom0, order, pos; };
static TreeTableOffsets put_tree_tables(const CompiledModel& c, std::vector<uint8_t>& blob, size_t align) {
    const int nv = c.nv;
    std::vector<uint16_t> order(nv), pos(nv);
    for (int i = 0; i < nv; i++) { order[i] = (uint16_t)c.order[i]; pos[i] = (uint16_t)c.pos_of[i]; }
    // domain words on the device: 32 bits unless some domain has more than 32 values
    std::vector<uint32_t> masks32, dom032;
    if (!c.wide()) { masks32.assign(c.masks.begin(), c.masks.end()); dom032.assign(c.dom0.begin(), c.dom0.end()); }
    TreeTableOffsets o;
    o.ent_off = put_table(blob, c.ent_off, align);
    o.ent = put_table(blob, c.ent, align);
    o.ent_moff = put_table(blob, c.ent_moff, align);
    o.masks = c.wide() ? put_table(blob, c.masks, align) : put_table(blob, masks32, align);
    o.dom0 = c.wide() ? put_table(blob, c.dom0, align) : put_table(blob, dom032, align);
    o.order = put_table(blob, order, align);
    o.pos = put_table(blob, pos, align);
    return o;
}

static int upload(dq_model* m) {
    int dev = 0;
    DQ_CUDA(cudaGetDevice(&dev));
    if (m->ctx) return check_bound(m, dev);
    DeviceCtx* ctx = nullptr;
    DQ_CUDA(device_ctx(&ctx));
    const CompiledModel& c = m->cm;
    const int nv = c.nv;
    // every table goes into ONE device block with ONE stream-ordered copy (the solve's kernels follow on the same stream)
    std::vector<int32_t> values((size_t)nv * 32, 0);
    std::vector<uint8_t> lut((size_t)nv * 256, 0xFF);
    for (int v = 0; v < nv; v++)
        for (size_t j = 0; j < c.values[v].size(); j++) {
            if (j < 32) values[(size_t)v * 32 + j] = c.values[v][j];     // (batch kernels: 32-bit models only)
            if (c.values[v][j] >= 1 && c.values[v][j] <= 255) lut[(size_t)v * 256 + c.values[v][j]] = (uint8_t)j;
        }
    std::vector<int32_t> sizes = c.distinct_sizes;
    if (std::find(sizes.begin(), sizes.end(), 1) == sizes.end()) sizes.push_back(1);
    std::sort(sizes.begin(), sizes.end());
    m->n_sizes = (int)sizes.size();
    std::vector<uint8_t>& blob = m->h_blob;
    blob.clear();
    auto put = [&](const auto& vec) -> size_t { return put_table(blob, vec, 256); };
    const TreeTableOffsets t = put_tree_tables(c, blob, 256);
    const size_t o_values = put(values), o_lut = put(lut), o_sizes = put(sizes);
    std::vector<uint32_t> dom0_pos(32, 0xFFFFFFFFu);
    for (int p = 0; p < nv && p < 32; p++) dom0_pos[p] = (uint32_t)c.dom0[c.order[p]];
    const size_t o_s_and = put(c.small_and), o_s_weq = put(c.small_weq), o_s_weq_on = put(c.small_weq_on), o_s_chk = put(c.small_chk),
                 o_s_dom0 = put(dom0_pos);
    DQ_CUDA(m->d_blob.reserve(blob.size()));
    DQ_CUDA(cudaMemcpyAsync(m->d_blob.p, blob.data(), blob.size(), cudaMemcpyHostToDevice, ctx->stream));
    uint8_t* base = m->d_blob.p;
    m->t_ent_off = (uint32_t*)(base + t.ent_off); m->t_ent = (uint32_t*)(base + t.ent); m->t_ent_moff = (uint32_t*)(base + t.ent_moff);
    m->t_masks = (uint32_t*)(base + t.masks); m->t_dom0 = (uint32_t*)(base + t.dom0); m->t_order = (uint16_t*)(base + t.order); m->t_pos = (uint16_t*)(base + t.pos);
    m->t_values = (int32_t*)(base + o_values); m->t_cell_lut = base + o_lut; m->t_sizes = (int32_t*)(base + o_sizes);
    m->t_s_and = (uint32_t*)(base + o_s_and); m->t_s_weq = (uint32_t*)(base + o_s_weq); m->t_s_weq_on = (uint32_t*)(base + o_s_weq_on);
    m->t_s_chk = (uint32_t*)(base + o_s_chk); m->t_s_dom0 = (uint32_t*)(base + o_s_dom0);
    DQ_CUDA(m->d_ctrl.reserve(32));
    m->ctx = ctx;
    return DQ_OK;
}

typedef unsigned long long W64;     // the device's 64-bit domain word

template <typename W>
static TreeModelDevT<W> dev_model_t(const dq_model* m) {
    TreeModelDevT<W> M;
    M.T.nv = m->cm.nv;
    M.T.ent_off = m->t_ent_off;
    M.T.ent = m->t_ent;
    M.T.ent_moff = m->t_ent_moff;
    M.T.masks = reinterpret_cast<const W*>(m->t_masks);
    M.dom0 = reinterpret_cast<const W*>(m->t_dom0);
    M.order = m->t_order;
    M.pos = m->t_pos;
    M.trail = m->cm.trail_bound;
    return M;
}
static TreeModelDev dev_model(const dq_model* m) { return dev_model_t<uint32_t>(m); }

template <typename W> struct LevelWords;
template <> struct LevelWords<uint32_t> {
    static DevBuf<uint32_t>& dmask(LevelArrays& L) { return L.dmask; }
    static DevBuf<uint32_t>& surv(LevelArrays& L) { return L.surv; }
};
template <> struct LevelWords<W64> {
    static DevBuf<W64>& dmask(LevelArrays& L) { return L.dmask64; }
    static DevBuf<W64>& surv(LevelArrays& L) { return L.surv64; }
};

// Calls f(has_f, has_table) with the model's feature flags as std::bool_constant, so that f can name the kernel
// instantiation for them: with_features(m->cm, [&](auto hf, auto ht) { k<hf, ht><<<...>>>(...); }).
template <class F>
static auto with_features(bool has_f, bool has_table, F&& f) {
    if (has_f) return has_table ? f(std::true_type{}, std::true_type{}) : f(std::true_type{}, std::false_type{});
    return has_table ? f(std::false_type{}, std::true_type{}) : f(std::false_type{}, std::false_type{});
}
template <class F>
static auto with_features(const CompiledModel& cm, F&& f) { return with_features(cm.has_f, cm.has_table, std::forward<F>(f)); }

template <class K>
static int max_ctas_per_sm(K kernel, int threads, size_t smem, int* out) {
    // (always the device's full opt-in size, never the size asked for: several host threads may be sizing launches of the
    // same kernel at once — dq_solve_tree_multi — and the attribute is per kernel, not per launch)
    if (smem > 48 * 1024) DQ_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DQ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(out, kernel, threads, smem));
    return DQ_OK;
}

// FIRST mode on a CLASS_QUEENS model, whole tree in one partition, no node budget: one warp walks the reference's own
// DFS (k_queens_first_nodes) — the solution, and every value tried on the way counted as the node it is.  One launch, one
// synchronisation; the generic path's prefix split searches the winning subtree with one warp as well, after paying for
// the frontier and for the subtrees that hold nothing (20-Queens: 43 ms there).
static int solve_queens_first(dq_model* m, dq_tree_result* res, int32_t* first_solution) {
    const int N = m->cm.queens_n;
    DeviceCtx* ctx = m->ctx;
    DQ_CUDA(m->q_first.reserve(32));
    DQ_CUDA(m->d_ctrl.reserve(32));
    unsigned long long* ctrl = m->d_ctrl.p;
    auto& P = ctx->pin->queens_first;
    unsigned long long* h = P.key_nodes;
    h[0] = KEY_NONE; h[1] = 0;
    QueensLaneArgs A;
    A.n = N; A.k = 0; A.part_rank = 0; A.part_count = 1; A.part_level = -1;
    A.records = nullptr; A.record_cap = 0; A.n_records = nullptr; A.cursor = nullptr; A.totals = nullptr; A.dfs_nodes = nullptr;
    A.best_key = ctrl + 3; A.first_out = m->q_first.p;
    DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    DQ_CUDA(cudaMemcpyAsync(ctrl + 3, h, sizeof P.key_nodes, cudaMemcpyHostToDevice, ctx->stream));
    k_queens_first_nodes<<<1, 32, 0, ctx->stream>>>(A, ctrl + 4);
    DQ_CUDA(cudaGetLastError());
    DQ_CUDA(cudaMemcpyAsync(h, ctrl + 3, sizeof P.key_nodes, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaMemcpyAsync(P.solution, m->q_first.p, sizeof P.solution, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    const bool found = h[0] != KEY_NONE;
    res->kernel_ms = ms; res->search_kernel_ms = 0; res->kernel_launches = 1; res->frontier_nodes = 0;
    res->engine_used = DQ_ENGINE_LANE; res->split_depth_used = 0; res->n_prefixes = 1;
    res->n_solutions = found ? 1 : 0; res->n_nodes = h[1]; res->first_key = found ? 0 : KEY_NONE;
    res->outcome = found ? DQ_SAT : DQ_UNSAT;
    if (found && first_solution)
        for (int i = 0; i < N; i++) first_solution[i] = m->cm.values[i][P.solution[i]];
    m->last_queens_first = true; m->last_queens_first_nodes = h[1];
    m->last_n_prefix = 0; m->last_depth = 0;
    return DQ_OK;
}

// COUNT_ALL on a CLASS_QUEENS model with the lane-per-subtree engine: K level kernels + DFS + first-solution
// kernel queued back to back, one host synchronisation at the end.
static int solve_queens_lane(dq_model* m, const dq_tree_opts* opts, dq_tree_result* res, int32_t* first_solution) {
    const int N = m->cm.queens_n;
    DeviceCtx* ctx = m->ctx;
    // Split depth: measured per board size on B200 (scripts/sweep_k.py, profiles/r2_queens_split_depth.txt), see below.
    int K = 0;
    // estimated FC-surviving prefixes per depth (sizes the record lists): each level multiplies by about N - 2.2*depth
    auto estimate = [&](int k) { double e = 1; for (int i = 0; i < k; i++) e *= std::max(N - 2.2 * i, 3.6); return e; };
    int occ = 0;
    int rc = DQ_OK;
    if (opts->split_depth > 0) K = std::min(opts->split_depth, std::min(N - 3, 12));
    else {
        // measured per N (scripts/sweep_k.py, profiles/r2_queens_split_depth.txt): small boards are bound by the launches of
        // the levels, large ones by keeping the pools fed to the end; the same depths serve the partitions of a strongly
        // scaled solve (scripts/parts_k.py: 17-Queens in 8 partitions, slowest partition 1.52 / 1.38 / 1.43 ms at depth 7 / 8 / 9)
        if (N <= 13) K = std::max(N - 8, 0);
        else if (N <= 16) K = 7;                   // 14: 0.179 ms (depth 5: 0.172 with a bucket kernel twice as long: the step is
                                                   // bound by the first-solution warp either way); 15: 0.34 ms (depth 6 / 8: 0.40 /
                                                   // 0.38); 16: 1.51 ms (depth 8: 1.55)
        else K = 8;                                // 17: 35 M records, 9.65 ms (depth 7 / 9: 9.68 / 10.24; the levels cost 0.16 / 0.44 / 1.44 ms)
    }
    // (the bucket search reads no prefix keys from its records — its first-solution warp computes 64-bit keys, and the
    // partition deal happens at depth <= 5 — so the split may go deeper than 32-bit keys would allow)
    // warps per CTA chosen so that the pools (buckets x 128 frames x 16 B per warp) pack an SM's shared memory best
    int bucket_warps = 4;
    // up to eight buckets (variables k+1 .. N-3; the records themselves stay in registers): the kernel compiled for exactly
    // that many; more: the general one (variables k .. N-3)
    typedef void (*BucketKernel)(QueensLaneArgs);
    // rows 1 .. 5 of the forward check in shifted frames (left shifts only, the FMA pipe), the rest plain (the ALU pipe):
    // the mix that balances the two pipes (measured: 0 / 3 / 4 / 5 / 6 / 7 / all rows shifted give 12.6 / 9.98 / 10.11 /
    // 9.65 / 9.79 / 9.80 / 9.81 ms on 17-Queens at split depth 8); exact while N + 2 * 5 <= 32
#define DQ_QB_ROW(J) {nullptr, k_queens_bucket_t<1, J>, k_queens_bucket_t<2, J>, k_queens_bucket_t<3, J>, k_queens_bucket_t<4, J>, \
                      k_queens_bucket_t<5, J>, k_queens_bucket_t<6, J>, k_queens_bucket_t<7, J>, k_queens_bucket_t<8, J>}
    static const BucketKernel kBucketKernels[2][9] = {DQ_QB_ROW(0), DQ_QB_ROW(5)};
#undef DQ_QB_ROW
    // DQ_QUEENS_PLAIN_ROWS=1 (test hook): the plain-row kernels on every board, so that boards a test can count reach the
    // kernels that boards of 23 and more queens get
    static const bool plain_rows = getenv("DQ_QUEENS_PLAIN_ROWS") != nullptr;
    const bool compiled = N - 3 - K >= 1 && N - 3 - K <= 8;
    const int n_buckets = compiled ? N - 3 - K : N - 2 - K;
    const BucketKernel bucket_kernel = compiled ? kBucketKernels[(N + 10 <= 32 && !plain_rows) ? 1 : 0][n_buckets] : k_queens_bucket;
    const size_t per_warp = (size_t)n_buckets * kQueensBucketCap * sizeof(uint4);
    {
        int best = 0;
        for (int w = 2; w <= kQueensBucketMaxWarps; w++) {
            if (per_warp * w > 200 * 1024) break;
            int o = 0;
            rc = max_ctas_per_sm(bucket_kernel, w * 32, per_warp * w, &o);
            if (rc != DQ_OK) return rc;
            if (o * w > best) { best = o * w; bucket_warps = w; occ = o; }
        }
        if (best == 0) { g_err = "board too large for the shared-memory pools"; return DQ_ERR_UNSUPPORTED; }
    }
    const size_t smem = per_warp * bucket_warps;
    if (occ < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    const int ctas = occ * ctx->sm_count;
    DQ_CUDA(m->q_first.reserve(32));
    DQ_CUDA(m->d_ctrl.reserve(32));
    size_t cap = std::max<size_t>(m->q_records.cap, (size_t)std::min(std::max(2.5 * estimate(K), 1024.0), 512.0 * 1024 * 1024));
    // control words live in pinned host memory that outlives the call: the queue below may be replayed as a CUDA graph
    auto& P = ctx->pin->queens_lane;
    unsigned long long* h_init = P.init;
    uint4* h_root = &P.root;
    unsigned long long* h_ctrl = P.ctrl;
    uint8_t* h_first = P.first;
    unsigned long long* ctrl = m->d_ctrl.p;     // [0]=cursor [1]=sols [2]=nodes [3]=best [8+l]=frontier size at depth l
    unsigned long long launches = 0, h_frontier_nodes = 0;
    float ms_total = 0, ms_search = 0;
    constexpr int kQueensPartLevel = 4;                     // measured: depth-5 keys balance 2/4/8 partitions within 3 %
    const int part_level = std::min(K - 1, kQueensPartLevel);
    // levels 0 .. head-1 in one single-CTA launch (a few hundred records at most, all above the partition level)
    const int head = std::max(0, std::min(std::min(K, part_level), 3));
    for (int attempt = 0; attempt < 3; attempt++) {
        DQ_CUDA(m->q_records.reserve(cap));
        DQ_CUDA(m->q_records2.reserve(m->q_records.cap));
        const size_t rcap = std::min(m->q_records.cap, m->q_records2.cap);
        uint4* buf[2] = {m->q_records.p, m->q_records2.p};
        QueensLaneArgs A;
        A.n = N; A.k = K;
        A.part_rank = opts->part_rank; A.part_count = opts->part_count;
        A.part_level = part_level;
        A.records = buf[K & 1]; A.record_cap = rcap; A.n_records = ctrl + 8 + K;
        A.cursor = ctrl + 0; A.totals = ctrl + 1; A.best_key = ctrl + 3; A.dfs_nodes = ctrl + 24;
        A.first_out = m->q_first.p;
        for (int i = 0; i < 32; i++) h_init[i] = 0;
        h_init[3] = KEY_NONE;
        h_init[8] = (K > 0 || opts->part_rank == 0) ? 1 : 0;   // the root prefix (key 0) belongs to partition 0
        *h_root = make_uint4(0, 0, 0, 0);

        // The queue of one solve: nothing in it comes back to the host before the end.
        // Multi-GPU: the frontier is dealt to the partitions (key mod parts) as soon as it is wide enough to balance —
        // below that level every partition expands only its own records, above it all of them expand the same few
        // hundred thousand records and partition 0 alone counts their nodes.
        // (timing events cannot be read back from inside a graph: the graph is bracketed by ev0 / ev1 from outside, and the
        // per-kernel pair ev2 / ev3 exists only in the call-by-call queue, DQ_TREE_TIME_KERNELS)
        auto enqueue = [&](const bool with_events) -> int {
            if (with_events) DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
            DQ_CUDA(cudaMemcpyAsync(ctrl, h_init, sizeof P.init, cudaMemcpyHostToDevice, ctx->stream));
            DQ_CUDA(cudaMemcpyAsync(buf[0], h_root, sizeof(uint4), cudaMemcpyHostToDevice, ctx->stream));
            // the DFS-first solution needs nothing from the frontier: one warp looks for it on the side stream
            DQ_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
            DQ_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
            k_queens_first_warp<<<1, 32, 0, ctx->stream2>>>(A);
            DQ_CUDA(cudaEventRecord(ctx->ev_join, ctx->stream2));
            if (head > 0)
                k_queens_levels_head<<<1, kQueensBlock, 0, ctx->stream>>>(A, head, buf[0], buf[1], ctrl + 8, opts->part_rank == 0 ? 1 : 0);
            for (int l = head; l < K; l++) {
                const int grid = (int)std::min<double>(std::max(estimate(l) * N / kQueensBlock, 1.0), (double)ctx->sm_count * 8);
                const int count_nodes = (l > part_level || opts->part_rank == 0) ? 1 : 0;
                // wide frontiers: lane per record (k_queens_level_wide); narrow ones: lane per (record, value) pair
                if (estimate(l) >= 150000.0) {      // (below that the pair kernel's single trip has the shorter latency)
                    const int wgrid = (int)std::min<double>(std::max(estimate(l) / kQueensBlock, 1.0), (double)ctx->sm_count * 8);
                    k_queens_level_wide<<<wgrid, kQueensBlock, 0, ctx->stream>>>(A, l, buf[l & 1], ctrl + 8 + l, buf[(l + 1) & 1], ctrl + 8 + l + 1,
                                                                                count_nodes, (l == part_level && opts->part_count > 1) ? 1 : 0);
                } else
                k_queens_level<<<grid, kQueensBlock, 0, ctx->stream>>>(A, l, buf[l & 1], ctrl + 8 + l, buf[(l + 1) & 1], ctrl + 8 + l + 1,
                                                                       count_nodes, (l == part_level && opts->part_count > 1) ? 1 : 0);
            }
            if (with_events) DQ_CUDA(cudaEventRecord(ctx->ev2, ctx->stream));
            bucket_kernel<<<ctas, bucket_warps * 32, smem, ctx->stream>>>(A);
            if (with_events) DQ_CUDA(cudaEventRecord(ctx->ev3, ctx->stream));
            DQ_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
            DQ_CUDA(cudaGetLastError());
            DQ_CUDA(cudaMemcpyAsync(h_ctrl, ctrl, sizeof P.ctrl, cudaMemcpyDeviceToHost, ctx->stream));
            DQ_CUDA(cudaMemcpyAsync(h_first, m->q_first.p, sizeof P.first, cudaMemcpyDeviceToHost, ctx->stream));
            if (with_events) DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
            return DQ_OK;
        };
        launches += (K - head) + (head > 0 ? 1 : 0) + 2;

        // One graph launch instead of ~20 API calls (a 14-Queens solve is 0.16 ms of kernels): the queue is captured once
        // per (model, split, partition, buffers) and replayed; anything that changes one of those re-captures it.
        bool queued = false;
        const bool time_kernels = (opts->flags & DQ_TREE_TIME_KERNELS) != 0;
        if (!time_kernels) {
            const unsigned long long key[6] = {(unsigned long long)K | ((unsigned long long)opts->part_rank << 16) | ((unsigned long long)opts->part_count << 32),
                                               (unsigned long long)rcap, (unsigned long long)(uintptr_t)buf[0], (unsigned long long)(uintptr_t)buf[1],
                                               (unsigned long long)(uintptr_t)ctrl, (unsigned long long)(uintptr_t)m->q_first.p};
            // a model solved once (the drop-in path compiles, solves, frees) is not worth a capture: the graph is built when
            // the same queue comes round a second time
            const bool seen = memcmp(key, m->q_seen_key, sizeof key) == 0;
            memcpy(m->q_seen_key, key, sizeof key);
            if (seen && (!m->q_exec || memcmp(key, m->q_exec_key, sizeof key) != 0)) {
                if (m->q_exec) { cudaGraphExecDestroy(m->q_exec); m->q_exec = nullptr; }
                cudaGraph_t graph = nullptr;
                if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                    const int qrc = enqueue(false);
                    const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
                    if (qrc == DQ_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&m->q_exec, graph, 0) == cudaSuccess)
                        memcpy(m->q_exec_key, key, sizeof key);
                    else m->q_exec = nullptr;
                    if (graph) cudaGraphDestroy(graph);
                }
                (void)cudaGetLastError();                      // a failed capture falls back to the plain queue below
            }
            if (m->q_exec && memcmp(key, m->q_exec_key, sizeof key) == 0) {
                DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
                if (cudaGraphLaunch(m->q_exec, ctx->stream) == cudaSuccess) { queued = true; DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream)); }
                else (void)cudaGetLastError();
            }
        }
        if (!queued) {
            rc = enqueue(true);
            if (rc != DQ_OK) return rc;
        }
        DQ_CUDA(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        ms_total += ms;
        if (!queued) DQ_CUDA(cudaEventElapsedTime(&ms_search, ctx->ev2, ctx->ev3));
        h_frontier_nodes = h_ctrl[2];
        unsigned long long biggest = 0;
        for (int l = 0; l <= K; l++) biggest = std::max(biggest, h_ctrl[8 + l]);
        if (biggest <= rcap) break;
        // a frontier overflowed its list: grow (the last level's count is exact only if the earlier ones fitted) and rerun
        if (biggest > 512ull * 1024 * 1024) { g_err = "frontier of more than 2^29 records: lower split_depth"; return DQ_ERR_UNSUPPORTED; }
        cap = (size_t)std::min<unsigned long long>(std::max<unsigned long long>(biggest, 2 * rcap), 512ull * 1024 * 1024);
        if (attempt == 2) { g_err = "internal: record list overflow persists"; return DQ_ERR_INTERNAL; }
    }
    res->kernel_ms = ms_total;
    res->search_kernel_ms = ms_search;
    res->frontier_nodes = h_frontier_nodes;
    res->kernel_launches = launches;
    res->engine_used = DQ_ENGINE_LANE;
    res->split_depth_used = K;
    res->n_prefixes = (int32_t)std::min<unsigned long long>(h_ctrl[8 + K], 0x7FFFFFFF);
    res->n_solutions = h_ctrl[1];
    res->n_nodes = h_ctrl[2] + h_ctrl[24];
    res->first_key = h_ctrl[3];
    res->outcome = res->n_solutions ? DQ_SAT : DQ_UNSAT;
    m->last_n_prefix = 0; m->last_depth = 0;
    if (h_ctrl[3] != KEY_NONE && first_solution)
        for (int v = 0; v < N; v++) first_solution[v] = m->cm.values[v][h_first[v]];
    return DQ_OK;
}

}  // namespace dq

extern "C" {

const char* dq_last_error(void) { return g_err.c_str(); }
const char* dq_version(void) { return "dequan_b200 0.1 (sm_100a)"; }

int dq_device_info(int32_t* sm_count, int32_t* cc, char* name, size_t name_len) {
    int dev = 0;
    DQ_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    DQ_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc) *cc = p.major * 10 + p.minor;
    if (name && name_len) { strncpy(name, p.name, name_len - 1); name[name_len - 1] = 0; }
    return DQ_OK;
}

int dq_set_device(int32_t ordinal) {
    DQ_CUDA(cudaSetDevice(ordinal));
    return DQ_OK;
}

int dq_compile(const dq_model_desc* desc, dq_model** out) {
    if (!out) { g_err = "null out"; return DQ_ERR_INVALID; }
    *out = nullptr;
    dq_model* m = new (std::nothrow) dq_model();
    if (!m) return DQ_ERR_NOMEM;
    std::string err;
    int rc = compile_model(desc, m->cm, err);
    if (rc != DQ_OK) { g_err = err; delete m; return rc; }
    *out = m;
    return DQ_OK;
}

void dq_free(dq_model* m) { delete m; }

int dq_model_info(const dq_model* m, int32_t* n_vars, int32_t* max_dom, int32_t* n_arcs, int32_t* model_class) {
    if (!m) { g_err = "null model"; return DQ_ERR_INVALID; }
    if (n_vars) *n_vars = m->cm.nv;
    if (max_dom) *max_dom = m->cm.kmax;
    if (n_arcs) *n_arcs = (int32_t)m->cm.ent.size();
    if (model_class) *model_class = m->cm.model_class;
    return DQ_OK;
}

int dq_model_order(const dq_model* m, int32_t* order_out) {
    if (!m || !order_out) { g_err = "null argument"; return DQ_ERR_INVALID; }
    for (int i = 0; i < m->cm.nv; i++) order_out[i] = m->cm.order[i];
    return DQ_OK;
}

int dq_model_table_bytes(const dq_model* m, uint64_t* bytes) {
    if (!m || !bytes) { g_err = "null argument"; return DQ_ERR_INVALID; }
    const CompiledModel& c = m->cm;
    *bytes = c.ent_off.size() * 4 + c.ent.size() * 4 + c.ent_moff.size() * 4 + c.masks.size() * (c.wide() ? 8 : 4) + c.dom0.size() * (c.wide() ? 8 : 4) +
             (size_t)c.nv * 2 + (size_t)c.nv * 32 * 4 + (size_t)c.nv * 256 + c.distinct_sizes.size() * 4 + 4;
    return DQ_OK;
}

}  // extern "C" (templates follow)

// node budget of the root probe of dq_solve_tree
constexpr unsigned long long kProbeNodes = 512;

// enumeration request of dq_enumerate_solutions (null for a plain solve)
struct EnumRequest {
    int32_t* out;                    // [cap][nv] values by var id, DFS order
    uint64_t cap;
    uint64_t written;
};

// The generic path (any compiled model): frontier expansion level by level, then the subtree DFS.  W = domain word type.
template <typename W>
static int solve_tree_generic(dq_model* m, const dq_tree_opts* opts, dq_tree_result* res, int32_t* first_solution, EnumRequest* er,
                              const bool count_all) {
    const int nv = m->cm.nv;
    DeviceCtx* ctx = m->ctx;
    int rc = DQ_OK;
    TreeModelDevT<W> M = dev_model_t<W>(m);
    m->last_wide = sizeof(W) == 8;
    const size_t wbytes = warp_state_bytes(nv, M.trail, sizeof(W));
    // warps per CTA: four, fewer when the per-warp state (domains + trail) of a large model would not fit a CTA
    const int wpc = (int)std::min<size_t>(kWarpsPerCta, (200 * 1024) / wbytes);
    if (wpc < 1) { g_err = "model state exceeds shared memory"; return DQ_ERR_UNSUPPORTED; }
    const size_t smem = wbytes * wpc;
    int occ = 0;
    rc = with_features(m->cm, [&](auto hf, auto ht) { return max_ctas_per_sm(k_tree_dfs<hf, ht, W>, wpc * 32, smem, &occ); });
    if (rc != DQ_OK) return rc;
    int occ_e = 0;
    rc = with_features(m->cm, [&](auto hf, auto ht) { return max_ctas_per_sm(k_expand<hf, ht, W>, wpc * 32, smem, &occ_e); });
    if (rc != DQ_OK) return rc;
    if (occ < 1 || occ_e < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    const long long resident_warps = (long long)occ * ctx->sm_count * wpc;
    const int max_depth = nv - 1;
    const int want_depth = opts->split_depth > 0 ? std::min(opts->split_depth, max_depth) : -1;
    // lane-per-subtree counting (dq_lane_tree.cuh) for small models whose pair filters are plain AND masks
    bool lanes = count_all && !er && sizeof(W) == 4 && m->cm.small_ok && !m->cm.has_f && m->cm.kmax <= kLaneTreeMaxDom &&
                 lane_tree_smem(nv, m->cm.kmax) <= 200 * 1024 && (opts->engine == DQ_ENGINE_AUTO || opts->engine == DQ_ENGINE_LANE);
    if (opts->engine == DQ_ENGINE_LANE && !lanes) { g_err = "the lane engine counts the trees of small models with plain AND filters (or the N-Queens class)"; return DQ_ERR_UNSUPPORTED; }
    int occ_l = 0;
    if (lanes) {
        rc = max_ctas_per_sm(k_tree_lanes, kLaneTreeThreads, lane_tree_smem(nv, m->cm.kmax), &occ_l);
        if (rc != DQ_OK) return rc;
        if (occ_l < 1) lanes = false;
    }
    // enough prefixes for 24 rounds of the resident warps — or, one subtree per lane, one round of the resident lanes
    // (2 or 4 rounds are no faster: profiles/r2_generic_lane_tree.txt)
    const long long want_prefixes = (lanes ? (long long)occ_l * ctx->sm_count * kLaneTreeThreads : resident_warps * 24) * opts->part_count;

    if (er) {
        DQ_CUDA(m->e_out.reserve(std::max<size_t>((size_t)er->cap * nv, 1)));
        DQ_CUDA(m->e_prefix.reserve(std::max<size_t>(er->cap, 1)));
        DQ_CUDA(m->e_seq.reserve(std::max<size_t>(er->cap, 1)));
    }
    unsigned long long* ctrl = m->d_ctrl.p;   // [0]=cursor [1]=sols [2]=nodes [3]=best [4]=scan children [5]=scan nodes [6]=probe gave up [7]=enumerated
    unsigned long long h_ctrl[8] = {0, 0, 0, KEY_NONE, 0, 0, 0, 0};
    DQ_CUDA(cudaMemcpyAsync(ctrl, h_ctrl, sizeof h_ctrl, cudaMemcpyHostToDevice, ctx->stream));
    DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));

    if ((int)m->levels.size() < nv + 1) m->levels.resize(nv + 1);   // sized up front: references below stay valid
    m->levels[0].n = 1;
    DQ_CUDA(m->levels[0].prefixes.reserve(1));
    int depth = 0;
    unsigned long long shallow_nodes = 0, launches = 0;
    bool empty = false;
    long long n_warps = 0;

    // One launch of the subtree DFS over the prefixes of level `depth`: the register engine for small models
    // (dq_small_tree.cuh), the generic warp engine otherwise.  Sizes and clears the per-run buffers.
    if (opts->engine == DQ_ENGINE_REG && !m->cm.small_ok) { g_err = "the register engine serves models of at most 32 variables with simple pair filters"; return DQ_ERR_UNSUPPORTED; }
    const bool small = sizeof(W) == 4 && m->cm.small_ok && opts->engine != DQ_ENGINE_WARP;
    const size_t ssm = small ? small_tree_smem(nv, m->cm.kmax, m->cm.has_f, kWarpsPerCta) : 0;
    int socc = 0;
    if (small) {
        rc = m->cm.has_f ? max_ctas_per_sm(k_tree_small<true>, kWarpsPerCta * 32, ssm, &socc)
                         : max_ctas_per_sm(k_tree_small<false>, kWarpsPerCta * 32, ssm, &socc);
        if (rc != DQ_OK) return rc;
        if (socc < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    }
    auto launch_dfs = [&](int at_depth, unsigned long long n_prefix, int part_rank, int part_count, unsigned long long node_budget) -> int {
        const unsigned long long mine = (n_prefix + part_count - 1 - part_rank) / part_count;
        const bool by_lane = lanes && !node_budget && mine >= 2048;          // (a handful of prefixes: the warp-cooperative engines)
        const long long per_sm = by_lane ? occ_l : (small ? socc : occ);
        const int w_cta = by_lane ? kLaneTreeThreads : (small ? kWarpsPerCta : wpc);     // result slots per CTA: lanes or warps
        const long long ctas = std::max<long long>(1, std::min<long long>((long long)((mine + w_cta - 1) / w_cta), per_sm * ctx->sm_count));
        n_warps = ctas * w_cta;
        DQ_CUDA(m->d_sub_nodes.reserve(n_prefix));
        DQ_CUDA(m->d_sol_key.reserve(n_warps));
        DQ_CUDA(m->d_sol.reserve((size_t)n_warps * nv));
        DQ_CUDA(cudaMemsetAsync(m->d_sub_nodes.p, 0, n_prefix * sizeof(unsigned long long), ctx->stream));
        DQ_CUDA(cudaMemsetAsync(m->d_sol_key.p, 0xFF, n_warps * sizeof(unsigned long long), ctx->stream));
        TreeDfsArgs A;
        A.prefixes = m->levels[at_depth].prefixes.p; A.depth = at_depth; A.n_prefix = n_prefix;
        A.part_rank = part_rank; A.part_count = part_count; A.count_all = count_all ? 1 : 0;
        A.cursor = ctrl + 0; A.totals = ctrl + 1; A.best_key = ctrl + 3;
        A.sub_nodes = m->d_sub_nodes.p; A.sol_key = m->d_sol_key.p; A.sol = m->d_sol.p;
        A.node_budget = node_budget; A.gave_up = ctrl + 6;
        A.enum_out = er ? m->e_out.p : nullptr; A.enum_prefix = m->e_prefix.p; A.enum_seq = m->e_seq.p;
        A.enum_count = ctrl + 7; A.enum_cap = er ? er->cap : 0;
        if (by_lane) {
            SmallTablesDev ST;
            ST.nv = nv; ST.kmax = m->cm.kmax; ST.t_and = m->t_s_and; ST.t_weq = m->t_s_weq; ST.t_weq_on = m->t_s_weq_on;
            ST.t_chk = m->t_s_chk; ST.dom0_pos = m->t_s_dom0; ST.order = m->t_order;
            k_tree_lanes<<<(int)ctas, kLaneTreeThreads, lane_tree_smem(nv, m->cm.kmax), ctx->stream>>>(ST, A);
            res->engine_used = DQ_ENGINE_LANE;
        } else if (small) {
            SmallTablesDev ST;
            ST.nv = nv; ST.kmax = m->cm.kmax; ST.t_and = m->t_s_and; ST.t_weq = m->t_s_weq; ST.t_weq_on = m->t_s_weq_on;
            ST.t_chk = m->t_s_chk; ST.dom0_pos = m->t_s_dom0; ST.order = m->t_order;
            if (m->cm.has_f) k_tree_small<true><<<(int)ctas, kWarpsPerCta * 32, ssm, ctx->stream>>>(ST, A);
            else k_tree_small<false><<<(int)ctas, kWarpsPerCta * 32, ssm, ctx->stream>>>(ST, A);
            res->engine_used = DQ_ENGINE_REG;
        } else with_features(m->cm, [&](auto hf, auto ht) { k_tree_dfs<hf, ht, W><<<(int)ctas, wpc * 32, smem, ctx->stream>>>(M, A); });
        launches++;
        DQ_CUDA(cudaGetLastError());
        return DQ_OK;
    };

    // ---- root probe: ONE warp walks the whole tree under a small node budget ----
    // Most ForwardCheckingStep calls of a modelling session are small (the reference's own scenarios take 88-193
    // nodes): one launch and one synchronisation answer them, instead of a synchronisation per frontier level.
    // Past the budget the probe's counts are dropped and the split search below starts over.
    bool probed = false;
    if (want_depth < 0 && opts->part_count == 1 && !er) {
        rc = launch_dfs(0, 1, 0, 1, kProbeNodes);
        if (rc != DQ_OK) return rc;
        DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
        DQ_CUDA(cudaMemcpyAsync(h_ctrl, ctrl, sizeof h_ctrl, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CUDA(cudaStreamSynchronize(ctx->stream));
        if (h_ctrl[6] == 0) probed = true;
        else {
            const unsigned long long z[8] = {0, 0, 0, KEY_NONE, 0, 0, 0, 0};
            memcpy(h_ctrl, z, sizeof z);
            DQ_CUDA(cudaMemcpyAsync(ctrl, h_ctrl, sizeof h_ctrl, cudaMemcpyHostToDevice, ctx->stream));
        }
    }

    // ---- the forced head of the tree (one prefix per level) in one launch (k_expand_head) ----
    constexpr int kHeadCap = 1, kHeadMaxLevels = 96;
    if (!probed && max_depth > 0) {
        const int head_max = std::min(std::min(max_depth, kHeadMaxLevels), want_depth >= 0 ? want_depth : max_depth);
        // one slab: per level dmask, surv (W), child_off, parent_of (u32), node_off (u64), prefixes (cap x level bytes); then the table
        const size_t per_level = (size_t)kHeadCap * (2 * sizeof(W) + 4 + 4 + 8);
        size_t bytes = 0;
        std::vector<size_t> off_lvl(head_max + 2), off_pre(head_max + 2);
        for (int l = 0; l <= head_max; l++) { off_lvl[l] = bytes; bytes += per_level; off_pre[l] = bytes; bytes += ((size_t)kHeadCap * l + 15) & ~(size_t)15; }
        const size_t off_tab = bytes;
        bytes += (size_t)(head_max + 1) * sizeof(HeadLevel<W>);
        const size_t off_base = (bytes + 15) & ~(size_t)15;
        bytes = off_base + 2 * (size_t)nv * sizeof(W);
        if (m->d_head.cap < bytes || m->head_levels < head_max + 1) {
            for (auto& L : m->levels) L.release_views();     // views of the old slab go first
            DQ_CUDA(cudaStreamSynchronize(ctx->stream));
            DQ_CUDA(m->d_head.reserve(bytes));
            m->head_levels = head_max + 1;
        }
        std::vector<HeadLevel<W>> tab(head_max + 1);
        for (int l = 0; l <= head_max; l++) {
            uint8_t* b0 = m->d_head.p + off_lvl[l];
            LevelArrays& L = m->levels[l];
            HeadLevel<W>& H = tab[l];
            H.node_off = reinterpret_cast<unsigned long long*>(b0);
            H.dmask = reinterpret_cast<W*>(b0 + (size_t)kHeadCap * 8);
            H.surv = H.dmask + kHeadCap;
            H.child_off = reinterpret_cast<uint32_t*>(H.surv + kHeadCap);
            H.parent_of = H.child_off + kHeadCap;
            H.prefixes = m->d_head.p + off_pre[l];
            // the level arrays of `levels` become views of the slab unless they already own something at least as large
            if (LevelWords<W>::dmask(L).cap < (size_t)kHeadCap || LevelWords<W>::dmask(L).view) LevelWords<W>::dmask(L).set_view(H.dmask, kHeadCap); else H.dmask = LevelWords<W>::dmask(L).p;
            if (LevelWords<W>::surv(L).cap < (size_t)kHeadCap || LevelWords<W>::surv(L).view) LevelWords<W>::surv(L).set_view(H.surv, kHeadCap); else H.surv = LevelWords<W>::surv(L).p;
            if (L.child_off.cap < (size_t)kHeadCap || L.child_off.view) L.child_off.set_view(H.child_off, kHeadCap); else H.child_off = L.child_off.p;
            if (L.parent_of.cap < (size_t)kHeadCap || L.parent_of.view) L.parent_of.set_view(H.parent_of, kHeadCap); else H.parent_of = L.parent_of.p;
            if (L.node_off.cap < (size_t)kHeadCap || L.node_off.view) L.node_off.set_view(H.node_off, kHeadCap); else H.node_off = L.node_off.p;
            if (L.prefixes.cap < (size_t)kHeadCap * std::max(l, 1) || L.prefixes.view) L.prefixes.set_view(H.prefixes, (size_t)kHeadCap * std::max(l, 1)); else H.prefixes = L.prefixes.p;
        }
        HeadLevel<W>* d_tab = reinterpret_cast<HeadLevel<W>*>(m->d_head.p + off_tab);
        DQ_CUDA(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(HeadLevel<W>), cudaMemcpyHostToDevice, ctx->stream));
        DQ_CUDA(m->d_lvl_ptrs.reserve((size_t)(kHeadMaxLevels + 8) * 8 + 4096));
        unsigned long long* d_out = reinterpret_cast<unsigned long long*>(m->d_lvl_ptrs.p);
        int occ_h = 0;
        // (also lifts the 48 KB dynamic shared-memory limit)
        rc = with_features(m->cm, [&](auto hf, auto ht) { return max_ctas_per_sm(k_expand_head<hf, ht, W>, 32, wbytes, &occ_h); });
        if (rc != DQ_OK) return rc;
        W* base_D = reinterpret_cast<W*>(m->d_head.p + off_base);
        with_features(m->cm, [&](auto hf, auto ht) {
            k_expand_head<hf, ht, W><<<1, 32, wbytes, ctx->stream>>>(M, d_tab, head_max, base_D, base_D + nv, d_out);
        });
        launches++;
        unsigned long long* h_out = ctx->pin->head;
        const int n_read = std::min(4 + head_max + 1, (int)std::size(ctx->pin->head));
        DQ_CUDA(cudaMemcpyAsync(h_out, d_out, (size_t)n_read * 8, cudaMemcpyDeviceToHost, ctx->stream));
        std::vector<unsigned long long> h_all;
        if (4 + head_max + 1 > n_read) { h_all.resize(4 + head_max + 1); DQ_CUDA(cudaMemcpyAsync(h_all.data(), d_out, h_all.size() * 8, cudaMemcpyDeviceToHost, ctx->stream)); }
        DQ_CUDA(cudaStreamSynchronize(ctx->stream));
        DQ_CUDA(cudaGetLastError());
        const unsigned long long* ho = h_all.empty() ? h_out : h_all.data();
        depth = (int)ho[0];
        shallow_nodes += ho[1];
        for (int l = 0; l <= depth; l++) m->levels[l].n = (int)ho[4 + l];
        if (ho[2]) empty = true;
        if (depth > 0) { M.base_D = base_D; M.base_F = base_D + nv; M.base_depth = depth; }    // prefixes are replayed from the chain's end
    }

    // ---- frontier expansion, level by level, children kept in DFS order ----
  if (!probed && !empty) {
    while (depth < max_depth && (want_depth >= 0 ? depth < want_depth : m->levels[depth].n < want_prefixes)) {
        LevelArrays& L = m->levels[depth];
        const int n = L.n;
        DevBuf<W>& Ldmask = LevelWords<W>::dmask(L);
        DevBuf<W>& Lsurv = LevelWords<W>::surv(L);
        DQ_CUDA(Ldmask.reserve(n)); DQ_CUDA(Lsurv.reserve(n)); DQ_CUDA(L.child_off.reserve(n)); DQ_CUDA(L.node_off.reserve(n));
        const int grid = (n + wpc - 1) / wpc;
        with_features(m->cm, [&](auto hf, auto ht) {
            k_expand<hf, ht, W><<<grid, wpc * 32, smem, ctx->stream>>>(M, L.prefixes.p, depth, n, Ldmask.p, Lsurv.p);
        });
        k_scan_level<W><<<1, 1024, 0, ctx->stream>>>(Ldmask.p, Lsurv.p, n, L.child_off.p, L.node_off.p, ctrl + 4);
        launches += 2;
        unsigned long long* tot = ctx->pin->level_totals;
        DQ_CUDA(cudaMemcpyAsync(tot, ctrl + 4, sizeof ctx->pin->level_totals, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CUDA(cudaStreamSynchronize(ctx->stream));
        shallow_nodes += tot[1];
        if (tot[0] == 0) { empty = true; depth++; m->levels[depth].n = 0; break; }
        if (tot[0] > 0x7FFFFFFFull / (unsigned)(depth + 1)) { g_err = "frontier too large"; return DQ_ERR_NOMEM; }
        LevelArrays& C = m->levels[depth + 1];
        C.n = (int)tot[0];
        DQ_CUDA(C.prefixes.reserve((size_t)C.n * (depth + 1)));
        DQ_CUDA(C.parent_of.reserve(C.n));
        k_write_children<W><<<(n + 255) / 256, 256, 0, ctx->stream>>>(L.prefixes.p, depth, n, Lsurv.p, L.child_off.p, C.prefixes.p, C.parent_of.p);
        launches++;
        depth++;
    }
    DQ_CUDA(cudaGetLastError());

  }
    const unsigned long long n_prefix = empty ? 0 : (unsigned long long)m->levels[depth].n;
    m->last_depth = depth; m->last_n_prefix = n_prefix;
    m->last_part_rank = opts->part_rank; m->last_part_count = opts->part_count;
    res->n_prefixes = (int32_t)n_prefix;
    res->split_depth_used = depth;

    // ---- subtree DFS ----
    if (n_prefix && !probed) {
        DQ_CUDA(cudaEventRecord(ctx->ev2, ctx->stream));
        rc = launch_dfs(depth, n_prefix, opts->part_rank, opts->part_count, 0ull);
        if (rc != DQ_OK) return rc;
        DQ_CUDA(cudaEventRecord(ctx->ev3, ctx->stream));
    }
    if (!probed) {
        DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
        DQ_CUDA(cudaMemcpyAsync(h_ctrl, ctrl, sizeof h_ctrl, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    float ms = 0;
    DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    res->kernel_ms = ms;
    res->kernel_launches = launches;
    if (n_prefix && !probed) {                            // the subtree search alone (the frontier levels are the rest)
        DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev2, ctx->ev3));
        res->search_kernel_ms = ms;
    }

    const unsigned long long best = h_ctrl[3];
    res->first_key = best;
    const unsigned long long my_shallow = opts->part_rank == 0 ? shallow_nodes : 0;
    if (count_all) {
        res->n_solutions = h_ctrl[1];
        res->n_nodes = h_ctrl[2] + my_shallow;
        res->outcome = res->n_solutions ? DQ_SAT : DQ_UNSAT;
    } else {
        res->n_solutions = best != KEY_NONE ? 1 : 0;
        res->outcome = res->n_solutions ? DQ_SAT : DQ_UNSAT;
        uint64_t upto = 0;
        rc = dq_tree_nodes_upto(m, best, &upto);
        if (rc != DQ_OK) return rc;
        res->n_nodes = upto;
        res->nodes_before_first = upto;
    }
    if (best != KEY_NONE && first_solution) {
        std::vector<unsigned long long> keys(n_warps);
        DQ_CUDA(cudaMemcpy(keys.data(), m->d_sol_key.p, n_warps * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        long long w = -1;
        for (long long i = 0; i < n_warps; i++) if (keys[i] == best) { w = i; break; }
        if (w < 0) { g_err = "internal: winning solution not recorded"; return DQ_ERR_INTERNAL; }
        std::vector<uint8_t> sol(nv);
        DQ_CUDA(cudaMemcpy(sol.data(), m->d_sol.p + (size_t)w * nv, nv, cudaMemcpyDeviceToHost));
        for (int v = 0; v < nv; v++) first_solution[v] = m->cm.values[v][sol[v]];
    }
    if (er) {
        // solutions arrive in the order the warps found them; (prefix index, rank inside the subtree) is their DFS order
        const uint64_t found = h_ctrl[7];
        if (found != res->n_solutions) { g_err = "internal: enumeration count differs from the solution count"; return DQ_ERR_INTERNAL; }
        if (found > er->cap) { er->written = 0; g_err = "solution buffer too small (n_solutions holds the number needed)"; return DQ_ERR_NOMEM; }
        std::vector<uint8_t> raw((size_t)found * nv);
        std::vector<unsigned long long> pre(found), seq(found);
        if (found) {
            DQ_CUDA(cudaMemcpy(raw.data(), m->e_out.p, raw.size(), cudaMemcpyDeviceToHost));
            DQ_CUDA(cudaMemcpy(pre.data(), m->e_prefix.p, found * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            DQ_CUDA(cudaMemcpy(seq.data(), m->e_seq.p, found * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        }
        std::vector<uint64_t> idx(found);
        for (uint64_t i = 0; i < found; i++) idx[i] = i;
        std::sort(idx.begin(), idx.end(), [&](uint64_t x, uint64_t y) { return pre[x] != pre[y] ? pre[x] < pre[y] : seq[x] < seq[y]; });
        for (uint64_t i = 0; i < found; i++)
            for (int v = 0; v < nv; v++) er->out[i * nv + v] = m->cm.values[v][raw[idx[i] * nv + v]];
        er->written = found;
    }
    return DQ_OK;
}

static int solve_tree_impl(dq_model* m, const dq_tree_opts* opts, dq_tree_result* res, int32_t* first_solution, EnumRequest* er) {
    if (!m || !opts || !res) { g_err = "null argument"; return DQ_ERR_INVALID; }
    if (opts->part_count < 1 || opts->part_rank < 0 || opts->part_rank >= opts->part_count) { g_err = "bad partition"; return DQ_ERR_INVALID; }
    if (opts->node_budget) { g_err = "node_budget is a batch option; single-tree solves have none"; return DQ_ERR_UNSUPPORTED; }
    memset(res, 0, sizeof *res);
    const int nv = m->cm.nv;
    const int UNASSIGNED = -2147483647;
    res->first_key = KEY_NONE;
    res->engine_used = DQ_ENGINE_WARP;
    if (first_solution) for (int i = 0; i < nv; i++) first_solution[i] = UNASSIGNED;
    if (nv == 0) { res->outcome = DQ_SAT; res->n_solutions = 1; res->first_key = 0; if (er) er->written = er->cap ? 1 : 0; return DQ_OK; }   // IsComplete at entry
    int rc = upload(m);
    if (rc != DQ_OK) return rc;
    const bool count_all = opts->mode == DQ_MODE_COUNT_ALL;
    if (er && !count_all) { g_err = "enumeration is a COUNT_ALL solve"; return DQ_ERR_INVALID; }
    if (er && opts->engine == DQ_ENGINE_LANE) { g_err = "the lane engine counts; enumeration runs on the warp or register engine"; return DQ_ERR_UNSUPPORTED; }
    if (opts->engine == DQ_ENGINE_LANE && !count_all) {
        g_err = "the lane engines serve COUNT_ALL only"; return DQ_ERR_UNSUPPORTED;
    }
    // DQ_NO_CLASS=1 (test hook, also used for measurements): no structural class engine, every model takes the generic path
    static const bool no_class = getenv("DQ_NO_CLASS") != nullptr;
    m->last_queens_first = false;
    if (!no_class && !er && !count_all && m->cm.model_class == CLASS_QUEENS && m->cm.queens_n >= 3 && m->cm.queens_n <= kQueensMaxN &&
        opts->engine == DQ_ENGINE_AUTO && opts->part_count == 1 && opts->node_budget == 0 && opts->split_depth <= 0)
        return solve_queens_first(m, res, first_solution);
    if (!no_class && !er && count_all && m->cm.model_class == CLASS_QUEENS && m->cm.queens_n >= 3 && m->cm.queens_n <= kQueensMaxN && opts->engine != DQ_ENGINE_WARP && opts->engine != DQ_ENGINE_REG)
        return solve_queens_lane(m, opts, res, first_solution);
    if (m->cm.wide()) {
        if (opts->engine == DQ_ENGINE_REG || opts->engine == DQ_ENGINE_LANE) { g_err = "domains of more than 32 values run on the generic warp engine only"; return DQ_ERR_UNSUPPORTED; }
        return solve_tree_generic<W64>(m, opts, res, first_solution, er, count_all);
    }
    return solve_tree_generic<uint32_t>(m, opts, res, first_solution, er, count_all);
}

extern "C" {

int dq_solve_tree(dq_model* m, const dq_tree_opts* opts, dq_tree_result* res, int32_t* first_solution) {
    return solve_tree_impl(m, opts, res, first_solution, nullptr);
}

// All solutions in the reference's DFS order: what a counting Constraint that snapshots inst_vars on every hit sees
// (SURVEY.md §8c).  DQ_ERR_NOMEM when there are more than `cap` (res->n_solutions then holds the number).
int dq_enumerate_solutions(dq_model* m, const dq_tree_opts* opts, dq_tree_result* res, int32_t* solutions, uint64_t cap,
                           uint64_t* n_written) {
    if (!solutions && cap) { g_err = "null solution buffer"; return DQ_ERR_INVALID; }
    if (n_written) *n_written = 0;
    if (!opts) { g_err = "null argument"; return DQ_ERR_INVALID; }
    dq_tree_opts o = *opts;
    o.mode = DQ_MODE_COUNT_ALL;
    EnumRequest er{solutions, cap, 0};
    const int rc = solve_tree_impl(m, &o, res, nullptr, &er);
    if (n_written) *n_written = er.written;
    return rc;
}

// Nodes the reference's sequential search visits up to and including the solution in prefix `key`,
// restricted to what THIS partition owns (rank 0 also owns the levels above the split).  With
// key == UINT64_MAX: everything this partition explored.  Summed over partitions for the global
// minimum key it equals Assignment::stats.assigned_vars of the reference (dequan.h:421).
int dq_tree_nodes_upto(dq_model* m, uint64_t key, uint64_t* nodes) {
    if (!m || !nodes) { g_err = "null argument"; return DQ_ERR_INVALID; }
    *nodes = 0;
    if (!m->ctx) { g_err = "no solve to account for"; return DQ_ERR_INVALID; }
    DeviceCtx* ctx = m->ctx;
    if (m->last_queens_first) { *nodes = m->last_queens_first_nodes; return DQ_OK; }     // (one partition: the whole count is its share)
    const int depth = m->last_depth;
    const unsigned long long n_prefix = m->last_n_prefix;
    unsigned long long total = 0;
    const bool wide = m->last_wide;
    auto read_dmask = [&](const LevelArrays& L, size_t i, unsigned long long* out) -> cudaError_t {
        if (wide) return cudaMemcpy(out, L.dmask64.p + i, 8, cudaMemcpyDeviceToHost);
        uint32_t w = 0;
        const cudaError_t e = cudaMemcpy(&w, L.dmask.p + i, 4, cudaMemcpyDeviceToHost);
        *out = w;
        return e;
    };
    // (a) subtrees with index <= key owned by this partition (the key subtree holds its partial count)
    if (n_prefix) {
        const unsigned long long lim = key == KEY_NONE ? n_prefix : std::min<unsigned long long>(key + 1, n_prefix);
        std::vector<unsigned long long> sub(lim);
        if (lim) DQ_CUDA(cudaMemcpy(sub.data(), m->d_sub_nodes.p, lim * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        for (unsigned long long i = m->last_part_rank; i < lim; i += m->last_part_count) total += sub[i];
    }
    // (b) levels above the split, in DFS order up to the node that creates prefix `key`
    if (m->last_part_rank == 0) {
        if (key == KEY_NONE || n_prefix == 0) {
            for (int l = 0; l < depth; l++) {
                const LevelArrays& L = m->levels[l];
                if (L.n == 0) continue;
                unsigned long long off = 0, dm = 0;
                DQ_CUDA(cudaMemcpy(&off, L.node_off.p + (L.n - 1), sizeof off, cudaMemcpyDeviceToHost));
                DQ_CUDA(read_dmask(L, (size_t)L.n - 1, &dm));
                total += off + __builtin_popcountll(dm);
            }
        } else if (depth > 0) {
            // the parent chain of prefix `key`, walked on the device (k_nodes_upto): one launch, one read-back
            std::vector<LevelPtrs> lp(depth + 1);
            for (int l = 0; l <= depth; l++) {
                const LevelArrays& L = m->levels[l];
                lp[l].parent_of = L.parent_of.p;
                lp[l].node_off = L.node_off.p;
                lp[l].dmask = wide ? (const void*)L.dmask64.p : (const void*)L.dmask.p;
            }
            DQ_CUDA(m->d_lvl_ptrs.reserve((size_t)(depth + 1) * sizeof(LevelPtrs) + 8));
            DQ_CUDA(cudaMemcpyAsync(m->d_lvl_ptrs.p + 8, lp.data(), lp.size() * sizeof(LevelPtrs), cudaMemcpyHostToDevice, ctx->stream));
            k_nodes_upto<<<1, 32, 0, ctx->stream>>>(reinterpret_cast<const LevelPtrs*>(m->d_lvl_ptrs.p + 8), depth, key,
                                                  m->levels[depth].prefixes.p + key * (size_t)depth, wide ? 1 : 0,
                                                  reinterpret_cast<unsigned long long*>(m->d_lvl_ptrs.p));
            unsigned long long above = 0;
            DQ_CUDA(cudaMemcpyAsync(&above, m->d_lvl_ptrs.p, sizeof above, cudaMemcpyDeviceToHost, ctx->stream));
            DQ_CUDA(cudaStreamSynchronize(ctx->stream));
            total += above;
        }
    }
    *nodes = total;
    return DQ_OK;
}

}  // extern "C"

// ---- single-process multi-GPU tree solve (SURVEY.md par. 8e) ----
// One worker thread per device (streams, events and the block cache of this library are per thread and device), each
// with its own clone of the compiled model; partition i of the prefix-split tree goes to worker i.  What comes back
// per device is three 64-bit words and one value per variable; the tail — solution-count and node-count sums, lowest
// first-solution key with its solution attached — is reduced on the calling thread.
struct MultiWorker {
    int dev = 0;
    dq_model* clone = nullptr;
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    int job = 0;                      // 0 idle, 1 solve, 2 nodes_upto, 3 quit
    bool done = false;
    dq_tree_opts opts{};
    dq_tree_result res{};
    std::vector<int32_t> first;
    uint64_t key = 0, upto = 0;
    int rc = DQ_OK;
    std::string err;
    void loop() {
        if (cudaSetDevice(dev) != cudaSuccess) { (void)cudaGetLastError(); }
        for (;;) {
            int j;
            { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return job != 0; }); j = job; }
            if (j == 3) { dq_free(clone); clone = nullptr; g_cache.trim(); return; }
            if (j == 1) rc = solve_tree_impl(clone, &opts, &res, first.data(), nullptr);
            else rc = dq_tree_nodes_upto(clone, key, &upto);
            err = g_err;
            { std::lock_guard<std::mutex> lk(mu); job = 0; done = true; }
            cv.notify_all();
        }
    }
    void post(int j) { { std::lock_guard<std::mutex> lk(mu); job = j; done = false; } cv.notify_all(); }
    void wait() { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return done; }); }
};
struct MultiCtx {
    std::vector<int> devices;
    std::vector<std::unique_ptr<MultiWorker>> w;
};
static void multi_destroy(MultiCtx* mc) {
    for (auto& w : mc->w) { w->post(3); if (w->th.joinable()) w->th.join(); }
    delete mc;
}

extern "C" {

int dq_solve_tree_multi(dq_model* m, const dq_tree_opts* opts, int32_t n_devices, const int32_t* devices, dq_tree_result* res,
                        int32_t* first_solution) {
    if (!m || !opts || !res) { g_err = "null argument"; return DQ_ERR_INVALID; }
    if (n_devices < 1 || n_devices > 64) { g_err = "bad device count"; return DQ_ERR_INVALID; }
    if (opts->part_count > 1 || opts->part_rank != 0) { g_err = "dq_solve_tree_multi partitions the tree itself: part_rank / part_count must be 0 / 1"; return DQ_ERR_INVALID; }
    int have = 0;
    DQ_CUDA(cudaGetDeviceCount(&have));
    std::vector<int> devs(n_devices);
    for (int i = 0; i < n_devices; i++) {
        devs[i] = devices ? devices[i] : i;
        if (devs[i] < 0 || devs[i] >= have) { g_err = "no CUDA device " + std::to_string(devs[i]); return DQ_ERR_INVALID; }
    }
    const int nv = m->cm.nv;
    if (!m->multi || m->multi->devices != devs) {
        if (m->multi) multi_destroy(m->multi);
        m->multi = new MultiCtx();
        m->multi->devices = devs;
        for (int i = 0; i < n_devices; i++) {
            std::unique_ptr<MultiWorker> w(new MultiWorker());
            w->dev = devs[i];
            w->clone = new dq_model();
            w->clone->cm = m->cm;
            w->first.assign(std::max(nv, 1), 0);
            MultiWorker* raw = w.get();
            w->th = std::thread([raw] { raw->loop(); });
            m->multi->w.push_back(std::move(w));
        }
    }
    MultiCtx* mc = m->multi;
    for (int i = 0; i < n_devices; i++) {
        MultiWorker& w = *mc->w[i];
        w.opts = *opts;
        w.opts.part_rank = i;
        w.opts.part_count = n_devices;
        w.post(1);
    }
    for (auto& w : mc->w) w->wait();
    for (auto& w : mc->w) if (w->rc != DQ_OK) { g_err = "device " + std::to_string(w->dev) + ": " + w->err; return w->rc; }
    // the tail: sums, and the solution of the lowest DFS key (keys of different partitions never tie)
    const bool count_all = opts->mode == DQ_MODE_COUNT_ALL;
    int owner = 0;
    for (int i = 1; i < n_devices; i++) if (mc->w[i]->res.first_key < mc->w[owner]->res.first_key) owner = i;
    const uint64_t key = mc->w[owner]->res.first_key;
    *res = mc->w[0]->res;
    res->first_key = key;
    res->n_solutions = 0; res->n_nodes = 0; res->kernel_launches = 0; res->frontier_nodes = 0;
    for (auto& w : mc->w) {
        res->kernel_ms = std::max(res->kernel_ms, w->res.kernel_ms);
        res->search_kernel_ms = std::max(res->search_kernel_ms, w->res.search_kernel_ms);
        res->kernel_launches += w->res.kernel_launches;
        res->frontier_nodes += w->res.frontier_nodes;
        if (count_all) { res->n_solutions += w->res.n_solutions; res->n_nodes += w->res.n_nodes; }
    }
    if (!count_all) {
        // nodes of the reference's sequential search up to the first solution: every partition's share below the GLOBAL key
        for (auto& w : mc->w) { w->key = key; w->post(2); }
        for (auto& w : mc->w) w->wait();
        for (auto& w : mc->w) {
            if (w->rc != DQ_OK) { g_err = "device " + std::to_string(w->dev) + ": " + w->err; return w->rc; }
            res->n_nodes += w->upto;
        }
        res->n_solutions = key != KEY_NONE ? 1 : 0;
        res->nodes_before_first = res->n_nodes;
    }
    res->outcome = res->n_solutions ? DQ_SAT : DQ_UNSAT;
    if (first_solution)
        for (int v = 0; v < nv; v++) first_solution[v] = key != KEY_NONE ? mc->w[owner]->first[v] : -2147483647;
    return DQ_OK;
}

}  // extern "C" (templates follow)

// ---- many independent models in one call (dq_solve_models) ----
// The models' generic tables are packed into one host image behind the slot records and the launch cursors, and go to
// the device in one copy.  Launches are grouped by domain word and by state size class (warp_state_bytes rounded up to a
// power of two), so that one large model does not cut the occupancy of many small ones.  Each warp takes whole models
// from its launch's cursor and searches each under kModelWarpNodes; a model past that budget is marked split and solved
// afterwards by solve_tree_impl, so every answer is what dq_solve_tree gives for that handle.
struct ModelsGroup {
    bool wide, has_f, has_table;
    size_t warp_bytes;             // the largest state of the group
    int wpc;                       // warps per CTA
    long long s0, s1;              // its slots
};

template <typename W>
static int launch_models(const ModelsGroup& g, const ModelsArgs& A, DeviceCtx* ctx) {
    const size_t smem = g.warp_bytes * g.wpc;
    int occ = 0;
    int rc = with_features(g.has_f, g.has_table, [&](auto hf, auto ht) { return max_ctas_per_sm(k_models_dfs<hf, ht, W>, g.wpc * 32, smem, &occ); });
    if (rc != DQ_OK) return rc;
    if (occ < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    const long long ctas = std::max<long long>(1, std::min<long long>((A.n + g.wpc - 1) / g.wpc, (long long)occ * ctx->sm_count));
    with_features(g.has_f, g.has_table, [&](auto hf, auto ht) { k_models_dfs<hf, ht, W><<<(int)ctas, g.wpc * 32, smem, ctx->stream>>>(A); });
    DQ_CUDA(cudaGetLastError());
    return DQ_OK;
}

extern "C" {

int dq_solve_models(dq_model* const* models, int64_t n, const dq_tree_opts* opts, int32_t* outcome, uint64_t* n_solutions,
                    uint64_t* n_nodes, int32_t* solutions, int64_t* n_split, dq_batch_stats* stats) {
    if (stats) memset(stats, 0, sizeof *stats);
    if (n_split) *n_split = 0;
    if (n < 0 || !opts) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    if (opts->mode != DQ_MODE_FIRST && opts->mode != DQ_MODE_COUNT_ALL) { g_err = "bad mode"; return DQ_ERR_INVALID; }
    if (opts->part_count < 1 || opts->part_rank < 0 || opts->part_rank >= opts->part_count) { g_err = "bad partition"; return DQ_ERR_INVALID; }
    if (opts->part_count > 1) { g_err = "dq_solve_models solves whole trees: one partition"; return DQ_ERR_UNSUPPORTED; }
    if (opts->split_depth > 0) { g_err = "dq_solve_models chooses the split itself: split_depth must be <= 0"; return DQ_ERR_UNSUPPORTED; }
    if (opts->node_budget) { g_err = "node_budget is a batch option; single-tree solves have none"; return DQ_ERR_UNSUPPORTED; }
    if (opts->engine != DQ_ENGINE_AUTO && opts->engine != DQ_ENGINE_WARP) { g_err = "dq_solve_models runs the generic warp engine: engine AUTO or WARP"; return DQ_ERR_UNSUPPORTED; }
    if (n == 0) return DQ_OK;
    if (!models || !outcome || !n_solutions || !n_nodes) { g_err = "null buffer"; return DQ_ERR_INVALID; }
    for (int64_t i = 0; i < n; i++)
        if (!models[i]) { g_err = "null model at index " + std::to_string(i); return DQ_ERR_INVALID; }
    int dev = 0;
    DQ_CUDA(cudaGetDevice(&dev));
    for (int64_t i = 0; i < n; i++) {
        const int rc = check_bound(models[i], dev);
        if (rc != DQ_OK) return rc;
    }
    DeviceCtx* ctx = nullptr;
    DQ_CUDA(device_ctx(&ctx));
    const bool count_all = opts->mode == DQ_MODE_COUNT_ALL;
    const int UNASSIGNED = -2147483647;
    std::vector<int64_t> sol_off(n + 1, 0);                // each model's first value in `solutions`
    for (int64_t i = 0; i < n; i++) sol_off[i + 1] = sol_off[i] + models[i]->cm.nv;

    // slots in launch order: by domain word, then by state size class
    std::vector<int64_t> idx;
    std::vector<size_t> wbytes(n, 0);
    for (int64_t i = 0; i < n; i++) {
        const CompiledModel& c = models[i]->cm;
        if (c.nv == 0) continue;
        wbytes[i] = warp_state_bytes(c.nv, c.trail_bound, c.wide() ? 8 : 4);
        idx.push_back(i);
    }
    auto size_class = [&](int64_t i) { size_t s = 16; while (s < wbytes[i]) s <<= 1; return s; };
    std::stable_sort(idx.begin(), idx.end(), [&](int64_t a, int64_t b) {
        const bool wa = models[a]->cm.wide(), wb = models[b]->cm.wide();
        return wa != wb ? wb : size_class(a) < size_class(b);
    });
    const long long n_slots = (long long)idx.size();
    std::vector<ModelsGroup> groups;
    for (long long k = 0; k < n_slots; k++) {
        const CompiledModel& c = models[idx[k]]->cm;
        if (groups.empty() || groups.back().wide != c.wide() || size_class(idx[groups.back().s0]) != size_class(idx[k]))
            groups.push_back(ModelsGroup{c.wide(), false, false, 0, 0, k, k});
        ModelsGroup& g = groups.back();
        g.has_f |= c.has_f; g.has_table |= c.has_table;
        g.warp_bytes = std::max(g.warp_bytes, wbytes[idx[k]]);
        g.s1 = k + 1;
    }
    for (ModelsGroup& g : groups) {
        g.wpc = (int)std::min<size_t>(kWarpsPerCta, (200 * 1024) / g.warp_bytes);
        if (g.wpc < 1) { g_err = "model state exceeds shared memory"; return DQ_ERR_UNSUPPORTED; }
    }

    // host image: launch cursors, slot records, then every model's tables
    const size_t o_slots = ((groups.size() * 8 + 15) & ~(size_t)15);
    std::vector<uint8_t> blob(o_slots + (size_t)n_slots * sizeof(ModelSlot), 0);
    std::vector<ModelSlot> slots(n_slots);
    unsigned long long sol_bytes = 0;
    for (long long k = 0; k < n_slots; k++) {
        const CompiledModel& c = models[idx[k]]->cm;
        const TreeTableOffsets t = put_tree_tables(c, blob, 16);
        ModelSlot& s = slots[k];
        s.base = t.ent_off;
        s.o_ent = (uint32_t)(t.ent - t.ent_off); s.o_ent_moff = (uint32_t)(t.ent_moff - t.ent_off);
        s.o_masks = (uint32_t)(t.masks - t.ent_off); s.o_dom0 = (uint32_t)(t.dom0 - t.ent_off);
        s.o_order = (uint32_t)(t.order - t.ent_off); s.o_pos = (uint32_t)(t.pos - t.ent_off);
        s.nv = c.nv; s.trail = c.trail_bound;
        s.sol = sol_bytes;
        sol_bytes += (unsigned long long)c.nv;
    }
    if (n_slots) memcpy(blob.data() + o_slots, slots.data(), slots.size() * sizeof(ModelSlot));

    // results: one record per slot, then the value indices of every slot's first solution
    const size_t o_sol = (size_t)n_slots * sizeof(ModelOut);
    const size_t read_bytes = o_sol + (solutions ? (size_t)sol_bytes : 0);
    std::vector<uint8_t> h_out(read_bytes);
    DevBuf<uint8_t> d_in, d_out;
    StreamDrain drain{ctx->stream};
    float ms = 0;
    unsigned long long launches = 0;
    if (n_slots) {
        DQ_CUDA(d_in.reserve(blob.size()));
        DQ_CUDA(d_out.reserve(o_sol + (size_t)sol_bytes));
        DQ_CUDA(cudaMemcpyAsync(d_in.p, blob.data(), blob.size(), cudaMemcpyHostToDevice, ctx->stream));
        DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
        for (size_t gi = 0; gi < groups.size(); gi++) {
            const ModelsGroup& g = groups[gi];
            ModelsArgs A;
            A.slots = reinterpret_cast<const ModelSlot*>(d_in.p + o_slots) + g.s0;
            A.n = g.s1 - g.s0;
            A.tables = d_in.p;
            A.warp_bytes = g.warp_bytes;
            A.count_all = count_all ? 1 : 0;
            A.cursor = reinterpret_cast<unsigned long long*>(d_in.p) + gi;
            A.out = reinterpret_cast<ModelOut*>(d_out.p) + g.s0;
            A.sol = d_out.p + o_sol;
            const int rc = g.wide ? launch_models<W64>(g, A, ctx) : launch_models<uint32_t>(g, A, ctx);
            if (rc != DQ_OK) return rc;
            launches++;
        }
        DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
        DQ_CUDA(cudaMemcpyAsync(h_out.data(), d_out.p, read_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CUDA(cudaStreamSynchronize(ctx->stream));
        DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    }

    unsigned long long n_sat = 0, total_nodes = 0;
    int64_t splits = 0;
    for (int64_t i = 0; i < n; i++)
        if (models[i]->cm.nv == 0) { outcome[i] = DQ_SAT; n_solutions[i] = 1; n_nodes[i] = 0; }      // IsComplete at entry
    for (long long k = 0; k < n_slots; k++) {
        const int64_t i = idx[k];
        ModelOut o;
        memcpy(&o, h_out.data() + (size_t)k * sizeof(ModelOut), sizeof o);
        const CompiledModel& c = models[i]->cm;
        if (o.outcome == DQ_BUDGET) {                       // past the warp's budget: the split search, as dq_solve_tree runs it
            dq_tree_result r;
            const int rc = solve_tree_impl(models[i], opts, &r, solutions ? solutions + sol_off[i] : nullptr, nullptr);
            if (rc != DQ_OK) return rc;
            outcome[i] = r.outcome; n_solutions[i] = r.n_solutions; n_nodes[i] = r.n_nodes;
            launches += r.kernel_launches;
            splits++;
            continue;
        }
        outcome[i] = o.outcome; n_solutions[i] = o.sols; n_nodes[i] = o.nodes;
        if (solutions) {
            const uint8_t* v = h_out.data() + o_sol + slots[k].sol;
            for (int x = 0; x < c.nv; x++) solutions[sol_off[i] + x] = o.sols ? c.values[x][v[x]] : UNASSIGNED;
        }
    }
    for (int64_t i = 0; i < n; i++) { n_sat += outcome[i] == DQ_SAT; total_nodes += n_nodes[i]; }
    if (n_split) *n_split = splits;
    if (stats) {
        stats->n_sat = n_sat; stats->n_unsat = (uint64_t)n - n_sat; stats->n_budget = 0; stats->total_nodes = total_nodes;
        stats->kernel_ms = ms; stats->kernel_launches = launches;
        stats->h2d_bytes = n_slots ? blob.size() : 0; stats->d2h_bytes = n_slots ? read_bytes : 0;
    }
    return DQ_OK;
}

static int run_batch_sudoku(dq_model* m, const uint8_t* cells_dev, int64_t n, int32_t stride, const dq_batch_opts* opts,
                            uint8_t* sol_dev, unsigned long long* nodes_dev, uint8_t* status_dev, dq_batch_stats* st);

// nsol_dev non-null: the counting batch (k_count_batch_cells, engine WARP) with solution limit `limit`.
static int run_batch_cells(dq_model* m, const uint8_t* cells_dev, int64_t n, int32_t stride, const dq_batch_opts* opts,
                           uint8_t* sol_dev, unsigned long long* nodes_dev, uint8_t* status_dev, dq_batch_stats* st,
                           const int* idx_list = nullptr, bool timed = true, unsigned long long* nsol_dev = nullptr,
                           unsigned long long limit = 0) {
    if (m->cm.wide()) { g_err = "batches take template domains of at most 32 values"; return DQ_ERR_UNSUPPORTED; }
    if (!idx_list && m->cm.model_class == CLASS_SUDOKU9 && !(opts && opts->engine == DQ_ENGINE_WARP))
        return run_batch_sudoku(m, cells_dev, n, stride, opts, sol_dev, nodes_dev, status_dev, st);
    if (opts && opts->engine == DQ_ENGINE_LANE && m->cm.model_class != CLASS_SUDOKU9) {
        g_err = "the lane batch engine serves the 9x9 Sudoku class only"; return DQ_ERR_UNSUPPORTED;
    }
    const int nv = m->cm.nv;
    DeviceCtx* ctx = m->ctx;
    const TreeModelDev M = dev_model(m);
    const size_t smem = warp_state_bytes(nv, M.trail) * kWarpsPerCta;
    if (smem > 200 * 1024) { g_err = "model state exceeds shared memory"; return DQ_ERR_UNSUPPORTED; }
    const auto kernel = with_features(m->cm, [&](auto hf, auto ht) { return nsol_dev ? k_count_batch_cells<hf, ht> : k_batch_cells<hf, ht>; });
    int occ = 0;
    int rc = max_ctas_per_sm(kernel, kWarpsPerCta * 32, smem, &occ);
    if (rc != DQ_OK) return rc;
    if (occ < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    unsigned long long* ctrl = m->d_ctrl.p;
    DQ_CUDA(cudaMemsetAsync(ctrl, 0, 8 * sizeof(unsigned long long), ctx->stream));
    BatchCellsArgs A;
    A.idx_list = idx_list;
    A.cells = cells_dev; A.n = n; A.stride = stride; A.cell_lut = m->t_cell_lut; A.values = m->t_values;
    A.sizes = m->t_sizes; A.n_sizes = m->n_sizes; A.caller_order = m->cm.caller_order ? 1 : 0;
    A.budget = opts ? opts->node_budget : 0;
    A.cursor = ctrl; A.solution = sol_dev; A.nodes = nodes_dev; A.status = status_dev; A.totals = ctrl + 1;
    A.limit = limit; A.n_solutions = nsol_dev;
    long long ctas = std::min<long long>((n + kWarpsPerCta - 1) / kWarpsPerCta, (long long)occ * ctx->sm_count);
    if (ctas < 1) ctas = 1;
    if (timed) DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    kernel<<<(int)ctas, kWarpsPerCta * 32, smem, ctx->stream>>>(M, A);
    DQ_CUDA(cudaGetLastError());
    if (!timed) return DQ_OK;
    DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    unsigned long long h[8];
    DQ_CUDA(cudaMemcpyAsync(h, ctrl, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    if (st) {
        float ms = 0;
        DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        st->n_sat = h[1]; st->n_unsat = h[2]; st->n_budget = h[3]; st->total_nodes = h[4];
        st->kernel_ms = ms; st->kernel_launches = 1;
    }
    return DQ_OK;
}

// Batch of 9x9 Sudoku (dq_lane_sudoku.cuh): digest -> first (lane per instance, bounded) -> strong (warp per hard
// instance: the solution) -> walk + count (the reference's node total, exhaustive subtree tasks) -> finish, queued back
// to back on one stream; instances the digest cannot take (clashing givens, foreign bytes) go through the generic warp
// engine afterwards.
static int run_batch_sudoku(dq_model* m, const uint8_t* cells_dev, int64_t n, int32_t stride, const dq_batch_opts* opts,
                            uint8_t* sol_dev, unsigned long long* nodes_dev, uint8_t* status_dev, dq_batch_stats* st) {
    DeviceCtx* ctx = m->ctx;
    int rc = DQ_OK;
    // the number of pieces handed over at the tail does not shrink with the batch: generous floors (64 MB + 192 MB)
    const unsigned long long task_cap = std::max<unsigned long long>(1u << 24, std::min<unsigned long long>(8ull * n, 1ull << 26));   // (16 B each; a task per 512 counted nodes and more)
    // (one parked snapshot per hard instance stays for the whole call, the rest of the ring recycles; slots are 24-bit in the hard list)
    const unsigned long long snap_cap = std::min<unsigned long long>(std::max<unsigned long long>(1u << 20, (unsigned long long)n + (1u << 20)), 1ull << 24);
    const bool fresh_pool = m->s_tasks.cap < task_cap;
    DQ_CUDA(m->s_digest.reserve(n)); DQ_CUDA(m->s_hard.reserve(2 * (size_t)n)); DQ_CUDA(m->s_ctrl.reserve(16));
    DQ_CUDA(m->s_tasks.reserve(task_cap)); DQ_CUDA(m->s_snaps.reserve(snap_cap * kSnapWords)); DQ_CUDA(m->s_snap_state.reserve(snap_cap));
    unsigned long long* ctrl = m->s_ctrl.p;       // SkCtrl words
    DQ_CUDA(cudaMemsetAsync(ctrl, 0, 16 * sizeof(unsigned long long), ctx->stream));
    DQ_CUDA(cudaMemsetAsync(m->s_snap_state.p, 0, snap_cap * sizeof(uint32_t), ctx->stream));
    // task records double as "published" flags: the part the previous call used must read zero again
    const unsigned long long dirty = fresh_pool ? m->s_tasks.cap : std::min<unsigned long long>(m->s_tasks_used, m->s_tasks.cap);
    if (dirty) DQ_CUDA(cudaMemsetAsync(m->s_tasks.p, 0, dirty * sizeof(SudokuTask), ctx->stream));
    SudokuArgs A;
    A.digest = m->s_digest.p; A.n = n; A.stride = stride; A.cells = cells_dev; A.solution = sol_dev; A.nodes = nodes_dev;
    A.status = status_dev; A.hard = m->s_hard.p; A.tasks = m->s_tasks.p; A.task_cap = task_cap;
    A.snaps = m->s_snaps.p; A.snap_cap = snap_cap; A.snap_state = m->s_snap_state.p; A.ctrl = ctrl; A.user_budget = opts ? opts->node_budget : 0;
    A.force_donate = opts && opts->task_nodes > 0 ? (unsigned)opts->task_nodes : 0u;
    A.first_budget = n >= 400000 ? 3072u : 1024u;   // measured at 1 M: 1024 -> 32.7 ms, 2048 -> 30.3, 3072 -> 29.5; 125 k shards: flat 512-1024 (7.2 ms), 1536 -> 7.6
    if (A.force_donate) A.first_budget = std::min(A.first_budget, 4u * A.force_donate);       // tests: push work through the task path
    const long long sms = ctx->sm_count;
    DQ_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    {
        int occ_d = 0;
        rc = max_ctas_per_sm(k_sudoku_digest, kDigestTile, kDigestSmem, &occ_d);
        if (rc != DQ_OK) return rc;
        const long long tiles = (n + kDigestTile - 1) / kDigestTile;
        k_sudoku_digest<<<(unsigned)std::max<long long>(1, std::min<long long>(tiles, (long long)std::max(occ_d, 1) * sms)), kDigestTile, kDigestSmem, ctx->stream>>>(
            cells_dev, n, stride, m->s_digest.p, ctrl + SKC_MAX_BLANK);
    }
    // The lanes' stacks are sized for the instance with the most blanks (one 8-byte read-back after the digest, ~20 us):
    // with 30 givens that is 51 levels instead of 81, 354 bytes of shared memory per lane instead of 414, and a fifth CTA
    // (20 warps instead of 16) on every SM.
    unsigned long long* h_blank = &ctx->pin->sudoku_max_blank;
    DQ_CUDA(cudaMemcpyAsync(h_blank, ctrl + SKC_MAX_BLANK, sizeof *h_blank, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    const int levels = (int)std::min<unsigned long long>(std::max<unsigned long long>(*h_blank, 1), 81);
    const size_t smem = offsetof(SudokuSmem, stk) + (size_t)levels * kSudokuBlock * sizeof(uint16_t);
    const size_t smem_strong = sudoku_strong_smem(levels);       // (30 givens: 36 KB per CTA, 24 warps per SM instead of 16)
    A.stack_levels = levels;
    int occ_first = 0, occ_count = 0, occ_walk = 0, occ_strong = 0;
    rc = max_ctas_per_sm(k_sudoku_first, kSudokuBlock, smem, &occ_first);
    if (rc == DQ_OK) rc = max_ctas_per_sm(k_sudoku_count, kSudokuBlock, smem, &occ_count);
    if (rc == DQ_OK) rc = max_ctas_per_sm(k_sudoku_walk, kSudokuBlock, smem, &occ_walk);
    if (rc == DQ_OK) rc = max_ctas_per_sm(k_sudoku_strong, 128, smem_strong, &occ_strong);
    if (rc != DQ_OK) return rc;
    if (occ_first < 1 || occ_count < 1 || occ_walk < 1 || occ_strong < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    const long long ctas_first = std::max<long long>(1, std::min<long long>(occ_first * sms, (long long)((n + kSudokuBlock - 1) / kSudokuBlock)));
    k_sudoku_first<<<(unsigned)ctas_first, kSudokuBlock, smem, ctx->stream>>>(A);
    // the hard list's length stays on the device: the next three kernels are sized for the machine and find it in ctrl
    k_sudoku_strong<<<(unsigned)(occ_strong * sms), 128, smem_strong, ctx->stream>>>(A);
    // Host-buffer call without a node budget: every solution is final here (what follows only counts nodes), so the
    // 81 bytes per instance go home on the side stream while the counting stage runs.
    if (m->early_sol_host && !A.user_budget) {
        DQ_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
        DQ_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
        DQ_CUDA(cudaMemcpyAsync(m->early_sol_host, sol_dev, (size_t)n * stride, cudaMemcpyDeviceToHost, ctx->stream2));
        DQ_CUDA(cudaEventRecord(ctx->ev_join, ctx->stream2));
        m->early_sol_done = true;
    }
    k_sudoku_walk<<<(unsigned)std::min<long long>(occ_walk * sms, (long long)((n + kSudokuBlock - 1) / kSudokuBlock)), kSudokuBlock, smem, ctx->stream>>>(A);
    k_sudoku_count<<<(unsigned)(occ_count * sms), kSudokuBlock, smem, ctx->stream>>>(A);
    k_sudoku_finish<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(A, ctrl + SKC_TOTALS);
    DQ_CUDA(m->s_deferred.reserve(n));
    k_sudoku_collect_deferred<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(status_dev, n, m->s_deferred.p, ctrl + 10);
    unsigned long long launches = 7;
    DQ_CUDA(cudaGetLastError());
    unsigned long long hc[16];
    DQ_CUDA(cudaMemcpyAsync(hc, ctrl, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    m->s_tasks_used = std::min(hc[SKC_RESERVE], task_cap);
    if (hc[SKC_ERROR] & 2) { g_err = "sudoku task pool overflow"; return DQ_ERR_NOMEM; }
    if (hc[SKC_ERROR] || hc[SKC_OUTSTANDING]) {
        g_err = "internal: sudoku counting pipeline inconsistent (error bits " + std::to_string(hc[SKC_ERROR]) + ")";
        return DQ_ERR_INTERNAL;
    }
    const unsigned long long n_def = hc[10];
    unsigned long long hw[8] = {0};
    if (m->early_sol_done) DQ_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    if (n_def) {
        m->early_sol_done = false;                 // (the generic engine is about to write the deferred instances' solutions)
        dq_batch_opts o2 = opts ? *opts : dq_batch_opts{0, 0, 0};
        o2.engine = DQ_ENGINE_WARP;
        rc = run_batch_cells(m, cells_dev, (int64_t)n_def, stride, &o2, sol_dev, nodes_dev, status_dev, nullptr, m->s_deferred.p, false);
        if (rc != DQ_OK) return rc;
        launches++;
    }
    DQ_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    if (n_def) DQ_CUDA(cudaMemcpyAsync(hw, m->d_ctrl.p, sizeof hw, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    if (st) {
        float ms = 0;
        DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        const unsigned long long* ht = hc + SKC_TOTALS;
        st->n_sat = ht[0] + hw[1]; st->n_unsat = ht[1] + hw[2]; st->n_budget = ht[2] + hw[3]; st->total_nodes = ht[3] + hw[4];
        st->kernel_ms = ms; st->kernel_launches = launches;
    }
    return DQ_OK;
}

int dq_solve_batch_cells_dev(dq_model* m, const uint8_t* cells_dev, int64_t n, int32_t stride, const dq_batch_opts* opts,
                             uint8_t* solution_dev, uint64_t* nodes_dev, uint8_t* status_dev, dq_batch_stats* stats) {
    if (!m || n < 0 || stride < m->cm.nv) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return DQ_OK;
    int rc = upload(m);
    if (rc != DQ_OK) return rc;
    return run_batch_cells(m, cells_dev, n, stride, opts, solution_dev, (unsigned long long*)nodes_dev, status_dev, stats);
}

}  // extern "C"

// dq_solve_batch_cells and dq_count_batch_cells (n_solutions non-null) once their arguments are checked: the host
// buffers around run_batch_cells.
static int batch_cells_host(dq_model* m, const uint8_t* cells, int64_t n, int32_t stride, const dq_batch_opts* opts,
                            uint8_t* solution, uint64_t* nodes, uint8_t* status, dq_batch_stats* stats,
                            uint64_t* n_solutions = nullptr, unsigned long long limit = 0) {
    int rc = upload(m);
    if (rc != DQ_OK) return rc;
    DeviceCtx* ctx = m->ctx;
    const size_t bytes = (size_t)n * stride;
    DQ_CUDA(m->b_cells.reserve(bytes)); DQ_CUDA(m->b_solution.reserve(bytes));
    DQ_CUDA(m->b_status.reserve(n)); DQ_CUDA(m->b_nodes.reserve(n));
    DQ_CUDA(cudaMemcpyAsync(m->b_cells.p, cells, bytes, cudaMemcpyHostToDevice, ctx->stream));
    // (only into page-locked memory: an "asynchronous" copy into pageable memory holds the calling thread until it is
    // done, which would park the pipeline between its stages)
    cudaPointerAttributes pa;
    const bool pinned = cudaPointerGetAttributes(&pa, solution) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    if (!pinned) cudaGetLastError();
    m->early_sol_host = pinned ? solution : nullptr; m->early_sol_done = false;
    if (n_solutions) DQ_CUDA(m->b_nsol.reserve(n));
    rc = run_batch_cells(m, m->b_cells.p, n, stride, opts, m->b_solution.p, m->b_nodes.p, m->b_status.p, stats, nullptr, true,
                         n_solutions ? m->b_nsol.p : nullptr, limit);
    m->early_sol_host = nullptr;
    if (rc != DQ_OK) { cudaStreamSynchronize(ctx->stream2); return rc; }     // (nothing may still be writing the caller's buffer)
    if (!m->early_sol_done) DQ_CUDA(cudaMemcpyAsync(solution, m->b_solution.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaMemcpyAsync(nodes, m->b_nodes.p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaMemcpyAsync(status, m->b_status.p, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_solutions) DQ_CUDA(cudaMemcpyAsync(n_solutions, m->b_nsol.p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CUDA(cudaStreamSynchronize(ctx->stream));
    if (stats) { stats->h2d_bytes = bytes; stats->d2h_bytes = bytes + (size_t)n * (n_solutions ? 17 : 9); }
    return DQ_OK;
}

// The counting batches run on the generic warp engine only: engine AUTO or WARP.
static int check_count_opts(const dq_count_opts* opts) {
    const int engine = opts ? opts->engine : DQ_ENGINE_AUTO;
    if (engine == DQ_ENGINE_LANE || engine == DQ_ENGINE_REG) {
        g_err = "batch counting runs on the generic warp engine only: engine AUTO or WARP"; return DQ_ERR_UNSUPPORTED;
    }
    if (engine != DQ_ENGINE_AUTO && engine != DQ_ENGINE_WARP) { g_err = "bad engine"; return DQ_ERR_INVALID; }
    return DQ_OK;
}

extern "C" {

int dq_solve_batch_cells(dq_model* m, const uint8_t* cells, int64_t n, int32_t stride, const dq_batch_opts* opts,
                         uint8_t* solution, uint64_t* nodes, uint8_t* status, dq_batch_stats* stats) {
    if (!m || n < 0 || stride < m->cm.nv) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return DQ_OK;
    if (!cells || !solution || !nodes || !status) { g_err = "null buffer"; return DQ_ERR_INVALID; }
    return batch_cells_host(m, cells, n, stride, opts, solution, nodes, status, stats);
}

int dq_count_batch_cells(dq_model* m, const uint8_t* cells, int64_t n, int32_t stride, const dq_count_opts* opts,
                         uint64_t* n_solutions, uint8_t* solution, uint64_t* nodes, uint8_t* status, dq_batch_stats* stats) {
    if (!m || n < 0 || stride < m->cm.nv) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    int rc = check_count_opts(opts);
    if (rc != DQ_OK) return rc;
    if (m->cm.wide()) { g_err = "batches take template domains of at most 32 values"; return DQ_ERR_UNSUPPORTED; }
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return DQ_OK;
    if (!cells || !n_solutions || !solution || !nodes || !status) { g_err = "null buffer"; return DQ_ERR_INVALID; }
    const dq_batch_opts o{opts ? opts->node_budget : 0, DQ_ENGINE_WARP, 0};
    return batch_cells_host(m, cells, n, stride, &o, solution, nodes, status, stats, n_solutions, opts ? opts->solution_limit : 0);
}

}  // extern "C"

// Batches of k-colouring instances.  Device-level runner shared by the host-buffer and the device-buffer entry points:
// engine choice, scratch, kernels, totals.  `edge_off` is the HOST copy of the offsets (sizes the adjacency records).
struct GraphBatchDev {
    const long long* off; const uint8_t* edges; long long edge_bytes;    // edge_bytes: 2 * total rounded up to 16, readable
    uint8_t* colours; unsigned long long* nodes; uint8_t* status;
    const uint8_t* host_edges;                                           // host copy of the lists, if the caller has one
    unsigned long long* n_solutions = nullptr;                           // counting batch (warp engine): solutions per instance
};

// Lane-per-instance engine (dq_group_graphs.cuh): two passes of k_graphs_adjacency (overflow statistics, records),
// then the search.  DQ_ERR_UNSUPPORTED when the per-warp state does not fit an SM's shared memory.
static int run_graphs_lane(int nv, int k, const int64_t* edge_off, const GraphBatchDev& B, int64_t n, unsigned long long budget,
                           DeviceCtx* ctx, DevBuf<uint8_t>& d_adj, unsigned long long* d_ctrl) {
    cudaStream_t s = ctx->stream;
    const int sms = ctx->sm_count;
    long long max_m = 0;
    for (int64_t i = 0; i < n; i++) max_m = std::max<long long>(max_m, edge_off[i + 1] - edge_off[i]);
    GroupGraphsArgs A;
    A.nv = nv; A.k = k; A.nvp = (nv + 16) & ~15;
    A.rw = kGraphRow; A.over_cap = 0; A.over_smem = 0;
    A.stride = graphs_record_bytes(A.nvp, A.rw, 0);
    A.edge_off = B.off; A.edges = B.edges; A.edge_bytes = B.edge_bytes; A.n = n;
    A.budget = budget; A.cursor = d_ctrl; A.colours = B.colours; A.nodes = B.nodes; A.status = B.status;
    A.totals = d_ctrl + 1;
    A.adj = nullptr;
    const int stage_cap = (int)(((2 * max_m + 15) & ~15ll) + 32);
    // worst case of the record size: every edge of the largest instance in the overflow list
    if (graphs_adj_warp_bytes(A.nvp, graphs_record_bytes(A.nvp, A.rw, (int)std::min<long long>(max_m + 256, 65535)), stage_cap) * kAdjWarpsPerCta > 200 * 1024) {
        g_err = "edge list exceeds shared memory"; return DQ_ERR_UNSUPPORTED;
    }
    int occ_a = 0;
    int rc = max_ctas_per_sm(k_graphs_adjacency<true>, kAdjWarpsPerCta * 32, graphs_adj_warp_bytes(A.nvp, A.stride, stage_cap) * kAdjWarpsPerCta, &occ_a);
    if (rc != DQ_OK) return rc;
    if (occ_a < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    DQ_CUDA(cudaMemsetAsync(B.status, 0, (size_t)n, s));
    DQ_CUDA(cudaEventRecord(ctx->ev0, s));
    // pass 1 over the edge lists: how long an overflow list do rows of 8 slots leave behind?  (one 8-byte read-back)
    long long actas = std::max<long long>(1, std::min<long long>((n + kAdjWarpsPerCta - 1) / kAdjWarpsPerCta, (long long)occ_a * sms));
    k_graphs_adjacency<true><<<(unsigned)actas, kAdjWarpsPerCta * 32, graphs_adj_warp_bytes(A.nvp, A.stride, stage_cap) * kAdjWarpsPerCta, s>>>(A, stage_cap);
    unsigned long long* h_over = &ctx->pin->graphs_over;
    DQ_CUDA(cudaMemcpyAsync(h_over, d_ctrl + 6, sizeof *h_over, cudaMemcpyDeviceToHost, s));
    DQ_CUDA(cudaStreamSynchronize(s));
    if (*h_over > 65535) { g_err = "an instance leaves more than 65535 edges outside its neighbour rows"; return DQ_ERR_UNSUPPORTED; }
    A.over_cap = (int)((*h_over + 1) & ~1ull);
    A.stride = graphs_record_bytes(A.nvp, A.rw, A.over_cap);
    const bool packed = k <= 3;      // (byte 3 of the state words is free below four colours)
    // the overflow pairs a lane keeps in shared memory: as many as cost no CTA per SM (the rest are read from the record)
    A.over_smem = 0;
    {
        const size_t per_sm = 228 * 1024, cta_tax = 1024;
        const size_t base = graphs_lane_warp_bytes(A.nv, A.nvp, 0, packed);
        if (base > 220 * 1024) { g_err = "instance state exceeds shared memory"; return DQ_ERR_UNSUPPORTED; }
        const size_t ctas_base = std::min<size_t>(per_sm / (base + cta_tax), 32);
        const size_t room = per_sm / ctas_base - cta_tax - base;                 // bytes a CTA can grow by without losing a neighbour
        A.over_smem = (int)std::min<size_t>((size_t)A.over_cap, room / 64);
    }
    const size_t lane_smem = graphs_lane_warp_bytes(A.nv, A.nvp, A.over_smem, packed);
    DQ_CUDA(d_adj.reserve((size_t)n * A.stride));
    A.adj = d_adj.p;
    // pass 2: the records
    const size_t adj_warp = graphs_adj_warp_bytes(A.nvp, A.stride, stage_cap);
    rc = max_ctas_per_sm(k_graphs_adjacency<false>, kAdjWarpsPerCta * 32, adj_warp * kAdjWarpsPerCta, &occ_a);
    if (rc != DQ_OK) return rc;
    if (occ_a < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    actas = std::max<long long>(1, std::min<long long>((n + kAdjWarpsPerCta - 1) / kAdjWarpsPerCta, (long long)occ_a * sms));
    k_graphs_adjacency<false><<<(unsigned)actas, kAdjWarpsPerCta * 32, adj_warp * kAdjWarpsPerCta, s>>>(A, stage_cap);
    DQ_CUDA(cudaEventRecord(ctx->ev2, s));
    // the search: one warp per CTA, as many CTAs per SM as their state lets in
    int occ = 0;
    rc = packed ? max_ctas_per_sm(k_graphs_lane<true>, 32, lane_smem, &occ) : max_ctas_per_sm(k_graphs_lane<false>, 32, lane_smem, &occ);
    if (rc != DQ_OK) return rc;
    if (occ < 1) { g_err = "kernel does not fit an SM"; return DQ_ERR_UNSUPPORTED; }
    const long long ctas = std::max<long long>(1, std::min<long long>((n + 31) / 32, (long long)occ * sms));
    if (packed) k_graphs_lane<true><<<(unsigned)ctas, 32, lane_smem, s>>>(A);
    else k_graphs_lane<false><<<(unsigned)ctas, 32, lane_smem, s>>>(A);
    DQ_CUDA(cudaEventRecord(ctx->ev3, s));
    return DQ_OK;
}

// B.n_solutions non-null: the counting batch (k_count_batch_graphs, engine WARP) with solution limit `limit`.
static int run_batch_graphs(int nv, int k, const int64_t* edge_off, const GraphBatchDev& B, int64_t n, const dq_batch_opts* opts,
                            dq_batch_stats* stats, unsigned long long limit = 0) {
    DeviceCtx* ctx = nullptr;
    DQ_CUDA(device_ctx(&ctx));
    cudaStream_t s = ctx->stream;
    const int sms = ctx->sm_count;
    const long long total = edge_off[n];
    const int engine = opts ? opts->engine : DQ_ENGINE_AUTO;
    if (engine == DQ_ENGINE_LANE && k > 4) { g_err = "the lane engine serves k <= 4"; return DQ_ERR_UNSUPPORTED; }
    if (engine == DQ_ENGINE_REG && k > 4) { g_err = "the register engine serves k <= 4"; return DQ_ERR_UNSUPPORTED; }
    // measured on B200 (scripts/colour_sweep.py, G(200, 4.2/199), 100 k-node budget): the lane engine needs a few
    // thousand instances to fill its 32-instance warps (1 024 instances: 41 ms against 23 ms for one warp per instance,
    // 8 192: 50 against 83 ms, 65 536: 146 against 588 ms)
    bool lane_engine = k <= 4 && (engine == DQ_ENGINE_LANE || (engine == DQ_ENGINE_AUTO && n >= 4096));
    DevBuf<uint32_t> d_ent_off, d_ent; DevBuf<uint8_t> d_adj;
    DevBuf<unsigned long long> d_ctrl;
    StreamDrain drain{s};
    DQ_CUDA(d_ctrl.reserve(8));
    DQ_CUDA(cudaMemsetAsync(d_ctrl.p, 0, 8 * sizeof(unsigned long long), s));
    unsigned long long launches = 0;
    float ms = 0, ms_search = 0;
    if (lane_engine) {
        const int rc = run_graphs_lane(nv, k, edge_off, B, n, opts ? opts->node_budget : 0, ctx, d_adj, d_ctrl.p);
        if (rc == DQ_ERR_UNSUPPORTED && engine == DQ_ENGINE_AUTO && B.host_edges) {       // (graphs too dense for the lane state: the warp engine below)
            for (long long e = 0; e < total; e++) {                   // ... which trusts the lists
                const uint8_t u = B.host_edges[2 * e], v = B.host_edges[2 * e + 1];
                if (u >= nv || v >= nv) { g_err = "edge endpoint out of range"; return DQ_ERR_INVALID; }
                if (u == v) { g_err = "edge with u == v"; return DQ_ERR_UNSUPPORTED; }
            }
            lane_engine = false;
            DQ_CUDA(cudaStreamSynchronize(s));
            DQ_CUDA(cudaMemsetAsync(d_ctrl.p, 0, 8 * sizeof(unsigned long long), s));
        } else if (rc != DQ_OK) return rc;
        launches = 3;
    }
    const bool reg_engine = !lane_engine && k <= 4 && engine != DQ_ENGINE_WARP;   // register-resident warp engine (dq_reg_graphs.cuh)
    if (!lane_engine) {
        BatchGraphsArgs A;
        A.nv = nv; A.k = k; A.edge_off = B.off; A.edges = B.edges; A.n = n;
        A.budget = opts ? opts->node_budget : 0; A.cursor = d_ctrl.p; A.colours = B.colours; A.nodes = B.nodes;
        A.status = B.status; A.totals = d_ctrl.p + 1;
        A.trail = nv * k + 32;
        A.limit = limit; A.n_solutions = B.n_solutions;
        DQ_CUDA(cudaEventRecord(ctx->ev0, s));
        if (reg_engine) {
            RegGraphsArgs R;
            R.nv = nv; R.k = k; R.edge_off = B.off; R.edges = B.edges; R.n = n; R.budget = A.budget; R.cursor = d_ctrl.p;
            R.colours = B.colours; R.nodes = B.nodes; R.status = B.status; R.totals = d_ctrl.p + 1;
            const size_t rsmem = reg_graphs_warp_bytes(nv, k) * kRegWarpsPerCta;
            int rocc = 0;
            int rc = max_ctas_per_sm(k_batch_graphs_reg, kRegWarpsPerCta * 32, rsmem, &rocc);
            if (rc != DQ_OK) return rc;
            const long long rctas = std::min<long long>((n + kRegWarpsPerCta - 1) / kRegWarpsPerCta, (long long)std::max(rocc, 1) * sms);
            DQ_CUDA(cudaEventRecord(ctx->ev2, s));
            k_batch_graphs_reg<<<(unsigned)rctas, kRegWarpsPerCta * 32, rsmem, s>>>(R);
            launches = 1;
        } else {
            const size_t smem = warp_state_bytes(nv, A.trail) * kWarpsPerCta;
            if (smem > 200 * 1024) { g_err = "instance state exceeds shared memory"; return DQ_ERR_UNSUPPORTED; }
            const auto kernel = B.n_solutions ? k_count_batch_graphs : k_batch_graphs;
            int occ = 0;
            int rc = max_ctas_per_sm(kernel, kWarpsPerCta * 32, smem, &occ);
            if (rc != DQ_OK) return rc;
            DQ_CUDA(d_ent_off.reserve((size_t)n * (nv + 1))); DQ_CUDA(d_ent.reserve(2 * (size_t)std::max<long long>(total, 1)));
            A.ent_off = d_ent_off.p; A.ent = d_ent.p;
            k_graphs_build<<<(unsigned)((n + kWarpsPerCta - 1) / kWarpsPerCta), kWarpsPerCta * 32, kWarpsPerCta * graphs_build_warp_bytes(nv), s>>>(A);
            long long ctas = std::min<long long>((n + kWarpsPerCta - 1) / kWarpsPerCta, (long long)std::max(occ, 1) * sms);
            DQ_CUDA(cudaEventRecord(ctx->ev2, s));
            kernel<<<(unsigned)ctas, kWarpsPerCta * 32, smem, s>>>(A);
            launches = 2;
        }
        DQ_CUDA(cudaEventRecord(ctx->ev3, s));
    }
    DQ_CUDA(cudaGetLastError());
    DQ_CUDA(cudaEventRecord(ctx->ev1, s));
    unsigned long long* h = ctx->pin->graphs_ctrl;
    DQ_CUDA(cudaMemcpyAsync(h, d_ctrl.p, sizeof ctx->pin->graphs_ctrl, cudaMemcpyDeviceToHost, s));
    DQ_CUDA(cudaStreamSynchronize(s));
    DQ_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    DQ_CUDA(cudaEventElapsedTime(&ms_search, ctx->ev2, ctx->ev3));
    if (h[5]) { g_err = "an instance has an edge endpoint out of range or a self-loop"; return DQ_ERR_UNSUPPORTED; }
    if (stats) {
        stats->n_sat = h[1]; stats->n_unsat = h[2]; stats->n_budget = h[3]; stats->total_nodes = h[4];
        stats->kernel_ms = ms; stats->search_kernel_ms = ms_search; stats->kernel_launches = launches;
    }
    return DQ_OK;
}

static int check_edge_off(const int64_t* edge_off, int64_t n) {
    if (edge_off[0] != 0) { g_err = "edge_off[0] must be 0"; return DQ_ERR_INVALID; }
    for (int64_t i = 0; i < n; i++) if (edge_off[i + 1] < edge_off[i]) { g_err = "edge_off must be non-decreasing"; return DQ_ERR_INVALID; }
    return DQ_OK;
}

static int check_edges(int nv, const uint8_t* edges, long long total) {
    for (long long e = 0; e < total; e++) {
        const uint8_t u = edges[2 * e], v = edges[2 * e + 1];
        if (u >= nv || v >= nv) { g_err = "edge endpoint out of range"; return DQ_ERR_INVALID; }
        if (u == v) { g_err = "edge with u == v"; return DQ_ERR_UNSUPPORTED; }
    }
    return DQ_OK;
}

// dq_solve_batch_graphs and dq_count_batch_graphs (n_solutions non-null) once their arguments are checked: the host
// buffers around run_batch_graphs.
static int batch_graphs_host(int32_t nv, int32_t k, const int64_t* edge_off, const uint8_t* edges, int64_t n,
                             const dq_batch_opts* opts, uint8_t* colours, uint64_t* nodes, uint8_t* status,
                             dq_batch_stats* stats, uint64_t* n_solutions = nullptr, unsigned long long limit = 0) {
    const long long total = edge_off[n];
    DeviceCtx* ctx = nullptr;
    DQ_CUDA(device_ctx(&ctx));
    cudaStream_t s = ctx->stream;
    DevBuf<long long> d_off; DevBuf<uint8_t> d_edges, d_col, d_status; DevBuf<unsigned long long> d_nodes, d_nsol;
    StreamDrain drain{s};
    const long long edge_bytes = (2 * total + 15) & ~15ll;
    DQ_CUDA(d_off.reserve(n + 1)); DQ_CUDA(d_edges.reserve(std::max<long long>(edge_bytes, 16))); DQ_CUDA(d_col.reserve((size_t)n * nv));
    DQ_CUDA(d_status.reserve(n)); DQ_CUDA(d_nodes.reserve(n));
    if (n_solutions) DQ_CUDA(d_nsol.reserve(n));
    DQ_CUDA(cudaMemcpyAsync(d_off.p, edge_off, (n + 1) * sizeof(long long), cudaMemcpyHostToDevice, s));
    if (total) DQ_CUDA(cudaMemcpyAsync(d_edges.p, edges, 2 * total, cudaMemcpyHostToDevice, s));
    GraphBatchDev B{d_off.p, d_edges.p, edge_bytes, d_col.p, d_nodes.p, d_status.p, edges, d_nsol.p};
    int rc = run_batch_graphs(nv, k, edge_off, B, n, opts, stats, limit);
    if (rc != DQ_OK) return rc;
    DQ_CUDA(cudaMemcpyAsync(colours, d_col.p, (size_t)n * nv, cudaMemcpyDeviceToHost, s));
    DQ_CUDA(cudaMemcpyAsync(nodes, d_nodes.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    DQ_CUDA(cudaMemcpyAsync(status, d_status.p, (size_t)n, cudaMemcpyDeviceToHost, s));
    if (n_solutions) DQ_CUDA(cudaMemcpyAsync(n_solutions, d_nsol.p, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    DQ_CUDA(cudaStreamSynchronize(s));
    if (stats) { stats->h2d_bytes = (size_t)(n + 1) * 8 + 2 * (size_t)total; stats->d2h_bytes = (size_t)n * (nv + (n_solutions ? 17 : 9)); }
    return DQ_OK;
}

extern "C" {

int dq_solve_batch_graphs(int32_t nv, int32_t k, const int64_t* edge_off, const uint8_t* edges, int64_t n,
                          const dq_batch_opts* opts, uint8_t* colours, uint64_t* nodes, uint8_t* status,
                          dq_batch_stats* stats) {
    if (nv < 1 || nv > kMaxGraphVertices || k < 1 || k > 32 || n < 0) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return DQ_OK;
    if (!edge_off || !colours || !nodes || !status) { g_err = "null buffer"; return DQ_ERR_INVALID; }
    int rc = check_edge_off(edge_off, n);
    if (rc != DQ_OK) return rc;
    const long long total = edge_off[n];
    if (total && !edges) { g_err = "null edge buffer"; return DQ_ERR_INVALID; }
    if (opts && opts->engine == DQ_ENGINE_LANE && k > 4) { g_err = "the lane engine serves k <= 4"; return DQ_ERR_UNSUPPORTED; }
    // the lane engine checks the lists on the device (k_graphs_adjacency); the others trust them: one pass on the host
    const int engine = opts ? opts->engine : DQ_ENGINE_AUTO;
    if (!(k <= 4 && (engine == DQ_ENGINE_LANE || (engine == DQ_ENGINE_AUTO && n >= 4096)))) {
        rc = check_edges(nv, edges, total);
        if (rc != DQ_OK) return rc;
    }
    return batch_graphs_host(nv, k, edge_off, edges, n, opts, colours, nodes, status, stats);
}

int dq_count_batch_graphs(int32_t nv, int32_t k, const int64_t* edge_off, const uint8_t* edges, int64_t n,
                          const dq_count_opts* opts, uint64_t* n_solutions, uint8_t* colours, uint64_t* nodes,
                          uint8_t* status, dq_batch_stats* stats) {
    if (nv < 1 || nv > kMaxGraphVertices || k < 1 || k > 32 || n < 0) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    int rc = check_count_opts(opts);
    if (rc != DQ_OK) return rc;
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return DQ_OK;
    if (!edge_off || !n_solutions || !colours || !nodes || !status) { g_err = "null buffer"; return DQ_ERR_INVALID; }
    rc = check_edge_off(edge_off, n);
    if (rc != DQ_OK) return rc;
    const long long total = edge_off[n];
    if (total && !edges) { g_err = "null edge buffer"; return DQ_ERR_INVALID; }
    rc = check_edges(nv, edges, total);              // (the warp engine trusts the lists)
    if (rc != DQ_OK) return rc;
    const dq_batch_opts o{opts ? opts->node_budget : 0, DQ_ENGINE_WARP, 0};
    return batch_graphs_host(nv, k, edge_off, edges, n, &o, colours, nodes, status, stats, n_solutions,
                             opts ? opts->solution_limit : 0);
}

int dq_solve_batch_graphs_dev(int32_t nv, int32_t k, const int64_t* edge_off, const int64_t* edge_off_dev, const uint8_t* edges_dev,
                              int64_t n, const dq_batch_opts* opts, uint8_t* colours_dev, uint64_t* nodes_dev, uint8_t* status_dev,
                              dq_batch_stats* stats) {
    if (nv < 1 || nv > kMaxGraphVertices || k < 1 || k > 32 || n < 0) { g_err = "bad argument"; return DQ_ERR_INVALID; }
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return DQ_OK;
    if (!edge_off || !edge_off_dev || !colours_dev || !nodes_dev || !status_dev) { g_err = "null buffer"; return DQ_ERR_INVALID; }
    int rc = check_edge_off(edge_off, n);
    if (rc != DQ_OK) return rc;
    if (edge_off[n] && !edges_dev) { g_err = "null edge buffer"; return DQ_ERR_INVALID; }
    if (((uintptr_t)edges_dev & 15) != 0) { g_err = "edges_dev must be 16-byte aligned"; return DQ_ERR_INVALID; }
    // the edge lists cannot be validated on the host here: only the lane-group engine checks them on the device
    if (k > 4 || (opts && opts->engine != DQ_ENGINE_AUTO && opts->engine != DQ_ENGINE_LANE)) {
        g_err = "device-resident graph batches run on the lane engine (k <= 4) only"; return DQ_ERR_UNSUPPORTED;
    }
    GraphBatchDev B{(const long long*)edge_off_dev, edges_dev, (2 * (long long)edge_off[n] + 15) & ~15ll, colours_dev,
                    (unsigned long long*)nodes_dev, status_dev, nullptr};
    dq_batch_opts o = opts ? *opts : dq_batch_opts{0, 0, 0};
    o.engine = DQ_ENGINE_LANE;                           // (no fall-back to an engine that trusts the edge lists)
    return run_batch_graphs(nv, k, edge_off, B, n, &o, stats);
}

int dq_measure_int_peak(double* lane_ops_per_s, double* ms_out) {
    int dev = 0, sms = 0;
    DQ_CUDA(cudaGetDevice(&dev));
    DQ_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int blocks = sms * 2, threads = 1024, iters = 4096;
    uint32_t* out = nullptr;
    DQ_CUDA(cudaMalloc(&out, (size_t)blocks * threads * 4));
    cudaEvent_t e0, e1;
    DQ_CUDA(cudaEventCreate(&e0)); DQ_CUDA(cudaEventCreate(&e1));
    k_int_peak<<<blocks, threads>>>(out, 64);
    float best = 1e30f;
    for (int r = 0; r < 5; r++) {
        DQ_CUDA(cudaEventRecord(e0));
        k_int_peak<<<blocks, threads>>>(out, iters);
        DQ_CUDA(cudaEventRecord(e1));
        DQ_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        DQ_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        best = std::min(best, ms);
    }
    DQ_CUDA(cudaGetLastError());
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(out);
    const double ops = (double)blocks * threads * (double)iters * 16.0 * 8.0;   // exactly one lop3.b32 per statement
    if (lane_ops_per_s) *lane_ops_per_s = ops / (best * 1e-3);
    if (ms_out) *ms_out = best;
    return DQ_OK;
}

}  // extern "C"
