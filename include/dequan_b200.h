/*
 * dequan_b200.h — C ABI of the B200-native forward-checking search engine.
 *
 * The reference (nsweb/dequan) is a single C++ header with no FFI of its own
 * (SURVEY.md §8b): its "boundary" is the public C++ modelling API.  This header
 * is the flat, POD, caller-owned-memory interface that the drop-in C++ header
 * (include/dequan.h) lowers that API onto.  Each entry point names the
 * reference interface it stands in for.
 *
 *   reference                                         this ABI
 *   ------------------------------------------------  -------------------------
 *   CSP::AddIntVar/AddFixedVar/AddBoolVar             dq_model_desc.dom_*
 *     (dequan.h:454-476)
 *   CSP::AddConstraint<T> + FinalizeModel             dq_model_desc.con_* +
 *     (dequan.h:477-492)                                dq_compile()
 *   Assignment::Reset  (dequan.h:365-395)             dq_compile() (static order)
 *   CSP::ForwardCheckingStep (dequan.h:494-571)       dq_solve_tree(), dq_solve_batch*
 *   Assignment::inst_vars / stats.assigned_vars       dq_result
 *     (dequan.h:310, 67)
 *
 * Conventions: every function returns 0 (DQ_OK) or a negative dq_status error
 * code; no exceptions cross the ABI; all pointers are plain host pointers
 * unless the name says `_dev`; the library is thread-compatible (one handle
 * per thread), not thread-safe.  There is no CPU execution path: every solve
 * runs on the current CUDA device and fails with DQ_ERR_CUDA if there is none.
 */
#ifndef DEQUAN_B200_H
#define DEQUAN_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status / error codes ------------------------------------------------ */
enum dq_status {
    DQ_OK              =  0,
    DQ_ERR_INVALID     = -1,  /* malformed descriptor / argument                 */
    DQ_ERR_UNSUPPORTED = -2,  /* model outside the device engine's scope         */
    DQ_ERR_CUDA        = -3,  /* CUDA runtime error or no device                 */
    DQ_ERR_NOMEM       = -4,
    DQ_ERR_INTERNAL    = -5
};

/* search outcome, per tree / per instance */
enum dq_outcome {
    DQ_UNSAT  = 0,            /* ForwardCheckingStep would return false          */
    DQ_SAT    = 1,            /* ForwardCheckingStep would return true           */
    DQ_BUDGET = 2             /* node budget exhausted before either             */
};

/* ---- model descriptor ------------------------------------------------------
 * Mirrors CSP::vars / CSP::domains / CSP::constraints (dequan.h:349-354) as
 * flat int32 arrays.  Variable ids are dense 0..n_vars-1 in AddIntVar order.
 * Device scope: n_vars <= 1022, every domain <= 64 values (templates of the batch entry
 * points: <= 32 values), binary constraints; beyond it dq_compile / the solve returns
 * DQ_ERR_UNSUPPORTED.
 */
enum dq_domain_type {           /* dequan::DomainType (dequan.h:70-74)           */
    DQ_DOM_VALUES = 0,          /* explicit list, iteration = list order          */
    DQ_DOM_RANGES = 1           /* flat [min0,max0,min1,max1,...) half-open        */
};

enum dq_op {                    /* dequan::OpConstraint::Op (dequan.h:176-184)   */
    DQ_OP_EQUAL = 0, DQ_OP_NOTEQUAL = 1, DQ_OP_SUPEQUAL = 2,
    DQ_OP_SUP = 3, DQ_OP_INFEQUAL = 4, DQ_OP_INF = 5
};

enum dq_con_kind {
    DQ_CON_OP      = 0,  /* OpConstraint        data = {v0, v1, op, offset}      (dequan.h:174-197) */
    DQ_CON_EQ      = 1,  /* EqualityConstraint  data = {v0, v1}                  (dequan.h:200-211) */
    DQ_CON_ALLDIFF = 2,  /* AllDifferentConstraint data = {vars...}              (dequan.h:257-268) */
    DQ_CON_ORRANGE = 3,  /* OrRangeConstraint   data = {v0, v1, min, max}        (dequan.h:242-254) */
    DQ_CON_TABLE   = 4,  /* user-defined binary Constraint, tabulated Evaluate:
                            data = {v0, v1, a0, b0, a1, b1, ...} allowed (v0,v1)
                            value pairs; check-only (default AplyArcConsistency,
                            dequan.h:147)                                         */
    DQ_CON_FILTER  = 5   /* user-defined binary Constraint that overrides
                            AplyArcConsistency (dequan.h:145-147), tabulated:
                            data = {v0, v1, n_allow, n_keep01, n_keep10, then
                            n_allow pairs Evaluate accepts, n_keep01 pairs (a,b):
                            assigning v0=a leaves b in v1's domain, n_keep10 pairs
                            (a,b): assigning v1=b leaves a in v0's domain}; all
                            pairs are (value of v0, value of v1)                  */
};

typedef struct dq_model_desc {
    int32_t        n_vars;
    const int32_t *dom_type;   /* [n_vars]   dq_domain_type                       */
    const int32_t *dom_off;    /* [n_vars+1] offsets into dom_vals                */
    const int32_t *dom_vals;   /* flat domain storage                             */
    int32_t        n_cons;
    const int32_t *con_kind;   /* [n_cons]   dq_con_kind                          */
    const int32_t *con_off;    /* [n_cons+1] offsets into con_data                */
    const int32_t *con_data;   /* flat constraint payloads, see dq_con_kind       */
    const int32_t *assign_order; /* optional [n_vars] permutation of the var ids =
                                  Assignment::assign_order (dequan.h:316) when the
                                  caller supplies its own; NULL = the order
                                  Assignment::Reset computes (dequan.h:376-394)      */
} dq_model_desc;

/* ---- options / results ---------------------------------------------------- */
enum dq_mode {
    DQ_MODE_FIRST     = 0,   /* stop at the DFS-first solution (reference behaviour) */
    DQ_MODE_COUNT_ALL = 1    /* exhaust the tree: solution count + node count; the
                                reference equivalent is a counting Constraint linked
                                last to the last variable (SURVEY.md §8c)            */
};

enum dq_engine {
    DQ_ENGINE_AUTO  = 0,     /* fastest engine the compiled model qualifies for
                                (FIRST mode on the N-Queens class, one partition, no
                                budget: the class's first-solution warp, reported as
                                DQ_ENGINE_LANE)                                      */
    DQ_ENGINE_WARP  = 1,     /* generic warp-cooperative DFS (any supported model)  */
    DQ_ENGINE_LANE  = 2,     /* lane-per-subtree / lane-per-instance closed-form DFS
                                (N-Queens class trees, 9x9 Sudoku class batches,
                                colouring batches with k <= 4: a group of 1..32 lanes
                                per instance)                                       */
    DQ_ENGINE_REG   = 3      /* register-resident warp DFS: trees of models with at
                                most 32 variables, colouring batches with k <= 4     */
};

typedef struct dq_tree_opts {
    int32_t  mode;           /* dq_mode                                             */
    int32_t  split_depth;    /* prefix depth for subtree split; <=0 = automatic     */
    int32_t  part_rank;      /* this caller's partition id   (0 for single GPU)     */
    int32_t  part_count;     /* number of partitions         (1 for single GPU)     */
    uint64_t node_budget;    /* 0 = unlimited (FIRST mode only)                     */
    int32_t  engine;         /* dq_engine                                           */
    int32_t  flags;          /* DQ_TREE_* bits                                      */
} dq_tree_opts;

/* dq_tree_opts.flags: fill dq_tree_result.search_kernel_ms (CUDA events around the search kernel).  The solve is then
 * queued call by call; without the flag the N-Queens engine replays its queue as one CUDA graph and reports only
 * kernel_ms, measured around the graph.                                                                         */
#define DQ_TREE_TIME_KERNELS 1

typedef struct dq_tree_result {
    int32_t  outcome;        /* dq_outcome (COUNT_ALL: SAT iff n_solutions>0)       */
    int32_t  n_prefixes;     /* FC-surviving prefixes at split depth (all parts)    */
    uint64_t n_solutions;    /* COUNT_ALL: solutions in this partition; FIRST: 0/1  */
    uint64_t n_nodes;        /* Assignment::AssignVar calls (dequan.h:416-423)      */
    uint64_t first_key;      /* DFS index of the prefix holding the first solution
                                found by this partition, UINT64_MAX if none         */
    uint64_t nodes_before_first; /* FIRST: nodes dequan visits up to and including
                                the first solution, counting only this partition's
                                subtrees with index <= first_key (see DESIGN.md)    */
    double   kernel_ms;      /* device time of the search kernels (CUDA events)     */
    int32_t  engine_used;    /* dq_engine actually run                              */
    int32_t  split_depth_used;
    uint64_t kernel_launches;/* number of engine kernels launched by this call      */
    double   search_kernel_ms;/* device time of the dominant (subtree DFS) kernel alone */
    uint64_t frontier_nodes; /* nodes counted by the frontier-expansion kernels above
                                the split depth (the DFS kernel counted the rest)     */
} dq_tree_result;

typedef struct dq_batch_opts {
    uint64_t node_budget;    /* per instance, 0 = unlimited                         */
    int32_t  engine;         /* dq_engine                                           */
    int32_t  task_nodes;     /* lane engine test knob: > 0 makes every search older than
                                this many nodes hand stack levels to the task pool
                                whether or not other lanes are idle; 0 = demand
                                driven (production)                                 */
} dq_batch_opts;

typedef struct dq_batch_stats {
    uint64_t n_sat, n_unsat, n_budget;   /* n_sat + n_unsat + n_budget == n.  Status-3 rows (a given that is not
                                            in its variable's template domain) count under n_unsat.          */
    uint64_t total_nodes;
    double   kernel_ms;
    uint64_t kernel_launches;
    uint64_t h2d_bytes, d2h_bytes;
    double   search_kernel_ms; /* graph batches: device time of the search kernel alone    */
} dq_batch_stats;

typedef struct dq_model dq_model;   /* compiled model: flat tables, host + HBM copies */

/* ---- entry points ----------------------------------------------------------*/

/* Library / device probe.  Returns DQ_OK and fills *sm_count, *cc (e.g. 100).     */
int dq_device_info(int32_t *sm_count, int32_t *cc, char *name, size_t name_len);

/* Select the CUDA device this thread's subsequent calls run on (one process per GPU under
 * torchrun: pass LOCAL_RANK).  Handles are bound to the device current at their first solve. */
int dq_set_device(int32_t ordinal);

/* Lower a model to the flat position-space table: static assign order
 * (Assignment::Reset, dequan.h:376-394), bitset domains, forward arc programs.
 * Replaces CSP::FinalizeModel + Assignment::Reset.                               */
int dq_compile(const dq_model_desc *desc, dq_model **out);
void dq_free(dq_model *m);

/* Introspection of the compiled table (host side; used by the tests).            */
int dq_model_info(const dq_model *m, int32_t *n_vars, int32_t *max_dom,
                  int32_t *n_arcs, int32_t *model_class);
int dq_model_order(const dq_model *m, int32_t *order_out /* [n_vars] */);
/* Bytes of the flat tables a solve uploads to HBM for this model (h2d accounting). */
int dq_model_table_bytes(const dq_model *m, uint64_t *bytes);

/* Solve one model (single tree).  Replaces `a.Reset(csp); csp.ForwardCheckingStep(a)`
 * (dequan.h:292, 347).  first_solution[n_vars] receives InstVar values by var id
 * (all INT32_MIN+1 == InstVar::UNASSIGNED if none).                              */
int dq_solve_tree(dq_model *m, const dq_tree_opts *opts,
                  dq_tree_result *res, int32_t *first_solution);

/* The same solve on `n_devices` GPUs of this process: the prefix-split tree is dealt to the devices (partition i ->
 * devices[i]; NULL = ordinals 0..n_devices-1; an ordinal may repeat), one worker thread per device, and the tail —
 * solution-count and node-count sums, lexicographic-min first solution — is reduced here.  opts->part_rank /
 * part_count must be 0 / 1.  res: sums over the devices; kernel_ms = the slowest device.  One call, one answer: what
 * `a.Reset(csp); csp.ForwardCheckingStep(a)` (dequan.h:292, 347) is on one thread of the reference.            */
int dq_solve_tree_multi(dq_model *m, const dq_tree_opts *opts, int32_t n_devices, const int32_t *devices,
                        dq_tree_result *res, int32_t *first_solution);

/* Many independent models in one call: per model, what dq_solve_tree(models[i], opts, ...) returns.  Small trees are
 * searched one warp per model in one launch; a tree that outgrows a warp's node budget is solved by the split search
 * afterwards (*n_split counts them).  solutions: first solutions concatenated in list order, model i's n_vars values
 * starting at the sum of the earlier models' n_vars (InstVar::UNASSIGNED where none); NULL = not wanted.
 * opts: mode FIRST or COUNT_ALL, engine AUTO or WARP, one partition, no split depth, no node budget.  A handle may
 * appear more than once; every handle belongs to the calling thread and must not be bound to another device.
 * stats (may be NULL): n_sat / n_unsat, total_nodes, kernel_ms = device time of the in-batch launches,
 * kernel_launches including the split solves, h2d_bytes / d2h_bytes of the batch's own copies; n_budget is 0.      */
int dq_solve_models(dq_model *const *models, int64_t n, const dq_tree_opts *opts, int32_t *outcome,
                    uint64_t *n_solutions, uint64_t *n_nodes, int32_t *solutions, int64_t *n_split,
                    dq_batch_stats *stats);

/* FIRST-mode node accounting across partitions (multi-GPU): after dq_solve_tree, the number of
 * nodes (AssignVar calls, dequan.h:416-423) the reference's sequential search would have visited
 * up to and including the solution inside prefix `key`, restricted to the subtrees this
 * partition owns (partition 0 also owns the levels above the split).  Summed over all
 * partitions with key = the global minimum first_key it equals stats.assigned_vars of the
 * reference.  key == UINT64_MAX: everything this partition explored.                       */
int dq_tree_nodes_upto(dq_model *m, uint64_t key, uint64_t *nodes);

/* Every solution of the model, in the reference's DFS order (static variable order, domain value order): what a
 * counting Constraint linked last to the last variable sees when it snapshots Assignment::inst_vars on every
 * Evaluate (SURVEY.md par. 8c; the reference has no enumeration mode of its own, dequan.h:494-571 stops at the first
 * solution).  solutions[i * n_vars + v] = value of variable v in the i-th solution.  opts->mode is ignored (the
 * solve is COUNT_ALL); res is filled as by dq_solve_tree.  With opts->part_count > 1: this partition's solutions.
 * More than `cap` solutions: returns DQ_ERR_NOMEM, res->n_solutions holds the number, nothing is written.        */
int dq_enumerate_solutions(dq_model *m, const dq_tree_opts *opts, dq_tree_result *res,
                           int32_t *solutions /* [cap][n_vars] */, uint64_t cap, uint64_t *n_written);

/* Batch of independent instances sharing the template's constraint graph but with
 * per-instance initial domains: cells[i*stride + v] == 0 keeps variable v's template
 * domain, any other byte c fixes it to the single value c (AddFixedVar, dequan.h:467).
 * Per instance: FIRST-mode solve; outputs status[i] (dq_outcome, or 3 with 0 nodes when a
 * given byte is not a value of its variable's template domain), nodes[i],
 * solution[i*stride + v] (value as byte, 0 if none).  Each instance is searched in
 * Reset's order of its own domains, or in the template's assign_order if the caller
 * supplied one.  Host buffers.                                                    */
int dq_solve_batch_cells(dq_model *tmpl, const uint8_t *cells, int64_t n, int32_t stride,
                         const dq_batch_opts *opts, uint8_t *solution,
                         uint64_t *nodes, uint8_t *status, dq_batch_stats *stats);

/* Same, with all buffers already resident in device memory (bench "value" leg).  */
int dq_solve_batch_cells_dev(dq_model *tmpl, const uint8_t *cells_dev, int64_t n, int32_t stride,
                             const dq_batch_opts *opts, uint8_t *solution_dev,
                             uint64_t *nodes_dev, uint8_t *status_dev, dq_batch_stats *stats);

/* Batch of independent k-colouring instances (one graph per instance):
 * variables 0..n_vertices-1 = AddIntVar(0,k); one OpConstraint(u,v,NotEqual,0) per
 * edge.  edge_off[n+1] indexes edges[2*e], edges as (u,v) byte pairs (1 <= n_vertices <= 254;
 * more is refused with DQ_ERR_INVALID, as by every graph entry point).
 * colours[i*n_vertices + v] = colour or 0xFF.                                     */
int dq_solve_batch_graphs(int32_t n_vertices, int32_t k, const int64_t *edge_off,
                          const uint8_t *edges, int64_t n, const dq_batch_opts *opts,
                          uint8_t *colours, uint64_t *nodes, uint8_t *status,
                          dq_batch_stats *stats);

/* Same, with the edge lists and the outputs resident in device memory (bench "value" leg).
 * edge_off is the HOST copy of the offsets (it sizes the per-instance adjacency records),
 * edge_off_dev / edges_dev the device copies; edges_dev must be 16-byte aligned and readable up
 * to the next multiple of 16 bytes (the lists are fetched with 16-byte bulk copies).  k <= 4;
 * edge endpoints are checked on the device (DQ_ERR_UNSUPPORTED if an instance is malformed).    */
int dq_solve_batch_graphs_dev(int32_t n_vertices, int32_t k, const int64_t *edge_off,
                              const int64_t *edge_off_dev, const uint8_t *edges_dev, int64_t n,
                              const dq_batch_opts *opts, uint8_t *colours_dev, uint64_t *nodes_dev,
                              uint8_t *status_dev, dq_batch_stats *stats);

/* ---- counting batches --------------------------------------------------------
 * The instances of dq_solve_batch_cells / dq_solve_batch_graphs (same givens, status 3
 * rows, search order), each searched to the end with a counting Constraint linked last to
 * the last variable (SURVEY.md §8c) that passes, instead of failing, the solution_limit-th
 * solution: ForwardCheckingStep returns true there.  The node budget is checked on every
 * AssignVar before that constraint, as in the FIRST-mode batches.  Per instance:
 *   n_solutions[i]  every solution (limit 0); min(total, limit) (limit > 0: == limit means
 *                   "at least limit"); the solutions counted before the budget ran out;
 *   nodes[i]        AssignVar calls up to and including the node the search stopped at
 *                   (the whole tree, the one completing the limit-th solution, or budget + 1);
 *   status[i]       DQ_SAT (>= 1 solution, tree exhausted or limit reached), DQ_UNSAT,
 *                   DQ_BUDGET (budget ran out first, whatever was counted), 3 (bad given:
 *                   0 nodes, 0 solutions);
 *   solution[i] / colours[i]  the DFS-first solution whenever n_solutions[i] >= 1, in the
 *                   layout of the FIRST-mode batch; otherwise 0 (cells) / 0xFF (graphs).
 * With solution_limit 1, status, nodes and solution equal the FIRST-mode batch's.  The
 * count runs on the generic warp engine: engine AUTO or WARP (LANE and REG are refused
 * with DQ_ERR_UNSUPPORTED).  opts NULL = every solution, no budget, AUTO.  stats as for
 * the FIRST-mode batches.  Host buffers.                                                    */
typedef struct dq_count_opts {
    uint64_t node_budget;    /* per instance, 0 = unlimited                         */
    uint64_t solution_limit; /* per instance, 0 = count every solution              */
    int32_t  engine;         /* dq_engine: AUTO or WARP                             */
} dq_count_opts;

int dq_count_batch_cells(dq_model *tmpl, const uint8_t *cells, int64_t n, int32_t stride,
                         const dq_count_opts *opts, uint64_t *n_solutions, uint8_t *solution,
                         uint64_t *nodes, uint8_t *status, dq_batch_stats *stats);

int dq_count_batch_graphs(int32_t n_vertices, int32_t k, const int64_t *edge_off,
                          const uint8_t *edges, int64_t n, const dq_count_opts *opts,
                          uint64_t *n_solutions, uint8_t *colours, uint64_t *nodes,
                          uint8_t *status, dq_batch_stats *stats);

/* On-disk instance formats for the batch entry points (host-side parsing only).
 * Sudoku: one puzzle per line, 81 characters, '1'..'9' givens, '0' '.' '_' '*' blank; blank
 * lines and lines starting with '#' are skipped.  cells[i*81 + c] as dq_solve_batch_cells
 * expects (stride 81).  *n_out = puzzles parsed.                                          */
int dq_parse_sudoku_lines(const char *text, size_t len, uint8_t *cells, int64_t cap, int64_t *n_out);
/* DIMACS .col: "c" comments, one "p edge N M", then "e u v" (1-based).  edges[2*e] = (u-1, v-1)
 * as dq_solve_batch_graphs expects; N <= 254.                                               */
int dq_parse_dimacs_col(const char *text, size_t len, int32_t *n_vertices, uint8_t *edges,
                        int64_t cap_edges, int64_t *n_edges);

/* Integer-pipe microbenchmark (LOP3 issue rate) used as the search roofline
 * denominator: returns measured lane-ops/s on the current device.                */
int dq_measure_int_peak(double *lane_ops_per_s, double *ms);

const char *dq_last_error(void);
const char *dq_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DEQUAN_B200_H */
