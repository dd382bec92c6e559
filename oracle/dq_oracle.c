/*
 * oracle/dq_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT.
 *
 * Plain-C CPU restatement of the reference's forward-checking search
 * (/root/reference/dequan.h).  It deliberately keeps the reference's own data
 * representation — domains as value lists or half-open range lists, a
 * copy-on-first-write trail per depth, constraints walked in link order — so that
 * it is an independent statement of the algorithm from the bitset/arc-table design
 * of the CUDA engine it is used to check.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline leg may load this; the product never does.
 *
 * Parity pin: checked against the unmodified reference (oracle/_ref/dequan_ref,
 * built from /root/reference by oracle/Makefile) on the reference's own three test
 * scenarios, N-Queens 4..12 all-solutions and randomised models covering every
 * constraint kind and domain quirk; the outputs are committed under tests/golden/.
 *
 * Every function cites the reference lines it follows.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <limits.h>
#include "dequan_b200.h"

#define UNASSIGNED (-INT_MAX)            /* InstVar::UNASSIGNED, dequan.h:122 */

/* ---- growable int list (stands in for Array<int>, dequan.h:29-51) ---------- */
typedef struct { int *v; int n, cap; } ivec;

static void iv_reserve(ivec *a, int cap) {
    if (cap <= a->cap) return;
    int nc = a->cap ? a->cap * 2 : 8;
    if (nc < cap) nc = cap;
    a->v = (int *)realloc(a->v, (size_t)nc * sizeof(int));
    a->cap = nc;
}
static void iv_push(ivec *a, int x) { iv_reserve(a, a->n + 1); a->v[a->n++] = x; }
static void iv_erase(ivec *a, int first, int last) {          /* [first,last) */
    memmove(a->v + first, a->v + last, (size_t)(a->n - last) * sizeof(int));
    a->n -= last - first;
}
static void iv_insert(ivec *a, int idx, int x) {
    iv_reserve(a, a->n + 1);
    memmove(a->v + idx + 1, a->v + idx, (size_t)(a->n - idx) * sizeof(int));
    a->v[idx] = x; a->n++;
}
static void iv_copy(ivec *dst, const ivec *src) {
    iv_reserve(dst, src->n);
    memcpy(dst->v, src->v, (size_t)src->n * sizeof(int));
    dst->n = src->n;
}

/* ---- Domain (dequan.h:76-96) ----------------------------------------------- */
typedef struct { int type; ivec vals; } dom_t;

/* Domain::Size, dequan.h:941-956 */
static int dom_size(const dom_t *d) {
    if (d->type == DQ_DOM_VALUES) return d->vals.n;
    int s = 0;
    for (int r = 0; r < d->vals.n; r += 2) s += d->vals.v[r + 1] - d->vals.v[r];
    return s;
}
/* Domain::Intersect(val), dequan.h:957-984 — a no-op when val is absent (SURVEY §9 Q3) */
static void dom_intersect(dom_t *d, int val) {
    if (d->type == DQ_DOM_VALUES) {
        for (int i = 0; i < d->vals.n; i++)
            if (d->vals.v[i] == val) { d->vals.n = 0; iv_push(&d->vals, val); break; }
    } else {
        for (int r = 0; r < d->vals.n; r += 2)
            if (d->vals.v[r] <= val && val < d->vals.v[r + 1]) {
                d->type = DQ_DOM_VALUES; d->vals.n = 0; iv_push(&d->vals, val); break;
            }
    }
}
/* Domain::Exclude, dequan.h:985-1031 — Values: first match only; Ranges: shrink/split/drop */
static void dom_exclude(dom_t *d, int val) {
    if (d->type == DQ_DOM_VALUES) {
        for (int i = 0; i < d->vals.n; i++)
            if (d->vals.v[i] == val) { iv_erase(&d->vals, i, i + 1); break; }
        return;
    }
    for (int r = 0; r < d->vals.n; r += 2) {
        int lo = d->vals.v[r], hi = d->vals.v[r + 1];
        if (lo <= val && val < hi) {
            if (hi - lo <= 1) iv_erase(&d->vals, r, r + 2);
            else if (val == lo) d->vals.v[r] = val + 1;
            else if (val + 1 == hi) d->vals.v[r + 1] = val;
            else {
                d->vals.v[r + 1] = val;
                iv_insert(&d->vals, r + 2, hi);
                iv_insert(&d->vals, r + 2, val + 1);
            }
            break;
        }
    }
}
/* Domain::ExcludeSup, dequan.h:1105-1138 — drop values >= rmax */
static void dom_exclude_sup(dom_t *d, int rmax) {
    if (d->type == DQ_DOM_VALUES) {
        int w = 0;
        for (int i = 0; i < d->vals.n; i++) if (d->vals.v[i] < rmax) d->vals.v[w++] = d->vals.v[i];
        d->vals.n = w;
        return;
    }
    for (int r = 0; r < d->vals.n;) {
        int lo = d->vals.v[r], hi = d->vals.v[r + 1];
        int nh = hi < rmax ? hi : rmax;
        if (nh > lo) { d->vals.v[r + 1] = nh; r += 2; } else iv_erase(&d->vals, r, r + 2);
    }
}
/* Domain::ExcludeInf, dequan.h:1139-1172 — drop values < rmin */
static void dom_exclude_inf(dom_t *d, int rmin) {
    if (d->type == DQ_DOM_VALUES) {
        int w = 0;
        for (int i = 0; i < d->vals.n; i++) if (d->vals.v[i] >= rmin) d->vals.v[w++] = d->vals.v[i];
        d->vals.n = w;
        return;
    }
    for (int r = 0; r < d->vals.n;) {
        int lo = d->vals.v[r], hi = d->vals.v[r + 1];
        int nl = lo > rmin ? lo : rmin;
        if (hi > nl) { d->vals.v[r] = nl; r += 2; } else iv_erase(&d->vals, r, r + 2);
    }
}

/* ---- model + search state --------------------------------------------------- */
typedef struct { int kind; const int32_t *data; int n; } con_t;
typedef struct { int vid; dom_t saved; } saved_t;                 /* SavedDomain, dequan.h:98-106  */
typedef struct { saved_t *e; int n, cap; } frame_t;               /* SavedDomains, dequan.h:109-114 */

typedef struct {
    int nv, nc;
    con_t *cons;
    ivec *links;               /* Var::linked_constraints (dequan.h:280), constraint indices in link order */
    dom_t *dom0;               /* CSP::domains */
    /* Assignment (dequan.h:287-321) */
    int assigned;
    int *inst;
    dom_t *cur;
    frame_t *frames; int nframes;
    int *order;
    uint64_t validated, applied, nodes;
    /* harness extensions (mirror oracle/ref_driver.cpp's Counting/Budget constraints) */
    int count_all; uint64_t budget, evals, solutions; int busted;
    int32_t *first; int have_first;
    int32_t *all_out; uint64_t all_cap;      /* dqo_enumerate: inst_vars of every counted solution, in visiting order */
    /* prefix-partition emulation of the multi-GPU split (DESIGN.md "multi-GPU") */
    int split_depth, part_rank, part_count; uint64_t upto_key, prefix_counter, cur_prefix, first_key; int stop_all;
} search_t;

/* CSP::FinalizeModel -> Constraint::LinkVars, dequan.h:484-492, 588-592, 695-699, 839-843, 895-901 */
static void link_vars(search_t *s) {
    for (int c = 0; c < s->nc; c++) {
        const con_t *k = &s->cons[c];
        if (k->kind == DQ_CON_ALLDIFF) { for (int i = 0; i < k->n; i++) iv_push(&s->links[k->data[i]], c); }
        else { iv_push(&s->links[k->data[0]], c); iv_push(&s->links[k->data[1]], c); }
    }
}

/* Assignment::Reset, dequan.h:365-395: order by (initial Size asc, id asc) */
static search_t *g_sort_ctx;
static int order_cmp(const void *pa, const void *pb) {
    int a = *(const int *)pa, b = *(const int *)pb;
    int sa = dom_size(&g_sort_ctx->dom0[a]), sb = dom_size(&g_sort_ctx->dom0[b]);
    if (sa == sb) return a < b ? -1 : (a > b ? 1 : 0);
    return sa < sb ? -1 : 1;
}
static void reset_assignment(search_t *s) {
    s->assigned = 0;
    for (int i = 0; i < s->nv; i++) {
        s->inst[i] = UNASSIGNED;
        s->cur[i].type = s->dom0[i].type;
        iv_copy(&s->cur[i].vals, &s->dom0[i].vals);
        s->order[i] = i;
    }
    g_sort_ctx = s;
    qsort(s->order, (size_t)s->nv, sizeof(int), order_cmp);
    s->nframes = 0;
}

/* Assignment::EnsureSavedDomain, dequan.h:442-452 */
static void ensure_saved(search_t *s, int vid) {
    frame_t *f = &s->frames[s->nframes - 1];
    for (int i = 0; i < f->n; i++) if (f->e[i].vid == vid) return;
    if (f->n == f->cap) {
        int nc = f->cap ? f->cap * 2 : 8;
        f->e = (saved_t *)realloc(f->e, (size_t)nc * sizeof(saved_t));
        memset(f->e + f->cap, 0, (size_t)(nc - f->cap) * sizeof(saved_t));
        f->cap = nc;
    }
    saved_t *e = &f->e[f->n++];
    e->vid = vid; e->saved.type = s->cur[vid].type;
    iv_copy(&e->saved.vals, &s->cur[vid].vals);
}
/* Assignment::RestoreSavedDomainStep, dequan.h:431-440 (frame is NOT cleared) */
static void restore_step(search_t *s) {
    frame_t *f = &s->frames[s->nframes - 1];
    for (int i = 0; i < f->n; i++) {
        int vid = f->e[i].vid;
        s->cur[vid].type = f->e[i].saved.type;
        iv_copy(&s->cur[vid].vals, &f->e[i].saved.vals);
    }
}

enum { EV_NA = 0, EV_PASSED = 1, EV_FAILED = 2 };                 /* Constraint::Eval, dequan.h:136-141 */

/* (a, b) is one of the n value pairs at p (a FILTER's allow or keep list; repeats and foreign values are harmless) */
static int has_pair(const int32_t *p, int n, int a, int b) {
    for (int i = 0; i < n; i++) if (p[2 * i] == a && p[2 * i + 1] == b) return 1;
    return 0;
}

/* OpConstraint::Evaluate dequan.h:593-630; EqualityConstraint 700-709; OrRange 844-854;
 * AllDifferent 902-914; TABLE = user constraint as in oracle/ref_driver.cpp TableConstraint; FILTER = a user
 * constraint with its own filter, as tests/cpp/dropin_scenarios.cpp OrderedConstraint */
static int evaluate(search_t *s, const con_t *k, int last) {
    const int32_t *d = k->data;
    switch (k->kind) {
    case DQ_CON_OP: {
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED || b == UNASSIGNED) return EV_NA;
        int rhs = b + d[3], ok = 0;
        switch (d[2]) {
        case DQ_OP_EQUAL: ok = a == rhs; break;   case DQ_OP_NOTEQUAL: ok = a != rhs; break;
        case DQ_OP_SUPEQUAL: ok = a >= rhs; break; case DQ_OP_SUP: ok = a > rhs; break;
        case DQ_OP_INFEQUAL: ok = a <= rhs; break; case DQ_OP_INF: ok = a < rhs; break;
        }
        return ok ? EV_PASSED : EV_FAILED;
    }
    case DQ_CON_EQ: {
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED || b == UNASSIGNED) return EV_NA;
        return a == b ? EV_PASSED : EV_FAILED;
    }
    case DQ_CON_ORRANGE: {
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED || b == UNASSIGNED) return EV_NA;
        return ((a >= d[2] && a < d[3]) || (b >= d[2] && b < d[3])) ? EV_PASSED : EV_FAILED;
    }
    case DQ_CON_ALLDIFF: {
        int v = s->inst[last];
        for (int i = 0; i < k->n; i++) if (s->inst[d[i]] == v && d[i] != last) return EV_FAILED;
        return EV_PASSED;
    }
    case DQ_CON_TABLE: {
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED || b == UNASSIGNED) return EV_NA;
        for (int i = 2; i + 1 < k->n; i += 2) if (d[i] == a && d[i + 1] == b) return EV_PASSED;
        return EV_FAILED;
    }
    case DQ_CON_FILTER: {
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED || b == UNASSIGNED) return EV_NA;
        return has_pair(d + 5, d[2], a, b) ? EV_PASSED : EV_FAILED;
    }
    }
    return EV_NA;
}

/* DoCheck lambda of OpConstraint::AplyArcConsistency, dequan.h:636-669 */
static int op_filter(search_t *s, int vid, int oth, int op) {
    dom_t *dm = &s->cur[vid];
    ensure_saved(s, vid);
    switch (op) {
    case DQ_OP_EQUAL: dom_intersect(dm, oth); break;
    case DQ_OP_NOTEQUAL: dom_exclude(dm, oth); break;
    case DQ_OP_SUPEQUAL: dom_exclude_inf(dm, oth); break;
    case DQ_OP_SUP: dom_exclude_inf(dm, oth + 1); break;
    case DQ_OP_INFEQUAL: dom_exclude_sup(dm, oth + 1); break;
    case DQ_OP_INF: dom_exclude_sup(dm, oth); break;
    }
    return dm->vals.n != 0;
}

/* AplyArcConsistency of each kind: Op dequan.h:631-694 (op reversal 681-690), Equality 710-743,
 * OrRange 855-894 (body compiled out), AllDifferent 915-939, TABLE = base-class default 147, FILTER = the user's
 * override (dequan.h:145-147) */
static int apply_arc(search_t *s, const con_t *k, int last) {
    const int32_t *d = k->data;
    switch (k->kind) {
    case DQ_CON_OP: {
        s->applied++;
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED) return op_filter(s, d[0], b + d[3], d[2]);
        if (b == UNASSIGNED) {
            int rev = d[2];
            switch (d[2]) {
            case DQ_OP_SUPEQUAL: rev = DQ_OP_INFEQUAL; break; case DQ_OP_SUP: rev = DQ_OP_INF; break;
            case DQ_OP_INFEQUAL: rev = DQ_OP_SUPEQUAL; break; case DQ_OP_INF: rev = DQ_OP_SUP; break;
            default: break;
            }
            return op_filter(s, d[1], a - d[3], rev);
        }
        return 1;
    }
    case DQ_CON_EQ: {
        s->applied++;
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if (a == UNASSIGNED) return op_filter(s, d[0], b, DQ_OP_EQUAL);
        if (b == UNASSIGNED) return op_filter(s, d[1], a, DQ_OP_EQUAL);
        return 1;
    }
    case DQ_CON_ORRANGE:
        s->applied++;
        return 1;
    case DQ_CON_ALLDIFF: {
        s->applied++;
        int val = s->inst[last];
        for (int i = 0; i < k->n; i++) {
            int vid = d[i];
            if (s->inst[vid] == UNASSIGNED) {
                ensure_saved(s, vid);
                dom_exclude(&s->cur[vid], val);
                if (s->cur[vid].vals.n == 0) return 0;
            }
        }
        return 1;
    }
    case DQ_CON_FILTER: {
        /* a user constraint's own AplyArcConsistency, tabulated (include/dequan.h TabulateUserConstraint): with one
         * endpoint assigned, the other keeps the values its keep list pairs with the assigned value.  Values leave
         * through Exclude, so the order of the rest is unchanged. */
        s->applied++;
        int a = s->inst[d[0]], b = s->inst[d[1]];
        if ((a == UNASSIGNED) == (b == UNASSIGNED)) return 1;
        const int x_is_v0 = a != UNASSIGNED, q = x_is_v0 ? d[1] : d[0];
        const int32_t *keep = d + 5 + 2 * d[2] + (x_is_v0 ? 0 : 2 * d[3]);
        const int n_keep = x_is_v0 ? d[3] : d[4];
        ensure_saved(s, q);
        dom_t *dm = &s->cur[q];
        ivec vals = {0};                                  /* a snapshot: Exclude edits dm */
        if (dm->type == DQ_DOM_VALUES) {
            for (int i = 0; i < dm->vals.n; i++) iv_push(&vals, dm->vals.v[i]);
        } else {
            for (int r = 0; r < dm->vals.n; r += 2)
                for (int w = dm->vals.v[r]; w < dm->vals.v[r + 1]; w++) iv_push(&vals, w);
        }
        for (int i = 0; i < vals.n; i++) {
            const int w = vals.v[i];
            if (!(x_is_v0 ? has_pair(keep, n_keep, a, w) : has_pair(keep, n_keep, w, b))) dom_exclude(dm, w);
        }
        free(vals.v);
        return dm->vals.n != 0;
    }
    default: return 1;
    }
}

/* Assignment::ValidateVarConstraints, dequan.h:573-587, with the harness's Budget constraint
 * evaluated first and its Counting constraint evaluated last on the last variable. */
static int validate(search_t *s, int vid) {
    if (s->budget) {
        s->validated++;
        if (++s->evals > s->budget) { s->busted = 1; return 0; }
    }
    const ivec *l = &s->links[vid];
    for (int i = 0; i < l->n; i++) {
        s->validated++;
        if (evaluate(s, &s->cons[l->v[i]], vid) == EV_FAILED) return 0;
    }
    if (s->count_all && vid == s->order[s->nv - 1]) {
        s->validated++;
        if (!s->have_first) { for (int i = 0; i < s->nv; i++) s->first[i] = s->inst[i]; s->have_first = 1; s->first_key = s->cur_prefix; }
        if (s->all_out && s->solutions < s->all_cap)
            for (int i = 0; i < s->nv; i++) s->all_out[s->solutions * (uint64_t)s->nv + i] = s->inst[i];
        s->solutions++;
        return 0;
    }
    return 1;
}

static int fc_step(search_t *s);

/* LambdaStep of CSP::ForwardCheckingStep, dequan.h:508-541 */
static int try_value(search_t *s, int vid, int val) {
    /* Assignment::AssignVar, dequan.h:416-423 — this is "one node" */
    s->inst[vid] = val; s->assigned++;
    if (s->assigned > s->split_depth || s->part_rank == 0) s->nodes++;
    if (validate(s, vid)) {
        int ok = 1;
        const ivec *l = &s->links[vid];
        for (int i = 0; ok && i < l->n; i++) ok &= apply_arc(s, &s->cons[l->v[i]], vid);
        if (ok) ok = fc_step(s);
        if (ok) return 1;
        s->inst[vid] = UNASSIGNED; s->assigned--;          /* UnAssignVar, dequan.h:425-429 */
        restore_step(s);
    } else {
        s->inst[vid] = UNASSIGNED; s->assigned--;
    }
    return 0;
}

/* CSP::ForwardCheckingStep, dequan.h:494-571 */
static int fc_step(search_t *s) {
    if (s->assigned == s->nv) return 1;
    if (s->split_depth > 0 && s->assigned == s->split_depth) {
        /* an FC-surviving prefix = one unit of multi-GPU work, numbered in DFS order */
        uint64_t idx = s->prefix_counter++;
        int mine = (int)(idx % (uint64_t)s->part_count) == s->part_rank;
        if (idx == s->upto_key && !mine) { s->stop_all = 1; return 0; }
        if (!mine) return 0;
        s->cur_prefix = idx;
    }
    frame_t *f = &s->frames[s->nframes++];
    f->n = 0;
    int vid = s->order[s->assigned];
    const dom_t *dm = &s->cur[vid];
    int found = 0;
    if (dm->type == DQ_DOM_VALUES) {
        for (int i = 0; i < dm->vals.n && !found && !s->busted && !s->stop_all; i++)
            found = try_value(s, vid, dm->vals.v[i]);
    } else {
        for (int r = 0; r < dm->vals.n; r += 2) {
            int lo = dm->vals.v[r], hi = dm->vals.v[r + 1];
            for (int v = lo; v < hi && !found && !s->busted && !s->stop_all; v++) found = try_value(s, vid, v);
        }
    }
    if (found) return 1;
    s->nframes--;
    return 0;
}

/* ---- public entry points (loaded with ctypes by the tests) -------------------- */
typedef struct dqo_result {
    int32_t outcome;
    uint64_t solutions, nodes, validated_constraints, applied_arcs, first_key, n_prefixes;
} dqo_result;

typedef struct dqo_opts {
    int32_t mode;            /* dq_mode */
    int32_t split_depth;     /* 0 = no partition emulation */
    int32_t part_rank, part_count;
    uint64_t node_budget;
    uint64_t upto_key;       /* UINT64_MAX = no cut-off */
} dqo_opts;

static int dqo_run(const dq_model_desc *m, const dqo_opts *o, dqo_result *res,
                   int32_t *first /* [n_vars] */, int32_t *order_out /* [n_vars] or NULL */,
                   int32_t *all_out, uint64_t all_cap) {
    search_t s;
    memset(&s, 0, sizeof s);
    s.all_out = all_out; s.all_cap = all_cap;
    s.nv = m->n_vars; s.nc = m->n_cons;
    s.cons = (con_t *)calloc((size_t)(s.nc ? s.nc : 1), sizeof(con_t));
    s.links = (ivec *)calloc((size_t)(s.nv ? s.nv : 1), sizeof(ivec));
    s.dom0 = (dom_t *)calloc((size_t)(s.nv ? s.nv : 1), sizeof(dom_t));
    s.cur = (dom_t *)calloc((size_t)(s.nv ? s.nv : 1), sizeof(dom_t));
    s.inst = (int *)calloc((size_t)(s.nv ? s.nv : 1), sizeof(int));
    s.order = (int *)calloc((size_t)(s.nv ? s.nv : 1), sizeof(int));
    s.frames = (frame_t *)calloc((size_t)s.nv + 1, sizeof(frame_t));
    for (int i = 0; i < s.nv; i++) {
        s.dom0[i].type = m->dom_type[i];
        for (int j = m->dom_off[i]; j < m->dom_off[i + 1]; j++) iv_push(&s.dom0[i].vals, m->dom_vals[j]);
    }
    for (int c = 0; c < s.nc; c++) {
        s.cons[c].kind = m->con_kind[c];
        s.cons[c].data = m->con_data + m->con_off[c];
        s.cons[c].n = m->con_off[c + 1] - m->con_off[c];
    }
    link_vars(&s);
    reset_assignment(&s);
    if (m->assign_order)   /* a caller-edited Assignment::assign_order (public field, dequan.h:316) */
        for (int i = 0; i < s.nv; i++) s.order[i] = m->assign_order[i];
    s.count_all = o->mode == DQ_MODE_COUNT_ALL;
    s.budget = o->node_budget;
    s.first = first;
    s.split_depth = o->split_depth > 0 && o->split_depth < s.nv ? o->split_depth : 0;
    s.part_rank = s.split_depth ? o->part_rank : 0;
    s.part_count = s.split_depth ? o->part_count : 1;
    s.upto_key = o->upto_key;
    s.first_key = UINT64_MAX;
    if (order_out) for (int i = 0; i < s.nv; i++) order_out[i] = s.order[i];

    int ok = fc_step(&s);
    if (!s.count_all) {
        for (int i = 0; i < s.nv; i++) first[i] = ok ? s.inst[i] : UNASSIGNED;
        s.solutions = ok ? 1 : 0;
        s.first_key = ok ? s.cur_prefix : UINT64_MAX;
    } else if (!s.have_first) {
        for (int i = 0; i < s.nv; i++) first[i] = UNASSIGNED;
    }
    res->outcome = s.busted ? DQ_BUDGET : (s.solutions ? DQ_SAT : DQ_UNSAT);
    res->solutions = s.solutions; res->nodes = s.nodes;
    res->validated_constraints = s.validated; res->applied_arcs = s.applied;
    res->first_key = s.first_key; res->n_prefixes = s.prefix_counter;

    for (int i = 0; i < s.nv; i++) { free(s.dom0[i].vals.v); free(s.cur[i].vals.v); free(s.links[i].v); }
    for (int i = 0; i <= s.nv; i++) { for (int j = 0; j < s.frames[i].cap; j++) free(s.frames[i].e[j].saved.vals.v); free(s.frames[i].e); }
    free(s.cons); free(s.links); free(s.dom0); free(s.cur); free(s.inst); free(s.order); free(s.frames);
    return 0;
}

int dqo_solve(const dq_model_desc *m, const dqo_opts *o, dqo_result *res,
              int32_t *first /* [n_vars] */, int32_t *order_out /* [n_vars] or NULL */) {
    return dqo_run(m, o, res, first, order_out, NULL, 0);
}

/* Every solution in visiting order: the harness's Counting constraint (oracle/ref_driver.cpp, SURVEY.md par. 8c)
 * snapshotting Assignment::inst_vars on each hit.  out[i * n_vars + v]; at most `cap` are kept, res->solutions
 * counts them all. */
int dqo_enumerate(const dq_model_desc *m, dqo_result *res, int32_t *out /* [cap][n_vars] */, uint64_t cap) {
    dqo_opts o;
    memset(&o, 0, sizeof o);
    o.mode = DQ_MODE_COUNT_ALL; o.part_count = 1; o.upto_key = UINT64_MAX;
    int32_t *first = (int32_t *)calloc((size_t)(m->n_vars ? m->n_vars : 1), sizeof(int32_t));
    int rc = dqo_run(m, &o, res, first, NULL, out, cap);
    free(first);
    return rc;
}

const char *dqo_version(void) { return "dq_oracle 1 (restatement of nsweb/dequan dequan.h)"; }
