/*
 * tests/oracle_count_limit.c — TEST INFRASTRUCTURE, NOT PRODUCT.
 *
 * The CPU oracle's search with a solution limit, for tests/test_count_batches.py.  It includes oracle/dq_oracle.c
 * unchanged, so domains, constraints, filters, the trail and Assignment::Reset are the oracle's own; only the search
 * loop is restated here, with the harness's Counting constraint (SURVEY.md §8c) passing the limit-th solution
 * instead of failing it, so that ForwardCheckingStep returns true there.  The Budget constraint is evaluated before
 * it on every AssignVar, as in dqo_solve.  One search at a time (the limit is a file-level variable).
 */
#include "../oracle/dq_oracle.c"

static uint64_t g_limit;                 /* 0 = count every solution */

/* validate() in COUNT_ALL mode, the Counting constraint returning Passed on the limit-th solution */
static int lim_validate(search_t *s, int vid) {
    if (s->budget) {
        s->validated++;
        if (++s->evals > s->budget) { s->busted = 1; return 0; }
    }
    const ivec *l = &s->links[vid];
    for (int i = 0; i < l->n; i++) {
        s->validated++;
        if (evaluate(s, &s->cons[l->v[i]], vid) == EV_FAILED) return 0;
    }
    if (vid == s->order[s->nv - 1]) {
        s->validated++;
        if (!s->have_first) { for (int i = 0; i < s->nv; i++) s->first[i] = s->inst[i]; s->have_first = 1; }
        s->solutions++;
        return g_limit && s->solutions >= g_limit;
    }
    return 1;
}

static int lim_fc_step(search_t *s);

/* try_value() without the partition emulation */
static int lim_try_value(search_t *s, int vid, int val) {
    s->inst[vid] = val; s->assigned++;
    s->nodes++;
    if (lim_validate(s, vid)) {
        int ok = 1;
        const ivec *l = &s->links[vid];
        for (int i = 0; ok && i < l->n; i++) ok &= apply_arc(s, &s->cons[l->v[i]], vid);
        if (ok) ok = lim_fc_step(s);
        if (ok) return 1;
        s->inst[vid] = UNASSIGNED; s->assigned--;
        restore_step(s);
    } else {
        s->inst[vid] = UNASSIGNED; s->assigned--;
    }
    return 0;
}

static int lim_fc_step(search_t *s) {
    if (s->assigned == s->nv) return 1;
    frame_t *f = &s->frames[s->nframes++];
    f->n = 0;
    int vid = s->order[s->assigned];
    const dom_t *dm = &s->cur[vid];
    int found = 0;
    if (dm->type == DQ_DOM_VALUES) {
        for (int i = 0; i < dm->vals.n && !found && !s->busted; i++) found = lim_try_value(s, vid, dm->vals.v[i]);
    } else {
        for (int r = 0; r < dm->vals.n; r += 2) {
            int lo = dm->vals.v[r], hi = dm->vals.v[r + 1];
            for (int v = lo; v < hi && !found && !s->busted; v++) found = lim_try_value(s, vid, v);
        }
    }
    if (found) return 1;
    s->nframes--;
    return 0;
}

/* res->outcome: DQ_BUDGET if the budget ran out first, else DQ_SAT iff a solution was counted; res->solutions =
 * min(total, limit) or the solutions counted before the budget ran out; res->nodes = AssignVar calls up to the node
 * the search stopped at; first = the DFS-first solution whenever one was counted (UNASSIGNED otherwise). */
int dqo_count_limit(const dq_model_desc *m, uint64_t node_budget, uint64_t limit, dqo_result *res,
                    int32_t *first /* [n_vars] */) {
    search_t s;
    memset(&s, 0, sizeof s);
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
    if (m->assign_order)
        for (int i = 0; i < s.nv; i++) s.order[i] = m->assign_order[i];
    s.count_all = 1;
    s.budget = node_budget;
    s.first = first;
    g_limit = limit;
    lim_fc_step(&s);
    if (!s.have_first) for (int i = 0; i < s.nv; i++) first[i] = UNASSIGNED;
    memset(res, 0, sizeof *res);
    res->outcome = s.busted ? DQ_BUDGET : (s.solutions ? DQ_SAT : DQ_UNSAT);
    res->solutions = s.solutions; res->nodes = s.nodes;
    res->validated_constraints = s.validated; res->applied_arcs = s.applied;
    res->first_key = UINT64_MAX;

    for (int i = 0; i < s.nv; i++) { free(s.dom0[i].vals.v); free(s.cur[i].vals.v); free(s.links[i].v); }
    for (int i = 0; i <= s.nv; i++) { for (int j = 0; j < s.frames[i].cap; j++) free(s.frames[i].e[j].saved.vals.v); free(s.frames[i].e); }
    free(s.cons); free(s.links); free(s.dom0); free(s.cur); free(s.inst); free(s.order); free(s.frames);
    return 0;
}
