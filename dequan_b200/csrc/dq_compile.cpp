// dq_compile.cpp — host model compiler: dq_model_desc -> CompiledModel (see dq_model.hpp).
//
// Replaces CSP::FinalizeModel + Assignment::Reset (reference dequan.h:484-492, 365-395): the
// linked-constraint lists and per-constraint virtual AplyArcConsistency calls of the reference
// become, per ordered variable pair (x -> q), at most a few mask operations.
#include "dq_model.hpp"

#include <algorithm>
#include <map>
#include <set>

namespace dq {
namespace {

struct PairOp {
    EntryKind kind;
    std::vector<Mask> m;      // one mask per value index of x
    bool first = false;       // K_AND that erases only the first present position of m (duplicate values, ENT_FIRST)
};

// positions of q's value list that hold value t
Mask positions_of(const std::vector<int32_t>& qvals, int64_t t) {
    Mask m = 0;
    for (size_t j = 0; j < qvals.size(); j++) if ((int64_t)qvals[j] == t) m |= Mask(1) << j;
    return m;
}

// How assigning x = a filters q through one OpConstraint-style test "y (op) t"
// (DoCheck, dequan.h:636-669): returns the mask over q's value list.
Mask op_mask(const std::vector<int32_t>& qvals, int op, int64_t t) {
    Mask m = 0;
    for (size_t j = 0; j < qvals.size(); j++) {
        int64_t y = qvals[j];
        bool keep = false;
        switch (op) {
            case DQ_OP_EQUAL:    keep = (y == t); break;      // Intersect(t)      (weak, see K_WEQ)
            case DQ_OP_NOTEQUAL: keep = (y != t); break;      // Exclude(t)
            case DQ_OP_SUPEQUAL: keep = (y >= t); break;      // ExcludeInf(t)
            case DQ_OP_SUP:      keep = (y >= t + 1); break;  // ExcludeInf(t+1)
            case DQ_OP_INFEQUAL: keep = (y < t + 1); break;   // ExcludeSup(t+1)
            case DQ_OP_INF:      keep = (y < t); break;       // ExcludeSup(t)
        }
        if (keep) m |= Mask(1) << j;
    }
    return m;
}

// Same mask in O(1) when q's value list is one ascending run minv, minv+1, ... (every Ranges domain with a single
// range — AddIntVar(min, max) — which is what the BASELINE models use).
inline Mask low_bits(int64_t n, int k) { const int64_t c = n <= 0 ? 0 : (n >= k ? k : n); return c >= 64 ? ~Mask(0) : (Mask(1) << c) - 1; }
Mask op_mask_run(int64_t minv, int k, int op, int64_t t) {
    const Mask full = low_bits(k, k);
    const int64_t i = t - minv;                                   // index of value t
    switch (op) {
        case DQ_OP_EQUAL:    return (i >= 0 && i < k) ? Mask(1) << i : Mask(0);
        case DQ_OP_NOTEQUAL: return (i >= 0 && i < k) ? full & ~(Mask(1) << i) : full;
        case DQ_OP_SUPEQUAL: return full & ~low_bits(i, k);       // y >= t
        case DQ_OP_SUP:      return full & ~low_bits(i + 1, k);   // y >= t + 1
        case DQ_OP_INFEQUAL: return low_bits(i + 1, k);           // y <  t + 1
        case DQ_OP_INF:      return low_bits(i, k);               // y <  t
    }
    return 0;
}

int reverse_op(int op) {  // dequan.h:681-690
    switch (op) {
        case DQ_OP_SUPEQUAL: return DQ_OP_INFEQUAL;
        case DQ_OP_SUP:      return DQ_OP_INF;
        case DQ_OP_INFEQUAL: return DQ_OP_SUPEQUAL;
        case DQ_OP_INF:      return DQ_OP_SUP;
        default:             return op;
    }
}

}  // namespace

int compile_model(const dq_model_desc* d, CompiledModel& M, std::string& err) {
    if (!d || d->n_vars < 0 || d->n_cons < 0) { err = "null or negative-sized descriptor"; return DQ_ERR_INVALID; }
    const int nv = d->n_vars;
    if (nv > kMaxVars) { err = "more than 1022 variables"; return DQ_ERR_UNSUPPORTED; }
    M = CompiledModel();
    M.nv = nv;
    M.values.resize(nv);
    M.dom0.resize(nv);

    // ---- domains: expand to iteration-ordered value lists (dequan.h:544-563) ----
    for (int v = 0; v < nv; v++) {
        int lo = d->dom_off[v], hi = d->dom_off[v + 1];
        if (hi < lo) { err = "dom_off not monotone"; return DQ_ERR_INVALID; }
        std::vector<int32_t>& vals = M.values[v];
        if (d->dom_type[v] == DQ_DOM_VALUES) {
            vals.assign(d->dom_vals + lo, d->dom_vals + hi);     // (may list a value more than once: SURVEY.md Q2, see has_dup)
        } else if (d->dom_type[v] == DQ_DOM_RANGES) {
            if ((hi - lo) % 2) { err = "odd-length Ranges domain"; return DQ_ERR_INVALID; }
            int64_t prev_max = INT64_MIN;
            for (int r = lo; r < hi; r += 2) {
                int64_t a = d->dom_vals[r], b = d->dom_vals[r + 1];
                if (a < prev_max) { err = "Ranges domain not ascending/disjoint"; return DQ_ERR_UNSUPPORTED; }
                prev_max = b > a ? b : a;
                if (b - a > kMaxDom) { err = "domain larger than 64 values"; return DQ_ERR_UNSUPPORTED; }
                for (int64_t x = a; x < b; x++) vals.push_back((int32_t)x);
                if ((int)vals.size() > kMaxDom) { err = "domain larger than 64 values"; return DQ_ERR_UNSUPPORTED; }
            }
        } else { err = "bad domain type"; return DQ_ERR_INVALID; }
        if ((int)vals.size() > kMaxDom) { err = "domain larger than 64 values"; return DQ_ERR_UNSUPPORTED; }
        M.dom0[v] = low_bits((int64_t)vals.size(), (int)vals.size());
        M.kmax = std::max(M.kmax, (int)vals.size());
    }

    std::vector<char> is_run(nv, 0);                      // value list is minv, minv+1, ...
    for (int v = 0; v < nv; v++) {
        const std::vector<int32_t>& vals = M.values[v];
        bool run = !vals.empty();
        for (size_t j = 1; j < vals.size() && run; j++) run = (int64_t)vals[j] == (int64_t)vals[j - 1] + 1;
        is_run[v] = run;
    }
    // Values domains that list a value twice: iteration visits both copies, Exclude erases the first one only
    std::vector<char> has_dup(nv, 0);
    for (int v = 0; v < nv; v++) {
        std::set<int32_t> uniq(M.values[v].begin(), M.values[v].end());
        has_dup[v] = uniq.size() != M.values[v].size();
    }
    auto mask_of = [&](int q, int op, int64_t t) -> Mask {
        return is_run[q] ? op_mask_run(M.values[q][0], (int)M.values[q].size(), op, t) : op_mask(M.values[q], op, t);
    };

    // ---- static order: (initial size asc, id asc), Assignment::Reset dequan.h:384-394 ----
    M.order.resize(nv);
    for (int v = 0; v < nv; v++) M.order[v] = v;
    std::stable_sort(M.order.begin(), M.order.end(), [&](int a, int b) {
        return M.values[a].size() < M.values[b].size();
    });
    if (d->assign_order) {                                // caller-supplied Assignment::assign_order (dequan.h:316)
        std::vector<char> seen(nv, 0);
        for (int p = 0; p < nv; p++) {
            const int v = d->assign_order[p];
            if (v < 0 || v >= nv || seen[v]) { err = "assign_order is not a permutation of the variable ids"; return DQ_ERR_INVALID; }
            seen[v] = 1;
            M.order[p] = v;
        }
        M.caller_order = true;
    }
    M.pos_of.resize(nv);
    for (int p = 0; p < nv; p++) M.pos_of[M.order[p]] = p;
    {
        std::set<int32_t> sz;
        for (int v = 0; v < nv; v++) sz.insert((int32_t)M.values[v].size());
        M.distinct_sizes.assign(sz.begin(), sz.end());
    }

    // ---- link lists in FinalizeModel order (dequan.h:488-491 + each LinkVars) ----
    struct Con { int kind; const int32_t* data; int n; };
    std::vector<Con> cons(d->n_cons);
    std::vector<std::vector<int>> links(nv);
    {   // size the link lists once
        std::vector<int> deg(nv, 0);
        for (int c = 0; c < d->n_cons; c++) {
            const int32_t* p = d->con_data + d->con_off[c];
            const int cnt = d->con_kind[c] == DQ_CON_ALLDIFF ? d->con_off[c + 1] - d->con_off[c] : std::min(2, d->con_off[c + 1] - d->con_off[c]);
            for (int i = 0; i < cnt; i++) if (p[i] >= 0 && p[i] < nv) deg[p[i]]++;
        }
        for (int v = 0; v < nv; v++) links[v].reserve(deg[v]);
    }
    for (int c = 0; c < d->n_cons; c++) {
        cons[c] = {d->con_kind[c], d->con_data + d->con_off[c], d->con_off[c + 1] - d->con_off[c]};
        const Con& k = cons[c];
        auto chk = [&](int v) { return v >= 0 && v < nv; };
        switch (k.kind) {
            case DQ_CON_OP:      if (k.n != 4) { err = "OP payload"; return DQ_ERR_INVALID; } break;
            case DQ_CON_EQ:      if (k.n != 2) { err = "EQ payload"; return DQ_ERR_INVALID; } break;
            case DQ_CON_ORRANGE: if (k.n != 4) { err = "ORRANGE payload"; return DQ_ERR_INVALID; } break;
            case DQ_CON_TABLE:   if (k.n < 2 || (k.n % 2)) { err = "TABLE payload"; return DQ_ERR_INVALID; } break;
            case DQ_CON_FILTER:
                if (k.n < 5 || k.data[2] < 0 || k.data[3] < 0 || k.data[4] < 0 ||
                    (long long)k.n != 5 + 2 * ((long long)k.data[2] + k.data[3] + k.data[4])) { err = "FILTER payload"; return DQ_ERR_INVALID; }
                break;
            case DQ_CON_ALLDIFF: break;
            default: err = "constraint kind outside the engine's scope (ternary+ constraints are not lowered)"; return DQ_ERR_UNSUPPORTED;
        }
        if (k.kind == DQ_CON_ALLDIFF) {
            std::set<int> seen;
            for (int i = 0; i < k.n; i++) {
                if (!chk(k.data[i])) { err = "variable id out of range"; return DQ_ERR_INVALID; }
                if (!seen.insert(k.data[i]).second) { err = "AllDifferent with a repeated variable"; return DQ_ERR_UNSUPPORTED; }
                links[k.data[i]].push_back(c);
            }
        } else {
            if (!chk(k.data[0]) || !chk(k.data[1])) { err = "variable id out of range"; return DQ_ERR_INVALID; }
            if (k.data[0] == k.data[1]) { err = "constraint with v0 == v1"; return DQ_ERR_UNSUPPORTED; }
            if (k.kind == DQ_CON_OP && (k.data[2] < 0 || k.data[2] > 5)) { err = "bad op"; return DQ_ERR_INVALID; }
            links[k.data[0]].push_back(c);
            links[k.data[1]].push_back(c);
        }
    }

    // ---- per ordered pair (x -> q): the sequence of filters in x's link order ----
    M.ent_off.assign(nv + 1, 0);
    int forced_total = 0;
    // small-model tables (filled while the pairs are normalised below; dropped if some pair does not fit the pattern)
    bool small_try = nv >= 1 && nv <= 32 && M.kmax <= 32 && (size_t)nv * M.kmax * 32 * 4 * 3 + 40 * 1024 <= 200 * 1024;   // three tables + four warps of frames fit one CTA
    for (int v = 0; v < nv; v++) if (has_dup[v]) small_try = false;      // (first-match Exclude / one-copy Intersect: warp engine only)
    if (small_try) {
        M.small_and.assign((size_t)nv * M.kmax * 32, 0xFFFFFFFFu);
        M.small_weq_on.assign((size_t)nv * M.kmax, 0u);       // the WEQ / CHK tables are created when the first such op shows up
    }
    std::vector<int> qorder_buf;
    std::vector<std::vector<PairOp>> ops_buf(nv);
    std::vector<size_t> op_count(nv, 0);
    std::vector<std::vector<PairOp>> passes_buf;
    std::vector<std::vector<int>> pass_q_buf;
    for (int x = 0; x < nv; x++) {
        const std::vector<int32_t>& xv = M.values[x];
        const int kx = (int)xv.size();
        std::vector<int>& qorder = qorder_buf;         // neighbours in first-touch order
        std::vector<std::vector<PairOp>>& ops = ops_buf;
        for (int q : qorder) ops[q].clear();           // left over from the previous x
        qorder.clear();
        auto push = [&](int q, EntryKind kind, std::vector<Mask>&& m, bool first = false) {
            if (ops[q].empty()) qorder.push_back(q);
            if (first) { ops[q].push_back(PairOp{kind, std::move(m), true}); return; }
            // consecutive AND filters on the same pair compose into one (the normalisation below would do it anyway)
            if (kind == K_AND && !ops[q].empty() && ops[q].back().kind == K_AND && !ops[q].back().first) {
                std::vector<Mask>& acc = ops[q].back().m;
                for (int b = 0; b < kx; b++) acc[b] &= m[b];
                return;
            }
            ops[q].push_back(PairOp{kind, std::move(m)});
        };
        for (int c : links[x]) {
            const Con& k = cons[c];
            if (k.kind == DQ_CON_OP || k.kind == DQ_CON_EQ) {
                const bool x_is_v0 = (k.data[0] == x);
                const int q = x_is_v0 ? k.data[1] : k.data[0];
                int op = k.kind == DQ_CON_EQ ? DQ_OP_EQUAL : k.data[2];
                const int64_t off = k.kind == DQ_CON_EQ ? 0 : k.data[3];
                // x==v0 assigned -> q=v1 filtered with reversed op against a-off; x==v1 -> q=v0 with op against a+off
                if (x_is_v0) op = reverse_op(op);
                const EntryKind kind = op == DQ_OP_EQUAL ? K_WEQ : K_AND;
                auto mask_at = [&](int b) {
                    const int64_t t = x_is_v0 ? (int64_t)xv[b] - off : (int64_t)xv[b] + off;
                    return mask_of(q, op, t);
                };
                if (op == DQ_OP_NOTEQUAL && has_dup[q]) {                  // Exclude(t) on a list with duplicates: the first match only
                    std::vector<Mask> m(kx);
                    for (int b = 0; b < kx; b++) m[b] = positions_of(M.values[q], x_is_v0 ? (int64_t)xv[b] - off : (int64_t)xv[b] + off);
                    std::vector<Mask> again = m;                             // the copies that stay are still visited, and fail Evaluate
                    push(q, K_AND, std::move(m), true);
                    push(q, K_CHK, std::move(again));
                } else if (kind == K_AND && !ops[q].empty() && ops[q].back().kind == K_AND && !ops[q].back().first) {
                    std::vector<Mask>& acc = ops[q].back().m;              // compose in place, no temporary
                    for (int b = 0; b < kx; b++) acc[b] &= mask_at(b);
                } else {
                    std::vector<Mask> m(kx);
                    for (int b = 0; b < kx; b++) m[b] = mask_at(b);
                    push(q, kind, std::move(m));
                }
            } else if (k.kind == DQ_CON_ALLDIFF) {
                for (int i = 0; i < k.n; i++) {        // AllDifferent::AplyArcConsistency, dequan.h:915-939
                    int q = k.data[i];
                    if (q == x) continue;
                    std::vector<Mask> m(kx);
                    if (has_dup[q]) {
                        for (int b = 0; b < kx; b++) m[b] = positions_of(M.values[q], xv[b]);
                        std::vector<Mask> again = m;
                        push(q, K_AND, std::move(m), true);
                        push(q, K_CHK, std::move(again));
                        continue;
                    }
                    for (int b = 0; b < kx; b++) m[b] = mask_of(q, DQ_OP_NOTEQUAL, xv[b]);
                    push(q, K_AND, std::move(m));
                }
            } else if (k.kind == DQ_CON_ORRANGE) {     // Evaluate only (dequan.h:844-854); filter compiled out (860-893)
                const bool x_is_v0 = (k.data[0] == x);
                const int q = x_is_v0 ? k.data[1] : k.data[0];
                const int lo = k.data[2], hi = k.data[3];
                Mask q_out = 0;
                for (size_t j = 0; j < M.values[q].size(); j++)
                    if (!(M.values[q][j] >= lo && M.values[q][j] < hi)) q_out |= Mask(1) << j;
                std::vector<Mask> m(kx);
                for (int b = 0; b < kx; b++) m[b] = (xv[b] >= lo && xv[b] < hi) ? 0u : q_out;
                push(q, K_CHK, std::move(m));
            } else if (k.kind == DQ_CON_TABLE) {
                const bool x_is_v0 = (k.data[0] == x);
                const int q = x_is_v0 ? k.data[1] : k.data[0];
                std::set<std::pair<int, int>> allowed;
                for (int i = 2; i + 1 < k.n; i += 2) allowed.insert({k.data[i], k.data[i + 1]});
                std::vector<Mask> m(kx);
                for (int b = 0; b < kx; b++) {
                    Mask bad = 0;
                    for (size_t j = 0; j < M.values[q].size(); j++) {
                        std::pair<int, int> pr = x_is_v0 ? std::make_pair((int)xv[b], (int)M.values[q][j])
                                                         : std::make_pair((int)M.values[q][j], (int)xv[b]);
                        if (!allowed.count(pr)) bad |= Mask(1) << j;
                    }
                    m[b] = bad;
                }
                push(q, K_CHK, std::move(m));
            } else if (k.kind == DQ_CON_FILTER) {
                // a user constraint with its own AplyArcConsistency: what assigning x leaves of q (a plain AND mask, in
                // link order with the other filters on the pair) + the values of q its Evaluate will reject later
                const bool x_is_v0 = (k.data[0] == x);
                const int q = x_is_v0 ? k.data[1] : k.data[0];
                const int n_allow = k.data[2], n01 = k.data[3], n10 = k.data[4];
                const int32_t* pr = k.data + 5;
                std::set<std::pair<int, int>> allowed, keep;
                for (int i = 0; i < n_allow; i++) allowed.insert({pr[2 * i], pr[2 * i + 1]});
                const int32_t* kp = pr + 2 * n_allow + (x_is_v0 ? 0 : 2 * n01);
                for (int i = 0; i < (x_is_v0 ? n01 : n10); i++) keep.insert({kp[2 * i], kp[2 * i + 1]});
                std::vector<Mask> ma(kx), mc(kx);
                for (int b = 0; b < kx; b++) {
                    Mask kept = 0, bad = 0;
                    for (size_t j = 0; j < M.values[q].size(); j++) {
                        std::pair<int, int> p2 = x_is_v0 ? std::make_pair((int)xv[b], (int)M.values[q][j])
                                                         : std::make_pair((int)M.values[q][j], (int)xv[b]);
                        if (keep.count(p2)) kept |= Mask(1) << j;
                        if (!allowed.count(p2)) bad |= Mask(1) << j;
                    }
                    ma[b] = kept;
                    mc[b] = bad;
                }
                push(q, K_AND, std::move(ma));
                push(q, K_CHK, std::move(mc));
            }
        }
        // normalise each pair: merge adjacent ANDs, gather all CHKs (they commute) at the end
        std::vector<std::vector<PairOp>>& passes = passes_buf;       // passes[p] = p-th op of every pair
        std::vector<std::vector<int>>& pass_q = pass_q_buf;
        for (auto& v : passes) v.clear();
        for (auto& v : pass_q) v.clear();
        int multi_pairs = 0;
        size_t n_pass = 0;                             // passes in use for this x (the buffers keep their length)
        for (int q : qorder) {
            std::vector<PairOp>& seq = ops[q];
            std::vector<PairOp> norm;
            PairOp chk{K_CHK, std::vector<Mask>(kx, Mask(0))};
            bool have_chk = false;
            for (PairOp& o : seq) {
                if (o.kind == K_CHK) { have_chk = true; for (int b = 0; b < kx; b++) chk.m[b] |= o.m[b]; }
                else if (o.kind == K_AND && !o.first && !norm.empty() && norm.back().kind == K_AND && !norm.back().first) { for (int b = 0; b < kx; b++) norm.back().m[b] &= o.m[b]; }
                else norm.push_back(std::move(o));
            }
            if (have_chk) norm.push_back(std::move(chk));
            // K_AND that is exactly "clear the same bit index" -> K_NE_SAME (no table needed)
            for (PairOp& o : norm) {
                if (o.kind != K_AND || o.first || M.values[q].size() != (size_t)kx) continue;
                bool same = true;
                for (int b = 0; b < kx && same; b++) same = (o.m[b] == (M.dom0[q] & ~(Mask(1) << b)));
                if (same) o.kind = K_NE_SAME;
            }
            if (norm.size() > 1) multi_pairs++;
            n_pass = std::max(n_pass, norm.size());
            for (const PairOp& o : norm) if (o.first) small_try = false;      // (the register engine's tables are plain AND masks)
            if (small_try) {
                size_t i = 0;
                const PairOp *pa = nullptr, *pw = nullptr, *pc = nullptr;
                if (i < norm.size() && (norm[i].kind == K_AND || norm[i].kind == K_NE_SAME)) pa = &norm[i++];
                if (i < norm.size() && norm[i].kind == K_WEQ) pw = &norm[i++];
                if (i < norm.size() && norm[i].kind == K_CHK) pc = &norm[i++];
                if (i != norm.size()) small_try = false;
                else {
                    const int px = M.pos_of[x], pq = M.pos_of[q];
                    if (pw && M.small_weq.empty()) M.small_weq.assign((size_t)nv * M.kmax * 32, 0u);
                    if (pc && M.small_chk.empty()) M.small_chk.assign((size_t)nv * M.kmax * 32, 0u);
                    for (int b = 0; b < kx; b++) {
                        const size_t at = ((size_t)px * M.kmax + b) * 32 + pq;
                        if (pa) M.small_and[at] = (uint32_t)pa->m[b];
                        if (pw) { M.small_weq[at] = (uint32_t)pw->m[b]; M.small_weq_on[(size_t)px * M.kmax + b] |= 1u << pq; }
                        if (pc) M.small_chk[at] = (uint32_t)pc->m[b];
                    }
                }
            }
            for (size_t p = 0; p < norm.size(); p++) {
                if (passes.size() <= p) { passes.resize(p + 1); pass_q.resize(p + 1); }
                passes[p].push_back(std::move(norm[p]));
                pass_q[p].push_back(q);
            }
            op_count[q] = norm.size();                 // for flagging below
        }
        forced_total += 2 * multi_pairs;
        for (size_t p = 0; p < n_pass; p++) {
            for (size_t i = 0; i < passes[p].size(); i++) {
                const PairOp& o = passes[p][i];
                const int q = pass_q[p][i];
                uint32_t w = (uint32_t)q | ((uint32_t)o.kind << ENT_KIND_SHIFT);
                const size_t cnt = op_count[q];
                if (cnt > 1) w |= (p == 0) ? (ENT_FORCE_D | ENT_FORCE_F) : (ENT_NOTRAIL_D | ENT_NOTRAIL_F);
                if (o.first) w |= ENT_FIRST;
                if (o.kind == K_WEQ || o.kind == K_CHK) M.has_f = true;
                if (o.kind != K_NE_SAME) {
                    M.has_table = true;
                    M.ent_moff.push_back((uint32_t)M.masks.size());
                    M.masks.insert(M.masks.end(), o.m.begin(), o.m.end());
                } else M.ent_moff.push_back(0);
                M.ent.push_back(w);
            }
            if (p + 1 < n_pass)                        // next pass must start on a 32-entry boundary
                while ((M.ent.size() - M.ent_off[x]) % 32) { M.ent.push_back(ENT_SKIP | ENT_Q_MASK); M.ent_moff.push_back(0); }
        }
        M.ent_off[x + 1] = (uint32_t)M.ent.size();
    }
    if (M.masks.empty()) M.masks.push_back(0);
    M.small_ok = small_try;
    if (!small_try) { M.small_and.clear(); M.small_weq.clear(); M.small_chk.clear(); M.small_weq_on.clear(); }
    else if (M.has_f) {                                   // the device kernel indexes both tables when the model has an F word
        if (M.small_weq.empty()) M.small_weq.assign((size_t)nv * M.kmax * 32, 0u);
        if (M.small_chk.empty()) M.small_chk.assign((size_t)nv * M.kmax * 32, 0u);
    }

    int ksum = 0;
    for (int v = 0; v < nv; v++) ksum += (int)M.values[v].size();
    M.trail_bound = ksum + (M.has_f ? ksum + nv : 0) + forced_total + 32;

    // ---- model class ----
    M.model_class = M.has_table ? CLASS_GENERIC : CLASS_NE_SAME;
    if (M.has_table && !M.has_f && nv >= 1 && nv <= 32) {
        bool queens = true;
        const uint32_t full = nv == 32 ? 0xFFFFFFFFu : ((1u << nv) - 1u);
        for (int v = 0; v < nv && queens; v++) {
            queens = (int)M.values[v].size() == nv;
            for (int b = 0; b < nv && queens; b++) queens = M.values[v][b] == b;
        }
        for (int x = 0; x < nv && queens; x++) {
            if ((int)(M.ent_off[x + 1] - M.ent_off[x]) != nv - 1) { queens = false; break; }
            std::set<int> qs;
            for (uint32_t e = M.ent_off[x]; e < M.ent_off[x + 1] && queens; e++) {
                const uint32_t w = M.ent[e];
                const int q = (int)(w & ENT_Q_MASK), dist = q > x ? q - x : x - q;
                if (((w >> ENT_KIND_SHIFT) & 3) != K_AND || (w & ENT_FLAGS) || !qs.insert(q).second) { queens = false; break; }
                for (int b = 0; b < nv; b++) {
                    uint32_t rm = 1u << b;
                    if (b + dist < nv) rm |= 1u << (b + dist);
                    if (b - dist >= 0) rm |= 1u << (b - dist);
                    if (M.masks[M.ent_moff[e] + b] != (full & ~rm)) { queens = false; break; }
                }
            }
        }
        // the class engine searches the variables in id order (all domains have N values: Reset's order is the identity);
        // a caller-supplied assign_order that differs from it changes node counts and the first solution: generic engine
        for (int p = 0; p < nv && queens; p++) queens = M.order[p] == p;
        if (queens && nv >= 2) { M.model_class = CLASS_QUEENS; M.queens_n = nv; }
    }
    // 9x9 Sudoku template: every variable on 1..9 (ascending), every arc a plain "different value", and the
    // neighbours of cell (r,c) exactly its row, column and box — whichever mix of binary NotEqual and
    // AllDifferent rows the user wrote (test/main-test.cpp:130-148 plus the boxes).
    if (M.model_class == CLASS_NE_SAME && nv == 81 && !d->assign_order) {
        bool sudoku = true;
        for (int v = 0; v < nv && sudoku; v++) {
            sudoku = M.values[v].size() == 9;
            for (int b = 0; b < 9 && sudoku; b++) sudoku = M.values[v][b] == b + 1;
        }
        for (int x = 0; x < nv && sudoku; x++) {
            std::set<int> want, got;
            const int r = x / 9, c = x % 9;
            for (int i = 0; i < 9; i++) {
                want.insert(r * 9 + i);
                want.insert(i * 9 + c);
                want.insert((r / 3 * 3 + i / 3) * 9 + (c / 3 * 3 + i % 3));
            }
            want.erase(x);
            for (uint32_t e = M.ent_off[x]; e < M.ent_off[x + 1]; e++)
                if (!(M.ent[e] & ENT_SKIP)) got.insert((int)(M.ent[e] & ENT_Q_MASK));
            sudoku = want == got;
        }
        if (sudoku) M.model_class = CLASS_SUDOKU9;
    }
    return DQ_OK;
}

}  // namespace dq
