// Filtering user constraints through the drop-in header (include/dequan.h): constraints that override
// AplyArcConsistency are lowered by TabulateUserConstraint to DQ_CON_FILTER rows.  tests/test_user_filters.py drives it.
//   user_filters refusals   three illegal filters; each lowering must throw dequan::b200::Error (no device needed)
//   user_filters            models whose filters keep more or fewer pairs than their Evaluate accepts, solved through
//                           ForwardCheckingStep and through b200::SolveAll; one JSON line per model and path, with the
//                           model's description so that the test can rebuild it as a FilterConstraint
#define DEQUAN_USE_STDVECTOR
#define DEQUAN_WITH_STATS
#define DEQUAN_SET_CONSTRAINT_SIZE 48              // TouchesThird holds a third variable id
#define DEQUAN_IMPLEMENTATION
#include "dequan.h"
#include <cstdio>
#include <string>
#include <vector>

using namespace dequan;

// The relations the test restates in Python (tests/test_user_filters.py REL): each is a function of (a, b) only.
static bool rel(int r, int a, int b, int g) {
    switch (r) {
        case 0: return a + g <= b;
        case 1: return a + g < b;                 // stronger than 0
        case 2: return a + g - 2 <= b;            // weaker than 0
        case 3: return (a + b + g) % 3 != 0;      // unrelated to 0
        case 4: return true;                      // keeps everything
        default: return a != b + g;
    }
}

// A binary user constraint: Evaluate accepts rel(ev); assigning x = a leaves the values b of y with rel(k01, a, b);
// assigning y = b leaves the values a of x with rel(k10, a, b).
struct RelConstraint : public Constraint {
    RelConstraint(VarId a, VarId b, int e, int f01, int f10, int gap) : x(a), y(b), ev(e), k01(f01), k10(f10), g(gap) {}
    virtual void LinkVars(Array<Var>& vars) {
        vars[x].linked_constraints.push_back(this);
        vars[y].linked_constraints.push_back(this);
    }
    virtual Eval Evaluate(const Array<InstVar>& iv, VarId) {
        if (iv[x].value == InstVar::UNASSIGNED || iv[y].value == InstVar::UNASSIGNED) return Eval::NA;
        return rel(ev, iv[x].value, iv[y].value, g) ? Eval::Passed : Eval::Failed;
    }
    static Array<int> values(const Domain& d) {
        Array<int> out;
        if (d.type == DomainType::Values) out = d.values;
        else
            for (size_t i = 0; i + 1 < d.values.size(); i += 2)
                for (int v = d.values[i]; v < d.values[i + 1]; v++) out.push_back(v);
        return out;
    }
    virtual bool AplyArcConsistency(Assignment& a, VarId) {
        const int xv = a.inst_vars[x].value, yv = a.inst_vars[y].value;
        if ((xv == InstVar::UNASSIGNED) == (yv == InstVar::UNASSIGNED)) return true;
        const bool from_x = xv != InstVar::UNASSIGNED;
        const VarId to = from_x ? y : x;
        Domain& d = a.current_domains[to];
        a.EnsureSavedDomain(to, d);
        const Array<int> vals = values(d);
        for (size_t i = 0; i < vals.size(); i++)
            if (!(from_x ? rel(k01, xv, vals[i], g) : rel(k10, vals[i], yv, g))) d.Exclude(vals[i]);
        return d.Size() > 0;
    }
    VarId x, y;
    int ev, k01, k10, g;
};

// ---- three illegal filters -------------------------------------------------------------------------------------------

struct TouchesThird : public RelConstraint {            // also empties a third variable's domain
    TouchesThird(VarId a, VarId b, VarId c) : RelConstraint(a, b, 0, 0, 0, 1), z(c) {}
    virtual bool AplyArcConsistency(Assignment& a, VarId v) {
        if (a.inst_vars[z].value == InstVar::UNASSIGNED) {
            a.EnsureSavedDomain(z, a.current_domains[z]);
            a.current_domains[z].Exclude(RelConstraint::values(a.current_domains[z])[0]);
        }
        return RelConstraint::AplyArcConsistency(a, v);
    }
    VarId z;
};

struct TrueWhenEmpty : public RelConstraint {           // answers true after a wipe-out
    TrueWhenEmpty(VarId a, VarId b) : RelConstraint(a, b, 0, 0, 0, 1) {}
    virtual bool AplyArcConsistency(Assignment& a, VarId v) {
        RelConstraint::AplyArcConsistency(a, v);
        return true;
    }
};

struct DependsOnOthers : public RelConstraint {         // keeps the largest value of the domain only
    DependsOnOthers(VarId a, VarId b) : RelConstraint(a, b, 0, 0, 0, 1) {}
    virtual bool AplyArcConsistency(Assignment& a, VarId) {
        const bool from_x = a.inst_vars[x].value != InstVar::UNASSIGNED;
        if (from_x == (a.inst_vars[y].value != InstVar::UNASSIGNED)) return true;
        const VarId to = from_x ? y : x;
        Domain& d = a.current_domains[to];
        a.EnsureSavedDomain(to, d);
        const Array<int> vals = RelConstraint::values(d);
        int top = vals[0];
        for (size_t i = 1; i < vals.size(); i++) top = vals[i] > top ? vals[i] : top;
        for (size_t i = 0; i < vals.size(); i++)
            if (vals[i] != top) d.Exclude(vals[i]);
        return d.Size() > 0;
    }
};

template <class C, class... Args>
static void refusal(const char* name, Args... args) {
    CSP csp;
    for (int i = 0; i < 3; i++) csp.AddIntVar(0, 5);
    csp.AddConstraint(C(args...));
    csp.FinalizeModel();
    Assignment a;
    a.Reset(csp);
    try {
        csp.ForwardCheckingStep(a);
        std::printf("{\"name\":\"%s\",\"thrown\":false}\n", name);
    } catch (const b200::Error& e) {
        std::printf("{\"name\":\"%s\",\"thrown\":true,\"what\":\"%s\"}\n", name, e.what());
    }
}

// ---- models that solve ----------------------------------------------------------------------------------------------

struct Rel { int x, y, ev, k01, k10, g; };

struct Spec {
    std::string name;
    std::vector<Domain> doms;
    std::vector<Rel> rels;
    bool alldiff;                                       // an AllDifferent over every variable, linked after the relations
};

static Domain values_dom(std::vector<int> v) { return Domain(DomainType::Values, Array<int>(v.begin(), v.end())); }
static Domain range_dom(int lo, int hi) { int r[] = {lo, hi}; return Domain(DomainType::Ranges, Array<int>(r, r + 2)); }

static std::vector<Spec> specs() {
    std::vector<Spec> out;
    // chains in the style of dropin_scenarios.cpp user_filter, each with one pair of filter classes
    const int classes[][3] = {{0, 1, 0}, {0, 0, 1}, {0, 2, 2}, {0, 1, 2}, {0, 4, 4}, {3, 4, 1}, {3, 0, 0}, {5, 4, 5}, {5, 1, 2}};
    for (int c = 0; c < 9; c++)
        for (int rev = 0; rev < 2; rev++) {
            Spec s;
            s.name = "chain" + std::to_string(c) + (rev ? "_rev" : "");
            const int n = 5 + c % 2;
            for (int i = 0; i < n; i++) {
                if (i % 2 == 0) s.doms.push_back(range_dom(0, n + 3));
                else {
                    std::vector<int> v;
                    for (int k = 0; k < n + 3; k++) v.push_back(rev ? n + 2 - k : k);
                    s.doms.push_back(values_dom(v));
                }
            }
            for (int i = 0; i + 1 < n; i++) s.rels.push_back({i, i + 1, classes[c][0], classes[c][1], classes[c][2], i % 2 ? c % 3 : 1});
            s.alldiff = c % 3 != 2;
            out.push_back(s);
        }
    // denser: every pair of four variables on shuffled values, filters that wipe a domain out on some values
    for (int c = 0; c < 4; c++) {
        Spec s;
        s.name = "dense" + std::to_string(c);
        s.doms = {values_dom({3, 0, 5, 1, 4}), range_dom(-1, 4), values_dom({2, 6, -1, 0}), range_dom(0, 6)};
        for (int i = 0; i < 4; i++)
            for (int j = i + 1; j < 4; j++) s.rels.push_back({i, j, (i + j + c) % 6 == 4 ? 5 : (i + j + c) % 6, (i * 3 + c) % 6, (j + 2 * c) % 6, c - 1});
        s.alldiff = c % 2 == 0;
        out.push_back(s);
    }
    return out;
}

static CSP* build(const Spec& s) {
    CSP* csp = new CSP();
    for (const Domain& d : s.doms) csp->AddIntVar(d);
    for (const Rel& r : s.rels) csp->AddConstraint(RelConstraint(r.x, r.y, r.ev, r.k01, r.k10, r.g));
    if (s.alldiff) {
        Array<VarId> all;
        for (size_t v = 0; v < s.doms.size(); v++) all.push_back((VarId)v);
        csp->AddConstraint(AllDifferentConstraint(all));
    }
    csp->FinalizeModel();
    return csp;
}

static void print_ints(const Array<int>& v) {
    std::printf("[");
    for (size_t i = 0; i < v.size(); i++) std::printf("%s%d", i ? "," : "", v[i]);
    std::printf("]");
}

static void report(const char* path, const Spec& s, bool ok, const Assignment& a) {
    std::printf("{\"path\":\"%s\",\"name\":\"%s\",\"ok\":%s,\"assigned_vars\":%llu,\"values\":[", path, s.name.c_str(),
                ok ? "true" : "false", a.stats.assigned_vars);
    for (size_t v = 0; v < a.inst_vars.size(); v++) std::printf("%s%d", v ? "," : "", a.GetInstVarValue((VarId)v));
    std::printf("],\"assign_order\":");
    print_ints(a.assign_order);
    std::printf(",\"domains\":[");
    for (size_t v = 0; v < s.doms.size(); v++) {
        std::printf("%s{\"t\":%d,\"v\":", v ? "," : "", (int)s.doms[v].type);
        print_ints(s.doms[v].values);
        std::printf("}");
    }
    std::printf("],\"rels\":[");
    for (size_t i = 0; i < s.rels.size(); i++) {
        const Rel& r = s.rels[i];
        std::printf("%s[%d,%d,%d,%d,%d,%d]", i ? "," : "", r.x, r.y, r.ev, r.k01, r.k10, r.g);
    }
    std::printf("],\"alldiff\":%s}\n", s.alldiff ? "true" : "false");
}

int main(int argc, char** argv) {
    if (argc > 1 && std::string(argv[1]) == "refusals") {
        refusal<TouchesThird>("touches_third", 0, 1, 2);
        refusal<TrueWhenEmpty>("true_when_empty", 0, 1);
        refusal<DependsOnOthers>("depends_on_others", 0, 1);
        return 0;
    }
    const std::vector<Spec> all = specs();
    std::vector<const CSP*> csps;
    std::vector<Assignment*> as;
    for (const Spec& s : all) {
        CSP* csp = build(s);
        Assignment a;
        a.Reset(*csp);
        report("step", s, csp->ForwardCheckingStep(a), a);
        csps.push_back(csp);
        as.push_back(new Assignment());
        as.back()->Reset(*csp);
    }
    const std::vector<bool> ok = b200::SolveAll(csps, as);
    for (size_t i = 0; i < all.size(); i++) report("all", all[i], ok[i], *as[i]);
    for (size_t i = 0; i < all.size(); i++) { delete as[i]; delete csps[i]; }
    return 0;
}
