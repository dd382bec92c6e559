// dequan::b200::SolveAll (no counterpart in the reference): many (CSP, Assignment) pairs in one device call.  Every pair is
// solved once through SolveAll and once, on a copy of its Assignment, through ForwardCheckingStep; one JSON line per pair
// and path with the outcome and the whole post-solve Assignment.  tests/test_solve_models.py requires the two paths'
// lines to be identical.
#define DEQUAN_USE_STDVECTOR
#define DEQUAN_WITH_STATS
#define DEQUAN_IMPLEMENTATION
#include "dequan.h"
#include <cstdio>
#include <string>
#include <vector>

using namespace dequan;

static void print_ints(const Array<int>& v) {
    std::printf("[");
    for (size_t i = 0; i < v.size(); i++) std::printf("%s%d", i ? "," : "", v[i]);
    std::printf("]");
}

static void report(const char* path, const std::string& name, bool ok, const Assignment& a) {
    std::printf("{\"path\":\"%s\",\"name\":\"%s\",\"ok\":%s,\"assigned_vars\":%llu,\"assigned_var_count\":%d,\"values\":[", path,
                name.c_str(), ok ? "true" : "false", a.stats.assigned_vars, a.assigned_var_count);
    for (size_t v = 0; v < a.inst_vars.size(); v++) std::printf("%s%d", v ? "," : "", a.GetInstVarValue((VarId)v));
    std::printf("],\"current_domains\":[");
    for (size_t v = 0; v < a.current_domains.size(); v++) {
        std::printf("%s{\"t\":%d,\"v\":", v ? "," : "", (int)a.current_domains[v].type);
        print_ints(a.current_domains[v].values);
        std::printf("}");
    }
    std::printf("],\"saved_domains\":[");
    for (size_t d = 0; d < a.saved_domains.size(); d++) {
        std::printf("%s[", d ? "," : "");
        const Array<SavedDomain>& f = a.saved_domains[d].domains;
        for (size_t i = 0; i < f.size(); i++) {
            std::printf("%s{\"id\":%d,\"t\":%d,\"v\":", i ? "," : "", f[i].var_id, (int)f[i].type);
            print_ints(f[i].values);
            std::printf("}");
        }
        std::printf("]");
    }
    std::printf("]}\n");
}

static CSP* queens(int n) {                                  // test/main-test.cpp:36-49
    CSP* csp = new CSP();
    for (int i = 0; i < n; i++) csp->AddIntVar(0, n);
    for (int i = 0; i < n; i++)
        for (int j = i + 1; j < n; j++) {
            csp->AddConstraint(OpConstraint(i, j, OpConstraint::Op::NotEqual, 0));
            csp->AddConstraint(OpConstraint(i, j, OpConstraint::Op::NotEqual, j - i));
            csp->AddConstraint(OpConstraint(i, j, OpConstraint::Op::NotEqual, i - j));
        }
    csp->FinalizeModel();
    return csp;
}

static const int kGrid[81] = {   // test/main-test.cpp:92-105
    0, 0, 3, 0, 2, 0, 6, 0, 0, 9, 0, 0, 3, 0, 5, 0, 0, 1, 0, 0, 1, 8, 0, 6, 4, 0, 0,
    0, 0, 8, 1, 0, 2, 9, 0, 0, 7, 0, 0, 0, 0, 0, 0, 0, 8, 0, 0, 6, 7, 0, 8, 2, 0, 0,
    0, 0, 2, 6, 0, 9, 5, 0, 0, 8, 0, 0, 2, 0, 3, 0, 0, 9, 0, 0, 5, 0, 1, 0, 3, 0, 0};

static CSP* sudoku_rows_cols() {                             // test/main-test.cpp:88-185: 1 336 467 nodes
    CSP* csp = new CSP();
    Array<VarId> cell(81);
    for (int i = 0; i < 81; i++) cell[i] = kGrid[i] ? csp->AddFixedVar(kGrid[i]) : csp->AddIntVar(1, 10);
    for (int r = 0; r < 9; r++) { Array<VarId> g; for (int c = 0; c < 9; c++) g.push_back(cell[r * 9 + c]); csp->AddConstraint(AllDifferentConstraint(g)); }
    for (int c = 0; c < 9; c++) { Array<VarId> g; for (int r = 0; r < 9; r++) g.push_back(cell[r * 9 + c]); csp->AddConstraint(AllDifferentConstraint(g)); }
    csp->FinalizeModel();
    return csp;
}

static CSP* op_inequality() {                                // test/main-test.cpp:187-233
    CSP* csp = new CSP();
    VarId v0 = csp->AddIntVar(0, 10), v1 = csp->AddIntVar(0, 10), v2 = csp->AddFixedVar(6), v3 = csp->AddFixedVar(5);
    csp->AddConstraint(OpConstraint(v0, v2, OpConstraint::Op::Inf, 0));
    csp->AddConstraint(OpConstraint(v0, v3, OpConstraint::Op::SupEqual, 0));
    csp->AddConstraint(OpConstraint(v1, v2, OpConstraint::Op::InfEqual, 0));
    csp->AddConstraint(OpConstraint(v1, v3, OpConstraint::Op::Sup, 0));
    csp->FinalizeModel();
    return csp;
}

int main() {
    std::vector<CSP*> owned;
    std::vector<const CSP*> csps;
    std::vector<Assignment> as;
    std::vector<std::string> names;
    auto add = [&](CSP* csp, bool own, const std::string& name) -> Assignment& {
        if (own) owned.push_back(csp);
        csps.push_back(csp);
        as.push_back(Assignment());
        as.back().Reset(*csp);
        names.push_back(name);
        return as.back();
    };
    try {
        add(op_inequality(), true, "op_inequality");
        add(queens(8), true, "nqueens8");
        add(sudoku_rows_cols(), true, "sudoku_rows_cols");
        for (int n = 4; n <= 12; n++) add(queens(n), true, "queens" + std::to_string(n));
        {
            CSP* csp = queens(8);                            // resumed: the first three of assign_order assigned by hand
            Assignment& a = add(csp, true, "resume_queens8_prefix024");
            const int vals[3] = {0, 2, 4};
            for (int i = 0; i < 3; i++) a.AssignVar(a.assign_order[i], vals[i]);
        }
        {
            CSP* csp = queens(6);                            // already complete: true without a device call
            Assignment& a = add(csp, true, "complete_queens6");
            if (!csp->ForwardCheckingStep(a)) throw b200::Error(DQ_ERR_INTERNAL, "6-Queens has a solution");
        }
        {
            CSP* csp = queens(9);                            // one CSP, three Assignments: two descriptors
            add(csp, true, "shared_queens9_full");
            Assignment& b = add(csp, false, "shared_queens9_col0_in_4_7");
            b.current_domains[0] = Domain(DomainType::Ranges, {4, 7});
            add(csp, false, "shared_queens9_full_again");
        }
        const std::vector<Assignment> copies = as;
        std::vector<Assignment*> ptrs;
        for (Assignment& a : as) ptrs.push_back(&a);
        const std::vector<bool> ok = b200::SolveAll(csps, ptrs);
        for (size_t i = 0; i < as.size(); i++) report("all", names[i], ok[i], as[i]);
        for (size_t i = 0; i < copies.size(); i++) {
            Assignment a = copies[i];
            const bool r = csps[i]->ForwardCheckingStep(a);
            report("step", names[i], r, a);
        }
    } catch (const b200::Error& e) {
        std::fprintf(stderr, "dequan::b200::Error %d: %s\n", e.code, e.what());
        return 1;
    }
    for (CSP* c : owned) delete c;
    return 0;
}
