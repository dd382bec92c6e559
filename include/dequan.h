/*
 * dequan.h — drop-in modelling header of the B200-native engine (dequan_b200).
 *
 * Source-compatible with the public API of nsweb/dequan's single header (reference
 * /root/reference/dequan.h, declarations 52-355): the same namespace, type, member and
 * method names, the same macros (DEQUAN_IMPLEMENTATION, DEQUAN_USE_STDVECTOR,
 * DEQUAN_WITH_STATS, DEQUAN_SET_CONSTRAINT_SIZE), so a model written against the reference
 * compiles unchanged.  What is different is everything behind it:
 *
 *   CSP::ForwardCheckingStep(a)  does NOT search on the host.  It flattens the model
 *   (a.current_domains, a.assign_order, the constraint list) into a dq_model_desc, hands it to the
 *   C ABI in dequan_b200.h (dq_compile + dq_solve_tree, hand-written CUDA for sm_100a) and writes
 *   the outcome back into the Assignment the way the reference leaves it:
 *       true  -> inst_vars complete, assigned_var_count == #vars, current_domains / saved_domains
 *                as they stand along the solution path, stats.assigned_vars += nodes visited
 *       false -> everything as after Reset, stats.assigned_vars += nodes visited
 *   There is no CPU search path.  Without the CUDA library or a device, or for a model outside
 *   the device engine's scope (see INTEGRATION.md), it throws dequan::b200::Error — it never
 *   falls back to a host solver.
 *
 *   The built-in constraints lower themselves to descriptor rows (OpConstraint, EqualityConstraint,
 *   AllDifferentConstraint, OrRangeConstraint).  A user-defined binary Constraint is lowered by
 *   tabulating its Evaluate over the two variables' value pairs (check-only, like the base-class
 *   AplyArcConsistency, reference dequan.h:147).  The host-side Evaluate / AplyArcConsistency
 *   bodies below exist for exactly two uses: that tabulation, and re-walking the ONE solution path
 *   after a successful solve to leave current_domains / saved_domains as the reference does.
 *
 * Link with -ldequan_b200 (dequan_b200/lib).  Header-only: DEQUAN_IMPLEMENTATION is accepted and
 * not needed.  Containers are always std::vector (the reference's custom-container mode is out of
 * scope, SURVEY.md §2).
 *
 * Extensions live in namespace dequan::b200 (all-solutions counting, engine options, multi-GPU
 * partitions) — see the bottom of this file.
 */
#ifndef DEQUAN_DROPIN_H
#define DEQUAN_DROPIN_H

#include <algorithm>
#include <climits>
#include <cstdint>
#include <cstring>
#include <new>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "dequan_b200.h"

#define DEQUAN_Array_Size(a)                a.size()
#define DEQUAN_Array_PushBack(a, val)       a.push_back(val)
#define DEQUAN_Array_Clear(a)               a.clear()
#define DEQUAN_Array_Resize(a, s)           a.resize(s)
#define DEQUAN_Array_Reserve(a, s)          a.reserve(s)
#define DEQUAN_Array_Back(a)                a.back()
#define DEQUAN_Array_PopBack(a)             a.pop_back()
#define DEQUAN_Array_Insert(a, idx, val)    a.insert(a.begin() + (idx), val)
#define DEQUAN_Array_Erase(a, first, last)  a.erase(a.begin() + (first), a.begin() + (last));
#define DEQUAN_Array_Sort(a, lambda)        std::sort(a.begin(), a.end(), lambda)

namespace dequan {

template <typename T>
using Array = std::vector<T>;
using VarId = int;

struct Var;
struct Constraint;
class Assignment;
class CSP;

namespace b200 {
/** Thrown by the solve entry points: no CUDA library/device, or a model the device engine does not cover. */
struct Error : std::runtime_error {
    Error(int c, const std::string& what) : std::runtime_error("dequan_b200: " + what), code(c) {}
    int code;   // dq_status
};
struct Lowering;   // descriptor under construction (defined below)
}  // namespace b200

/* Search counters (reference dequan.h:57-69).  Only assigned_vars (= nodes) is reproduced by the
 * device engine; the other two depend on the reference's sequential early-exit order and stay 0. */
struct Stats {
    unsigned long long validated_constraints = 0;
    unsigned long long applied_arcs = 0;
    unsigned long long assigned_vars = 0;
};

enum class DomainType : int { Values = 0, Ranges };

/* A finite integer domain: an explicit value list (iteration = list order) or sorted half-open
 * ranges [min0,max0,min1,max1,...).  Operations keep the reference's observable behaviour
 * (dequan.h:941-1172), including: Intersect(v) leaves the domain alone when v is absent. */
struct Domain {
    Domain() = default;
    Domain(DomainType t, const Array<int>& v) : type(t), values(v) {}

    int Size() const {
        if (type == DomainType::Values) return (int)values.size();
        int n = 0;
        for (size_t i = 0; i + 1 < values.size(); i += 2) n += values[i + 1] - values[i];
        return n;
    }
    bool Contains(int v) const {   // extension
        if (type == DomainType::Values) return std::find(values.begin(), values.end(), v) != values.end();
        for (size_t i = 0; i + 1 < values.size(); i += 2)
            if (values[i] <= v && v < values[i + 1]) return true;
        return false;
    }
    void Intersect(int val) {
        if (!Contains(val)) return;
        type = DomainType::Values;
        values.assign(1, val);
    }
    void Intersect(int val0, int val1) {
        Array<int> kept;
        if (type == DomainType::Values) {
            for (int v : values)
                if (v == val0 || v == val1) kept.push_back(v);
        } else {
            for (size_t i = 0; i + 1 < values.size(); i += 2) {
                if (values[i] <= val0 && val0 < values[i + 1]) kept.push_back(val0);
                if (values[i] <= val1 && val1 < values[i + 1]) kept.push_back(val1);
            }
            type = DomainType::Values;
        }
        values.swap(kept);
    }
    void IntersectRange(int rmin, int rmax) { Clip(rmin, rmax); }
    void Exclude(int val) {
        if (type == DomainType::Values) {
            auto it = std::find(values.begin(), values.end(), val);
            if (it != values.end()) values.erase(it);
            return;
        }
        for (size_t i = 0; i + 1 < values.size(); i += 2) {
            const int lo = values[i], hi = values[i + 1];
            if (val < lo || val >= hi) continue;
            if (hi - lo <= 1) values.erase(values.begin() + i, values.begin() + i + 2);
            else if (val == lo) values[i] = lo + 1;
            else if (val == hi - 1) values[i + 1] = val;
            else {                                   // split [lo,hi) into [lo,val) [val+1,hi)
                const int tail[2] = {val + 1, hi};
                values[i + 1] = val;
                values.insert(values.begin() + i + 2, tail, tail + 2);
            }
            return;
        }
    }
    void ExcludeSup(int rmax) { Clip(INT_MIN, rmax); }
    void ExcludeInf(int rmin) { Clip(rmin, INT_MAX); }
    bool operator==(const Domain& o) const { return type == o.type && values == o.values; }
    bool operator!=(const Domain& o) const { return !(*this == o); }

    DomainType type = DomainType::Values;
    Array<int> values;

private:
    void Clip(int rmin, int rmax) {                  // keep values in [rmin, rmax)
        size_t w = 0;
        if (type == DomainType::Values) {
            for (int v : values)
                if (rmin <= v && v < rmax) values[w++] = v;
        } else {
            for (size_t i = 0; i + 1 < values.size(); i += 2) {
                const int lo = std::max(values[i], rmin), hi = std::min(values[i + 1], rmax);
                if (hi > lo) { values[w++] = lo; values[w++] = hi; }
            }
        }
        values.resize(w);
    }
};

/* Copy of a domain taken before the first change at a search depth. */
struct SavedDomain {
    SavedDomain() = default;
    SavedDomain(VarId vid, DomainType t, const Array<int>& v) : var_id(vid), type(t), values(v) {}
    VarId var_id = -1;
    DomainType type = DomainType::Values;
    Array<int> values;
};
struct SavedDomains {
    Array<SavedDomain> domains;
};

struct InstVar {
    static const int UNASSIGNED = -INT_MAX;
    int value = InstVar::UNASSIGNED;
};

/* Constraint interface (reference dequan.h:134-148).  The spelling AplyArcConsistency is API. */
struct Constraint {
    enum class Eval : int { NA = 0, Passed, Failed };

    Constraint() = default;
    virtual ~Constraint() = default;
    virtual void LinkVars(Array<Var>& vars) = 0;
    virtual Eval Evaluate(const Array<InstVar>& inst_vars, VarId last_assigned_vid) = 0;
    virtual bool AplyArcConsistency(Assignment& /*a*/, VarId /*last_assigned_vid*/) { return true; }
    /* Extension: built-in constraints append their descriptor row and return true; a user-defined
     * constraint keeps this default and is lowered by tabulating Evaluate. */
    virtual bool LowerB200(b200::Lowering& /*out*/) const { return false; }
};

/* Inline polymorphic storage for any Constraint-derived object (reference dequan.h:155-171). */
struct GenericConstraint {
#ifdef DEQUAN_SET_CONSTRAINT_SIZE
    static constexpr int MAX_CONSTRAINT_SIZE = DEQUAN_SET_CONSTRAINT_SIZE;
#else
    struct MaxConstraint {
        virtual ~MaxConstraint() {}
        union { Array<int> a; int v[4]; };
    };
    static constexpr int MAX_CONSTRAINT_SIZE = sizeof(MaxConstraint);
#endif
    alignas(void*) char buffer[MAX_CONSTRAINT_SIZE];

    Constraint* operator->() { return reinterpret_cast<Constraint*>(buffer); }
    Constraint* get() { return reinterpret_cast<Constraint*>(buffer); }
    const Constraint* get() const { return reinterpret_cast<const Constraint*>(buffer); }
};

struct Var {
    Var() = default;
    Var(VarId vid, const Array<Constraint*>& lk) : var_id(vid), linked_constraints(lk) {}
    static const VarId INVALID = -1;
    VarId var_id = Var::INVALID;
    Array<Constraint*> linked_constraints;
};

/* Search state handed to and filled by CSP::ForwardCheckingStep (reference dequan.h:287-321). */
class Assignment {
public:
    Assignment() {}
    void Reset(const CSP& csp);
    bool IsComplete() { return assigned_var_count == (int)inst_vars.size(); }
    int GetInstVarValue(VarId vid) const { return inst_vars[vid].value; }
    const Domain& GetCurrentDomain(VarId vid) const { return current_domains[vid]; }
    VarId NextUnassignedVar() { return assign_order[assigned_var_count]; }
    void AssignVar(VarId vid, int val) {
        inst_vars[vid].value = val;
        ++assigned_var_count;
#ifdef DEQUAN_WITH_STATS
        ++stats.assigned_vars;
#endif
    }
    void UnAssignVar(VarId vid) {
        inst_vars[vid].value = InstVar::UNASSIGNED;
        --assigned_var_count;
    }
    bool ValidateVarConstraints(const Var& var) {
        for (Constraint* c : var.linked_constraints) {
#ifdef DEQUAN_WITH_STATS
            ++stats.validated_constraints;
#endif
            if (c->Evaluate(inst_vars, var.var_id) == Constraint::Eval::Failed) return false;
        }
        return true;
    }
    void EnsureSavedDomain(VarId vid, const Domain& dom) {
        Array<SavedDomain>& frame = saved_domains.back().domains;
        for (const SavedDomain& s : frame)
            if (s.var_id == vid) return;
        frame.emplace_back(vid, dom.type, dom.values);
    }
    void RestoreSavedDomainStep() {
        for (const SavedDomain& s : saved_domains.back().domains) {
            current_domains[s.var_id].type = s.type;
            current_domains[s.var_id].values = s.values;
        }
    }

    int assigned_var_count = 0;
    Array<InstVar> inst_vars;
    Array<Domain> current_domains;
    Array<SavedDomains> saved_domains;
    Array<VarId> assign_order;
#ifdef DEQUAN_WITH_STATS
    Stats stats;
#endif
};

namespace b200 {

/* Descriptor rows being collected for dq_compile (include/dequan_b200.h dq_model_desc). */
struct Lowering {
    std::vector<int32_t> con_kind, con_off{0}, con_data;
    void Row(int kind, std::initializer_list<int32_t> payload) { Row(kind, payload.begin(), payload.size()); }
    void Row(int kind, const int32_t* p, size_t n) {
        con_kind.push_back(kind);
        con_data.insert(con_data.end(), p, p + n);
        con_off.push_back((int32_t)con_data.size());
    }
};

namespace detail {
/* The one filtering step every built-in binary constraint performs on the endpoint that is still
 * unassigned (reference DoCheck, dequan.h:636-669): back the domain up once per depth, filter,
 * report a wipe-out. */
template <class F>
inline bool FilterDomain(Assignment& a, VarId target, F&& filter) {
    Domain& dom = a.current_domains[target];
    a.EnsureSavedDomain(target, dom);
    filter(dom);
    return !dom.values.empty();
}
inline void CountArc(Assignment& a) {
#ifdef DEQUAN_WITH_STATS
    ++a.stats.applied_arcs;
#else
    (void)a;
#endif
}
}  // namespace detail
}  // namespace b200

/* v0 (op) v1 + offset */
struct OpConstraint : public Constraint {
    enum class Op : int { Equal = 0, NotEqual, SupEqual, Sup, InfEqual, Inf };

    OpConstraint(VarId _v0, VarId _v1, Op _op, int _offset) : v0(_v0), v1(_v1), op(_op), offset(_offset) {
        static_assert(sizeof(OpConstraint) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "");
    }
    void LinkVars(Array<Var>& vars) override {
        vars[v0].linked_constraints.push_back(this);
        vars[v1].linked_constraints.push_back(this);
    }
    static bool Holds(Op o, long long lhs, long long rhs) {
        switch (o) {
            case Op::Equal:    return lhs == rhs;
            case Op::NotEqual: return lhs != rhs;
            case Op::SupEqual: return lhs >= rhs;
            case Op::Sup:      return lhs > rhs;
            case Op::InfEqual: return lhs <= rhs;
            case Op::Inf:      return lhs < rhs;
        }
        return false;
    }
    Eval Evaluate(const Array<InstVar>& iv, VarId) override {
        if (iv[v0].value == InstVar::UNASSIGNED || iv[v1].value == InstVar::UNASSIGNED) return Eval::NA;
        return Holds(op, iv[v0].value, (long long)iv[v1].value + offset) ? Eval::Passed : Eval::Failed;
    }
    /* target (o) bound  ->  the Domain operation that enforces it */
    static void Enforce(Domain& d, Op o, int bound) {
        switch (o) {
            case Op::Equal:    d.Intersect(bound); break;
            case Op::NotEqual: d.Exclude(bound); break;
            case Op::SupEqual: d.ExcludeInf(bound); break;
            case Op::Sup:      d.ExcludeInf(bound + 1); break;
            case Op::InfEqual: d.ExcludeSup(bound + 1); break;
            case Op::Inf:      d.ExcludeSup(bound); break;
        }
    }
    static Op Mirror(Op o) {
        switch (o) {
            case Op::SupEqual: return Op::InfEqual;
            case Op::Sup:      return Op::Inf;
            case Op::InfEqual: return Op::SupEqual;
            case Op::Inf:      return Op::Sup;
            default:           return o;
        }
    }
    bool AplyArcConsistency(Assignment& a, VarId) override {
        b200::detail::CountArc(a);
        const int x0 = a.inst_vars[v0].value, x1 = a.inst_vars[v1].value;
        if (x0 == InstVar::UNASSIGNED) {
            const Op o = op; const int bound = x1 + offset;
            return b200::detail::FilterDomain(a, v0, [o, bound](Domain& d) { Enforce(d, o, bound); });
        }
        if (x1 == InstVar::UNASSIGNED) {
            const Op o = Mirror(op); const int bound = x0 - offset;
            return b200::detail::FilterDomain(a, v1, [o, bound](Domain& d) { Enforce(d, o, bound); });
        }
        return true;
    }
    bool LowerB200(b200::Lowering& out) const override {
        out.Row(DQ_CON_OP, {v0, v1, (int32_t)op, offset});
        return true;
    }

    VarId v0, v1;
    Op op = Op::Equal;
    int offset = 0;
};

/* v0 == v1 */
struct EqualityConstraint : public Constraint {
    EqualityConstraint(VarId _v0, VarId _v1) : v0(_v0), v1(_v1) {
        static_assert(sizeof(EqualityConstraint) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "");
    }
    void LinkVars(Array<Var>& vars) override {
        vars[v0].linked_constraints.push_back(this);
        vars[v1].linked_constraints.push_back(this);
    }
    Eval Evaluate(const Array<InstVar>& iv, VarId) override {
        if (iv[v0].value == InstVar::UNASSIGNED || iv[v1].value == InstVar::UNASSIGNED) return Eval::NA;
        return iv[v0].value == iv[v1].value ? Eval::Passed : Eval::Failed;
    }
    bool AplyArcConsistency(Assignment& a, VarId) override {
        b200::detail::CountArc(a);
        const int x0 = a.inst_vars[v0].value, x1 = a.inst_vars[v1].value;
        if (x0 == InstVar::UNASSIGNED) return b200::detail::FilterDomain(a, v0, [x1](Domain& d) { d.Intersect(x1); });
        if (x1 == InstVar::UNASSIGNED) return b200::detail::FilterDomain(a, v1, [x0](Domain& d) { d.Intersect(x0); });
        return true;
    }
    bool LowerB200(b200::Lowering& out) const override {
        out.Row(DQ_CON_EQ, {v0, v1});
        return true;
    }
    VarId v0, v1;
};

/* v0 == v1 || v0 == v2 — ternary: declared for source compatibility, NOT covered by the device
 * engine (SURVEY.md §2: out of scope); a model that adds one makes the solve throw b200::Error. */
struct OrEqualityConstraint : public Constraint {
    OrEqualityConstraint(VarId _v0, VarId _v1, VarId _v2) : v0(_v0), v1(_v1), v2(_v2) {
        static_assert(sizeof(OrEqualityConstraint) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "");
    }
    void LinkVars(Array<Var>& vars) override {
        for (VarId v : {v0, v1, v2}) vars[v].linked_constraints.push_back(this);
    }
    Eval Evaluate(const Array<InstVar>& iv, VarId) override {
        for (VarId v : {v0, v1, v2})
            if (iv[v].value == InstVar::UNASSIGNED) return Eval::NA;
        return (iv[v0].value == iv[v1].value || iv[v0].value == iv[v2].value) ? Eval::Passed : Eval::Failed;
    }
    VarId v0, v1, v2;
};

/* v0 == v1 + v2 - v3 — 4-ary: declared for source compatibility, NOT covered by the device engine. */
struct CombinedEqualityConstraint : public Constraint {
    CombinedEqualityConstraint(VarId _v0, VarId _v1, VarId _v2, VarId _v3) : v0(_v0), v1(_v1), v2(_v2), v3(_v3) {
        static_assert(sizeof(CombinedEqualityConstraint) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "");
    }
    void LinkVars(Array<Var>& vars) override {
        for (VarId v : {v0, v1, v2, v3}) vars[v].linked_constraints.push_back(this);
    }
    Eval Evaluate(const Array<InstVar>& iv, VarId) override {
        for (VarId v : {v0, v1, v2, v3})
            if (iv[v].value == InstVar::UNASSIGNED) return Eval::NA;
        return iv[v0].value == iv[v1].value + iv[v2].value - iv[v3].value ? Eval::Passed : Eval::Failed;
    }
    VarId v0, v1, v2, v3;
};

/* (min <= v0 < max) || (min <= v1 < max) — check-only: the reference compiles its filter out
 * (dequan.h:860-893), so AplyArcConsistency is the base-class no-op plus the arc counter. */
struct OrRangeConstraint : public Constraint {
    OrRangeConstraint(VarId _v0, VarId _v1, int _min, int _max) : v0(_v0), v1(_v1), min(_min), max(_max) {
        static_assert(sizeof(OrRangeConstraint) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "");
    }
    void LinkVars(Array<Var>& vars) override {
        vars[v0].linked_constraints.push_back(this);
        vars[v1].linked_constraints.push_back(this);
    }
    Eval Evaluate(const Array<InstVar>& iv, VarId) override {
        if (iv[v0].value == InstVar::UNASSIGNED || iv[v1].value == InstVar::UNASSIGNED) return Eval::NA;
        const bool in0 = iv[v0].value >= min && iv[v0].value < max, in1 = iv[v1].value >= min && iv[v1].value < max;
        return (in0 || in1) ? Eval::Passed : Eval::Failed;
    }
    bool AplyArcConsistency(Assignment& a, VarId) override {
        b200::detail::CountArc(a);
        return true;
    }
    bool LowerB200(b200::Lowering& out) const override {
        out.Row(DQ_CON_ORRANGE, {v0, v1, min, max});
        return true;
    }
    VarId v0, v1;
    int min, max;
};

/* Pairwise-different over a set of variables. */
struct AllDifferentConstraint : public Constraint {
    AllDifferentConstraint(const Array<VarId>& vars) : alldiff_vars(vars) {
        static_assert(sizeof(AllDifferentConstraint) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "");
    }
    void LinkVars(Array<Var>& vars) override {
        for (VarId v : alldiff_vars) vars[v].linked_constraints.push_back(this);
    }
    Eval Evaluate(const Array<InstVar>& iv, VarId last) override {
        for (VarId v : alldiff_vars)
            if (v != last && iv[v].value == iv[last].value) return Eval::Failed;
        return Eval::Passed;
    }
    bool AplyArcConsistency(Assignment& a, VarId last) override {
        b200::detail::CountArc(a);
        const int taken = a.inst_vars[last].value;
        for (VarId v : alldiff_vars) {
            if (a.inst_vars[v].value != InstVar::UNASSIGNED) continue;
            if (!b200::detail::FilterDomain(a, v, [taken](Domain& d) { d.Exclude(taken); })) return false;
        }
        return true;
    }
    bool LowerB200(b200::Lowering& out) const override {
        out.Row(DQ_CON_ALLDIFF, alldiff_vars.data(), alldiff_vars.size());
        return true;
    }
    Array<VarId> alldiff_vars;
};

namespace b200 {

/* Options of the device solve (a superset of what ForwardCheckingStep needs). */
struct SolveOptions {
    int engine = DQ_ENGINE_AUTO;
    int split_depth = 0;        // <= 0: automatic
    int part_rank = 0;          // one process per GPU: this process' partition of the prefix-split tree
    int part_count = 1;
    int n_gpus = 1;             // > 1: this one call deals the tree to CUDA devices 0..n_gpus-1 (dq_solve_tree_multi)
};

/* What a device solve reports beyond the Assignment. */
struct SolveReport {
    dq_tree_result tree{};
    bool compiled_fresh = false;    // false: the cached device tables of an identical earlier call were reused
};

/* Owns the dq_model handle cached inside a CSP between solves. */
struct ModelCache {
    dq_model* handle = nullptr;
    std::vector<int32_t> key;       // the flattened descriptor the handle was compiled from
    ModelCache() = default;
    ModelCache(const ModelCache&) {}                       // a copied CSP recompiles
    ModelCache& operator=(const ModelCache&) { Drop(); return *this; }
    ~ModelCache() { Drop(); }
    void Drop() {
        if (handle) dq_free(handle);
        handle = nullptr;
        key.clear();
    }
};

/* Many (CSP, Assignment) pairs in one device call (dq_solve_models).  Element i is what csps[i]->ForwardCheckingStep(*as[i])
 * returns, and every Assignment is left exactly as that call leaves it.  Several pairs may share one CSP.  reps (may be
 * null) is resized to the number of pairs; its tree results carry outcome, n_solutions and n_nodes, first_key only as a
 * flag (0: a solution, UINT64_MAX: none; the batch reports no prefix keys), and every other field 0. */
inline std::vector<bool> SolveAll(const std::vector<const CSP*>& csps, const std::vector<Assignment*>& as,
                                  std::vector<SolveReport>* reps = nullptr);

}  // namespace b200

/* The model (reference dequan.h:328-355).  Static during the search. */
class CSP {
public:
    CSP() = default;

    VarId AddIntVar(int min_val, int max_val) { return AddIntVar(Domain(DomainType::Ranges, {min_val, max_val})); }
    VarId AddIntVar(const Domain& domain) {
        const VarId id = (VarId)vars.size();
        vars.push_back(Var(id, {}));
        domains.push_back(domain);
        return id;
    }
    VarId AddFixedVar(int val) { return AddIntVar(Domain(DomainType::Values, {val})); }
    VarId AddBoolVar() { return AddIntVar(Domain(DomainType::Values, {0, 1})); }

    template <class T>
    void AddConstraint(const T& con) {
        static_assert(sizeof(T) <= GenericConstraint::MAX_CONSTRAINT_SIZE, "raise DEQUAN_SET_CONSTRAINT_SIZE");
        GenericConstraint slot;
        new (slot.buffer) T(con);
        constraints.push_back(slot);                 // bit-copied like the reference (dequan.h:482)
    }

    /* Links every constraint to its variables; call once, after the last AddConstraint. */
    void FinalizeModel() {
        scopes_.assign(constraints.size(), {});
        std::vector<size_t> before(vars.size());
        for (size_t c = 0; c < constraints.size(); c++) {
            for (size_t v = 0; v < vars.size(); v++) before[v] = vars[v].linked_constraints.size();
            constraints[c]->LinkVars(vars);
            for (size_t v = 0; v < vars.size(); v++)
                if (vars[v].linked_constraints.size() != before[v]) scopes_[c].push_back((VarId)v);
        }
        cache_.Drop();
    }

    /* Solves from the state in `a` (as left by Assignment::Reset) on the current CUDA device:
     * DFS-first solution under a.assign_order and the domains' iteration order. */
    bool ForwardCheckingStep(Assignment& a) const;

    Array<Var> vars;
    Array<GenericConstraint> constraints;
    Array<Domain> domains;

    /* ---- extensions (namespace b200 has the free-function forms) ---- */
    bool SolveB200(Assignment& a, int mode, const b200::SolveOptions& opt, b200::SolveReport* rep) const;
    /* b200::EnumerateAll: every solution in the search's visiting order, values by var id. */
    void EnumerateB200(const Assignment& a, const b200::SolveOptions& opt, b200::SolveReport* rep,
                       std::vector<std::vector<int> >& out, unsigned long long max_solutions) const;

private:
    friend std::vector<bool> b200::SolveAll(const std::vector<const CSP*>&, const std::vector<Assignment*>&,
                                            std::vector<b200::SolveReport>*);
    /* The flattened descriptor of a lowering; `key` holds all of it in one flat vector (equal key: equal tables). */
    struct Lowered {
        b200::Lowering low;
        std::vector<int32_t> dom_type, dom_off, dom_vals, order, key;
    };
    void Lower(const Assignment& a, Lowered& out) const;
    static dq_model* Compile(const Lowered& l, int nv);
    bool CompileB200(const Assignment& a) const;
    int CheckResumable(const Assignment& a) const;
    bool FinishB200(Assignment& a, uint64_t nodes, bool have, const int32_t* first, int resumed) const;
    void Flatten(const Assignment& a, b200::Lowering& low, std::vector<int32_t>& dom_type, std::vector<int32_t>& dom_off,
                 std::vector<int32_t>& dom_vals) const;
    void TabulateUserConstraint(size_t c, b200::Lowering& low, const Assignment& a) const;

    std::vector<std::vector<VarId>> scopes_;        // per constraint: the variables LinkVars attached it to
    mutable b200::ModelCache cache_;
};

inline void Assignment::Reset(const CSP& csp) {
    assigned_var_count = 0;
    inst_vars.assign(csp.vars.size(), InstVar());
    current_domains = csp.domains;
    saved_domains.clear();
    saved_domains.reserve(csp.vars.size());
    assign_order.resize(csp.vars.size());
    for (size_t i = 0; i < assign_order.size(); i++) assign_order[i] = (VarId)i;
    // smallest initial domain first, ties by id: a stable sort on the size alone
    std::vector<int> size(csp.vars.size());
    for (size_t i = 0; i < size.size(); i++) size[i] = current_domains[i].Size();
    std::stable_sort(assign_order.begin(), assign_order.end(), [&size](VarId x, VarId y) { return size[x] < size[y]; });
}

/* A user-defined constraint becomes a DQ_CON_TABLE row — the (v0,v1) value pairs its Evaluate does not reject — or,
 * when it overrides AplyArcConsistency (reference dequan.h:145-147) with a step that filters the other endpoint's
 * domain, a DQ_CON_FILTER row that adds, per direction, the value pairs the filter keeps.  Requirements, each checked
 * on the Assignment's current domains: exactly two variables in scope; Evaluate does not fail with only one of them
 * assigned; the filter touches only the unassigned endpoint of the pair, answers false exactly when it leaves that
 * domain empty (what ForwardCheckingStep takes for a wipe-out, dequan.h:514-518), and removes a value whatever
 * else the domain holds (it is run on the full domain and on every other value of it: the answers must agree). */
inline void CSP::TabulateUserConstraint(size_t c, b200::Lowering& low, const Assignment& a) const {
    const std::vector<VarId>& scope = scopes_[c];
    if (scope.size() != 2)
        throw b200::Error(DQ_ERR_UNSUPPORTED, "constraint #" + std::to_string(c) + " links " + std::to_string(scope.size()) +
                                                  " variables; only binary user-defined constraints are lowered");
    Constraint* con = const_cast<GenericConstraint&>(constraints[c]).get();
    const VarId x = scope[0], y = scope[1];
    auto expand = [](const Domain& d) {
        Array<int> out;
        if (d.type == DomainType::Values) out = d.values;
        else
            for (size_t i = 0; i + 1 < d.values.size(); i += 2)
                for (int v = d.values[i]; v < d.values[i + 1]; v++) out.push_back(v);
        return out;
    };
    const Array<int> xs = expand(a.current_domains[x]), ys = expand(a.current_domains[y]);
    Array<InstVar> iv(vars.size());
    std::vector<int32_t> allow;
    for (int av : xs) {
        iv[x].value = av;
        if (con->Evaluate(iv, x) == Constraint::Eval::Failed)
            throw b200::Error(DQ_ERR_UNSUPPORTED, "user constraint fails with a single variable assigned (unary part)");
        for (int bv : ys) {
            iv[y].value = bv;
            if (con->Evaluate(iv, y) != Constraint::Eval::Failed && con->Evaluate(iv, x) != Constraint::Eval::Failed) {
                allow.push_back(av);
                allow.push_back(bv);
            }
        }
        iv[y].value = InstVar::UNASSIGNED;
    }
    iv[x].value = InstVar::UNASSIGNED;
    for (int bv : ys) {
        iv[y].value = bv;
        if (con->Evaluate(iv, y) == Constraint::Eval::Failed)
            throw b200::Error(DQ_ERR_UNSUPPORTED, "user constraint fails with a single variable assigned (unary part)");
    }
    // its AplyArcConsistency, once per value of either endpoint on a scratch state
    std::vector<int32_t> keep[2];
    bool filters = false;
    for (int side = 0; side < 2; side++) {
        const VarId from = side ? y : x, to = side ? x : y;
        const Array<int>& from_vals = side ? ys : xs;
        const Array<int>& to_vals = side ? xs : ys;
        for (int v : from_vals) {
            std::vector<char> kept_full(to_vals.size(), 0);
            for (int pass = 0; pass < 3; pass++) {               // the full domain, then its even / odd positions only
                Assignment scratch;
                scratch.inst_vars.assign(vars.size(), InstVar());
                scratch.current_domains = a.current_domains;
                scratch.assign_order = a.assign_order;
                scratch.saved_domains.emplace_back();
                if (pass) {
                    Array<int> sub;
                    for (size_t i = 0; i < to_vals.size(); i++) if ((int)(i & 1) == pass - 1) sub.push_back(to_vals[i]);
                    scratch.current_domains[to] = Domain(DomainType::Values, sub);
                }
                const Array<Domain> before = scratch.current_domains;
                scratch.inst_vars[from].value = v;
                scratch.assigned_var_count = 1;
                const bool ok = con->AplyArcConsistency(scratch, from);
                for (size_t u = 0; u < vars.size(); u++)
                    if ((VarId)u != to && scratch.current_domains[u] != before[u])
                        throw b200::Error(DQ_ERR_UNSUPPORTED, "user constraint's AplyArcConsistency changes a domain other than its unassigned endpoint's");
                const Array<int> left = expand(scratch.current_domains[to]);
                if (ok == left.empty())
                    throw b200::Error(DQ_ERR_UNSUPPORTED, "user constraint's AplyArcConsistency must answer false exactly when it empties the domain");
                if (scratch.current_domains[to] != before[to]) filters = true;
                for (size_t i = 0; i < to_vals.size(); i++) {
                    const bool in_start = pass == 0 || (int)(i & 1) == pass - 1;
                    if (!in_start) continue;
                    const bool kept = std::find(left.begin(), left.end(), to_vals[i]) != left.end();
                    if (pass == 0) kept_full[i] = kept;
                    else if (kept != (bool)kept_full[i])
                        throw b200::Error(DQ_ERR_UNSUPPORTED, "user constraint's AplyArcConsistency depends on the other values of the domain it filters");
                }
                for (int lv : left)
                    if (std::find(to_vals.begin(), to_vals.end(), lv) == to_vals.end())
                        throw b200::Error(DQ_ERR_UNSUPPORTED, "user constraint's AplyArcConsistency adds values to a domain");
            }
            for (size_t i = 0; i < to_vals.size(); i++)
                if (kept_full[i]) {
                    keep[side].push_back(side ? to_vals[i] : v);          // pairs are (value of scope[0], value of scope[1])
                    keep[side].push_back(side ? v : to_vals[i]);
                }
        }
    }
    if (!filters) {
        std::vector<int32_t> row{x, y};
        row.insert(row.end(), allow.begin(), allow.end());
        low.Row(DQ_CON_TABLE, row.data(), row.size());
        return;
    }
    std::vector<int32_t> row{x, y, (int32_t)(allow.size() / 2), (int32_t)(keep[0].size() / 2), (int32_t)(keep[1].size() / 2)};
    row.insert(row.end(), allow.begin(), allow.end());
    row.insert(row.end(), keep[0].begin(), keep[0].end());
    row.insert(row.end(), keep[1].begin(), keep[1].end());
    low.Row(DQ_CON_FILTER, row.data(), row.size());
}

inline void CSP::Flatten(const Assignment& a, b200::Lowering& low, std::vector<int32_t>& dom_type,
                         std::vector<int32_t>& dom_off, std::vector<int32_t>& dom_vals) const {
    if (scopes_.size() != constraints.size())
        throw b200::Error(DQ_ERR_INVALID, "FinalizeModel() must be called after the last AddConstraint()");
    // A partially assigned Assignment (the reference resumes at assign_order[assigned_var_count], dequan.h:411-414,
    // 504): the assigned variables become singleton domains at the head of the order, and because the reference never
    // filtered from them, every constraint between an assigned and an unassigned variable is lowered CHECK-ONLY (the
    // value pairs its Evaluate accepts: the unassigned side's values are still visited and fail validation, exactly as
    // in the reference); a constraint among assigned variables only is never evaluated again and is dropped.
    const int p = a.assigned_var_count;
    std::vector<char> pre(vars.size(), 0);
    for (int i = 0; i < p; i++) pre[a.assign_order[i]] = 1;
    dom_off.assign(1, 0);
    for (size_t v = 0; v < a.current_domains.size(); v++) {
        const Domain& d = a.current_domains[v];
        if (pre[v]) {
            dom_type.push_back(DQ_DOM_VALUES);
            dom_vals.push_back(a.inst_vars[v].value);
        } else {
            dom_type.push_back(d.type == DomainType::Ranges ? DQ_DOM_RANGES : DQ_DOM_VALUES);
            dom_vals.insert(dom_vals.end(), d.values.begin(), d.values.end());
        }
        dom_off.push_back((int32_t)dom_vals.size());
    }
    auto expand = [](const Domain& d) {
        Array<int> out;
        if (d.type == DomainType::Values) out = d.values;
        else
            for (size_t i = 0; i + 1 < d.values.size(); i += 2)
                for (int v = d.values[i]; v < d.values[i + 1]; v++) out.push_back(v);
        return out;
    };
    for (size_t c = 0; c < constraints.size(); c++) {
        const std::vector<VarId>& scope = scopes_[c];
        size_t n_pre = 0;
        for (VarId v : scope) n_pre += pre[v];
        Constraint* con = const_cast<GenericConstraint&>(constraints[c]).get();
        if (n_pre == 0) {
            if (!con->LowerB200(low)) {
                if (scope.size() > 2 || scope.empty()) {
                    // built-in ternary/4-ary constraints land here too
                    throw b200::Error(DQ_ERR_UNSUPPORTED, "constraint #" + std::to_string(c) + " links " + std::to_string(scope.size()) +
                                                              " variables; the device engine lowers unary-free binary constraints and AllDifferent only");
                }
                TabulateUserConstraint(c, low, a);
            }
            continue;
        }
        if (n_pre == scope.size()) continue;
        if (const AllDifferentConstraint* ad = dynamic_cast<const AllDifferentConstraint*>(con)) {
            std::vector<int32_t> open;
            for (VarId v : ad->alldiff_vars) if (!pre[v]) open.push_back(v);
            if (open.size() >= 2) low.Row(DQ_CON_ALLDIFF, open.data(), open.size());
            for (VarId pv : ad->alldiff_vars) {
                if (!pre[pv]) continue;
                const int held = a.inst_vars[pv].value;
                for (VarId x : open) {
                    std::vector<int32_t> row{pv, x};
                    for (int xv : expand(a.current_domains[x])) if (xv != held) { row.push_back(held); row.push_back(xv); }
                    low.Row(DQ_CON_TABLE, row.data(), row.size());
                }
            }
            continue;
        }
        if (scope.size() != 2)
            throw b200::Error(DQ_ERR_UNSUPPORTED, "constraint #" + std::to_string(c) + " links " + std::to_string(scope.size()) + " variables");
        const VarId x = pre[scope[0]] ? scope[1] : scope[0];          // the endpoint still to assign
        Array<InstVar> iv = a.inst_vars;
        std::vector<int32_t> row{scope[0], scope[1]};
        for (int xv : expand(a.current_domains[x])) {
            iv[x].value = xv;
            if (con->Evaluate(iv, x) == Constraint::Eval::Failed) continue;
            row.push_back(iv[scope[0]].value);
            row.push_back(iv[scope[1]].value);
        }
        low.Row(DQ_CON_TABLE, row.data(), row.size());
    }
}

/* Lowers the CSP with the Assignment's domains and order. */
inline void CSP::Lower(const Assignment& a, Lowered& l) const {
    l.order.assign(a.assign_order.begin(), a.assign_order.end());
    Flatten(a, l.low, l.dom_type, l.dom_off, l.dom_vals);
    // one flat key for the cache: identical descriptor -> identical device tables
    l.key.clear();
    l.key.reserve(l.dom_type.size() + l.dom_off.size() + l.dom_vals.size() + l.order.size() + l.low.con_kind.size() +
                  l.low.con_off.size() + l.low.con_data.size() + 8);
    for (const std::vector<int32_t>* part : {&l.dom_type, &l.dom_off, &l.dom_vals, &l.order, &l.low.con_kind, &l.low.con_off, &l.low.con_data}) {
        l.key.push_back((int32_t)part->size());
        l.key.insert(l.key.end(), part->begin(), part->end());
    }
}

inline dq_model* CSP::Compile(const Lowered& l, int nv) {
    const int32_t zero = 0;
    dq_model_desc desc{};
    desc.n_vars = nv;
    desc.dom_type = l.dom_type.empty() ? &zero : l.dom_type.data();
    desc.dom_off = l.dom_off.data();
    desc.dom_vals = l.dom_vals.empty() ? &zero : l.dom_vals.data();
    desc.n_cons = (int32_t)l.low.con_kind.size();
    desc.con_kind = l.low.con_kind.empty() ? &zero : l.low.con_kind.data();
    desc.con_off = l.low.con_off.data();
    desc.con_data = l.low.con_data.empty() ? &zero : l.low.con_data.data();
    desc.assign_order = l.order.empty() ? nullptr : l.order.data();
    dq_model* h = nullptr;
    const int rc = dq_compile(&desc, &h);
    if (rc != DQ_OK) throw b200::Error(rc, dq_last_error());
    return h;
}

/* Lowers the CSP with the Assignment's domains and order and compiles it, unless the cached handle was built from the
 * identical descriptor.  Returns whether it compiled afresh. */
inline bool CSP::CompileB200(const Assignment& a) const {
    Lowered l;
    Lower(a, l);
    const bool fresh = !cache_.handle || cache_.key != l.key;
    if (fresh) {
        cache_.Drop();
        cache_.handle = Compile(l, (int)vars.size());
        cache_.key.swap(l.key);
    }
    return fresh;
}

/* Checks that `a` belongs to this CSP and that its assigned variables are a prefix of assign_order; returns the prefix's
 * length (the reference resumes after it, dequan.h:504). */
inline int CSP::CheckResumable(const Assignment& a) const {
    const int nv = (int)vars.size();
    if ((int)a.inst_vars.size() != nv || (int)a.current_domains.size() != nv || (int)a.assign_order.size() != nv)
        throw b200::Error(DQ_ERR_INVALID, "Assignment does not belong to this CSP: call a.Reset(csp) first");
    const int resumed = a.assigned_var_count;
    for (int i = 0; i < nv; i++)
        if ((a.inst_vars[a.assign_order[i]].value != InstVar::UNASSIGNED) != (i < resumed))
            throw b200::Error(DQ_ERR_UNSUPPORTED, "the assigned variables must be the first assigned_var_count entries of assign_order");
    return resumed;
}

/* Writes a device answer back into `a`: `nodes` is the device's node count (it visits each of the `resumed` pre-assigned
 * singletons once; the reference does not), `first` the solution by var id when `have`.  Returns `have`. */
inline bool CSP::FinishB200(Assignment& a, uint64_t nodes, bool have, const int32_t* first, int resumed) const {
#ifdef DEQUAN_WITH_STATS
    a.stats.assigned_vars += nodes - (uint64_t)resumed;
#else
    (void)nodes;
#endif
    if (!have) return false;
    // Leave the Assignment as the reference's recursion leaves it on success: walk the one solution
    // path, one saved-domain frame per depth, each linked constraint filtering in link order.
    const int nv = (int)vars.size();
    for (int d = resumed; d < nv; d++) {
        const VarId vid = a.assign_order[d];
        a.saved_domains.emplace_back();
        a.inst_vars[vid].value = first[vid];
        ++a.assigned_var_count;
#ifdef DEQUAN_WITH_STATS
        Stats keep = a.stats;
#endif
        for (Constraint* c : vars[vid].linked_constraints) c->AplyArcConsistency(a, vid);
#ifdef DEQUAN_WITH_STATS
        a.stats = keep;                              // applied_arcs is not reproduced (sequential early-exit dependent)
#endif
    }
    return true;
}

inline bool CSP::SolveB200(Assignment& a, int mode, const b200::SolveOptions& opt, b200::SolveReport* rep) const {
    const int nv = (int)vars.size();
    const int resumed = CheckResumable(a);
    const bool fresh = CompileB200(a);

    dq_tree_opts o{};
    o.mode = mode;
    o.split_depth = opt.split_depth;
    o.part_rank = opt.part_rank;
    o.part_count = opt.part_count;
    o.engine = opt.engine;
    dq_tree_result r{};
    std::vector<int32_t> first((size_t)std::max(nv, 1), InstVar::UNASSIGNED);
    const int rc = opt.n_gpus > 1 ? dq_solve_tree_multi(cache_.handle, &o, opt.n_gpus, nullptr, &r, first.data())
                                  : dq_solve_tree(cache_.handle, &o, &r, first.data());
    if (rc != DQ_OK) throw b200::Error(rc, dq_last_error());
    if (rep) { rep->tree = r; rep->compiled_fresh = fresh; }
    if (rep) rep->tree.n_nodes -= (uint64_t)resumed;     // (the device visits each pre-assigned singleton once; the reference does not)
    const bool have = r.first_key != UINT64_MAX && (nv == 0 || first[0] != InstVar::UNASSIGNED);
    return FinishB200(a, r.n_nodes, have, first.data(), resumed);
}

inline void CSP::EnumerateB200(const Assignment& a, const b200::SolveOptions& opt, b200::SolveReport* rep,
                               std::vector<std::vector<int> >& out, unsigned long long max_solutions) const {
    const int nv = (int)vars.size();
    if ((int)a.inst_vars.size() != nv || (int)a.current_domains.size() != nv || (int)a.assign_order.size() != nv)
        throw b200::Error(DQ_ERR_INVALID, "Assignment does not belong to this CSP: call a.Reset(csp) first");
    if (a.assigned_var_count != 0)
        throw b200::Error(DQ_ERR_UNSUPPORTED, "resuming a partially assigned Assignment is not supported; Reset() it");
    const bool fresh = CompileB200(a);
    dq_tree_opts o{};
    o.mode = DQ_MODE_COUNT_ALL;
    o.split_depth = opt.split_depth;
    o.part_rank = opt.part_rank;
    o.part_count = opt.part_count;
    o.engine = opt.engine;
    dq_tree_result r{};
    // count first when the caller's bound is generous: the buffer is sized by what the tree holds
    unsigned long long cap = max_solutions;
    if (cap > 4096) {
        const int rc0 = dq_solve_tree(cache_.handle, &o, &r, nullptr);
        if (rc0 != DQ_OK) throw b200::Error(rc0, dq_last_error());
        if (r.n_solutions > max_solutions) throw b200::Error(DQ_ERR_NOMEM, "more solutions than max_solutions");
        cap = r.n_solutions;
    }
    std::vector<int32_t> flat((size_t)std::max<unsigned long long>(cap, 1) * (size_t)std::max(nv, 1));
    uint64_t n = 0;
    const int rc = dq_enumerate_solutions(cache_.handle, &o, &r, flat.data(), cap, &n);
    if (rc != DQ_OK) throw b200::Error(rc, dq_last_error());
    if (rep) { rep->tree = r; rep->compiled_fresh = fresh; }
    out.clear();
    out.reserve((size_t)n);
    for (uint64_t i = 0; i < n; i++) out.emplace_back(flat.begin() + (size_t)i * nv, flat.begin() + (size_t)(i + 1) * nv);
}

inline bool CSP::ForwardCheckingStep(Assignment& a) const {
    if (a.IsComplete()) return true;                 // also the reference's answer for a second call after success
    return SolveB200(a, DQ_MODE_FIRST, b200::SolveOptions(), nullptr);
}

namespace b200 {

/* First solution with explicit engine / partition options and the device-side report. */
inline bool Solve(const CSP& csp, Assignment& a, const SolveOptions& opt = SolveOptions(), SolveReport* rep = nullptr) {
    if (a.IsComplete()) return true;
    return csp.SolveB200(a, DQ_MODE_FIRST, opt, rep);
}

/* All solutions: exhausts the tree.  The reference has no such mode; the equivalent on the
 * reference is a counting Constraint linked last to the last variable that always fails
 * (SURVEY.md §8c) — node counts agree with that construction.  Returns the solution count of this
 * partition; `a` receives the DFS-first solution if the partition holds one. */
inline unsigned long long CountAll(const CSP& csp, Assignment& a, const SolveOptions& opt = SolveOptions(),
                                   SolveReport* rep = nullptr) {
    SolveReport local;
    SolveReport* r = rep ? rep : &local;
    csp.SolveB200(a, DQ_MODE_COUNT_ALL, opt, r);
    return r->tree.n_solutions;
}

/* Every solution, in the order the search visits them (the reference's static variable order and domain value
 * order): out[i][v] = value of variable v in the i-th solution.  On the reference the equivalent is a counting
 * Constraint linked last to the last variable that snapshots inst_vars on every Evaluate (SURVEY.md §8c).  Throws
 * Error(DQ_ERR_NOMEM) when the tree holds more than max_solutions.  `a` is left untouched. */
inline void EnumerateAll(const CSP& csp, const Assignment& a, std::vector<std::vector<int> >& out,
                         unsigned long long max_solutions = 1000000ULL, const SolveOptions& opt = SolveOptions(),
                         SolveReport* rep = nullptr) {
    csp.EnumerateB200(a, opt, rep, out, max_solutions);
}

/* Complete Assignments answer true without a device call; the others go to the device in one dq_solve_models call.  A
 * pair whose descriptor equals its CSP's cached one uses the cached handle; the first other descriptor of a CSP whose
 * cache no earlier pair uses replaces the cache; any further one gets a handle that lives for this call only. */
inline std::vector<bool> SolveAll(const std::vector<const CSP*>& csps, const std::vector<Assignment*>& as,
                                  std::vector<SolveReport>* reps) {
    if (csps.size() != as.size()) throw Error(DQ_ERR_INVALID, "SolveAll takes one Assignment per CSP");
    const size_t n = csps.size();
    std::vector<bool> out(n, false);
    if (reps) reps->assign(n, SolveReport());
    struct CallHandles {
        std::vector<dq_model*> h;
        ~CallHandles() { for (dq_model* p : h) dq_free(p); }
    } call_handles;
    struct Seen { const CSP* csp; std::vector<int32_t> key; dq_model* h; };
    std::vector<Seen> seen;                                   // descriptors given a handle in this call
    std::vector<size_t> todo;
    std::vector<dq_model*> handles;
    std::vector<int> resumed;
    std::vector<char> fresh;
    std::vector<size_t> off(1, 0);
    for (size_t i = 0; i < n; i++) {
        const CSP& csp = *csps[i];
        Assignment& a = *as[i];
        if (a.IsComplete()) { out[i] = true; continue; }     // also the reference's answer for a second call after success
        const int r = csp.CheckResumable(a);
        CSP::Lowered l;
        csp.Lower(a, l);
        dq_model* h = nullptr;
        bool compiled = false;
        for (const Seen& s : seen) if (s.csp == &csp && s.key == l.key) { h = s.h; break; }
        if (!h) {
            bool cache_used = false;
            for (const Seen& s : seen) if (s.csp == &csp && s.h == csp.cache_.handle) cache_used = true;
            if (csp.cache_.handle && csp.cache_.key == l.key) h = csp.cache_.handle;
            else if (!cache_used) {
                csp.cache_.Drop();
                csp.cache_.handle = h = CSP::Compile(l, (int)csp.vars.size());
                csp.cache_.key = l.key;
                compiled = true;
            } else {
                h = CSP::Compile(l, (int)csp.vars.size());
                call_handles.h.push_back(h);
                compiled = true;
            }
            seen.push_back(Seen{&csp, l.key, h});
        }
        todo.push_back(i);
        handles.push_back(h);
        resumed.push_back(r);
        fresh.push_back(compiled);
        off.push_back(off.back() + csp.vars.size());
    }
    if (todo.empty()) return out;
    const size_t m = todo.size();
    std::vector<int32_t> outcome(m), first(std::max<size_t>(off.back(), 1));
    std::vector<uint64_t> sols(m), nodes(m);
    int64_t n_split = 0;
    dq_tree_opts o{};
    o.mode = DQ_MODE_FIRST;
    o.part_count = 1;
    const int rc = dq_solve_models(handles.data(), (int64_t)m, &o, outcome.data(), sols.data(), nodes.data(), first.data(),
                                   &n_split, nullptr);
    if (rc != DQ_OK) throw Error(rc, dq_last_error());
    for (size_t k = 0; k < m; k++) {
        const size_t i = todo[k];
        const bool have = outcome[k] == DQ_SAT;
        out[i] = csps[i]->FinishB200(*as[i], nodes[k], have, first.data() + off[k], resumed[k]);
        if (reps) {
            SolveReport& rep = (*reps)[i];
            rep.tree.outcome = outcome[k];
            rep.tree.n_solutions = sols[k];
            rep.tree.n_nodes = nodes[k] - (uint64_t)resumed[k];
            rep.tree.first_key = have ? 0 : UINT64_MAX;
            rep.compiled_fresh = fresh[k] != 0;
        }
    }
    return out;
}

}  // namespace b200
}  // namespace dequan

#endif /* DEQUAN_DROPIN_H */
