// dq_model.hpp — host-side compiled model ("flat constraint/variable table").
//
// dq_compile() lowers a dq_model_desc (the flattened form of dequan::CSP, reference
// dequan.h:328-355) into var-id-space tables the CUDA engines walk:
//   * value lists  : per variable, the domain in the reference's ITERATION order
//                    (Values: list order, Ranges: ascending — dequan.h:544-563); bit b of a
//                    domain word stands for values[v][b].
//   * static order : Assignment::Reset's sort (dequan.h:376-394).
//   * arc entries  : per variable x, what assigning x=values[x][b] does to each neighbour q,
//                    i.e. the composition of every linked constraint's AplyArcConsistency
//                    (dequan.h:631-694, 710-743, 915-939) restricted to the pair (x,q), in link
//                    order, as bit masks (see EntryKind).
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "dequan_b200.h"

namespace dq {

constexpr int kMaxVars = 1022;     // q fits 10 bits with room to spare in the 16-bit id field; 0xFFFF reserved
constexpr int kMaxGraphVertices = 254;   // batch graphs: vertex ids are bytes in the edge list
constexpr int kMaxDom = 64;        // one domain word: 32 bits, or 64 for models whose largest domain has 33..64 values
typedef uint64_t Mask;             // host-side masks are always 64-bit; the upload narrows them for 32-bit models

// What one (x -> q) entry does to q's state (D = domain bits, F = "fails validation" bits):
enum EntryKind : uint32_t {
    K_NE_SAME = 0,   // D &= ~(1<<b)            NotEqual,0 / AllDifferent between identical value lists
    K_AND     = 1,   // D &= mask[b]            any composition of Exclude/ExcludeInf/ExcludeSup
    K_WEQ     = 2,   // if (D & mask[b]) D &= mask[b]; else F = ~0   Domain::Intersect(val) is a no-op when
                     //                          val is absent (dequan.h:957-984) and Evaluate fails later
    K_CHK     = 3    // F |= mask[b]            check-only constraints (OrRange, user tables): values of q
                     //                          that ValidateVarConstraints (dequan.h:573-587) will reject
};
// entry word (uint32): q (16 bits) | kind<<16 | flags
constexpr uint32_t ENT_Q_MASK    = 0xFFFFu;
constexpr int      ENT_KIND_SHIFT = 16;
constexpr uint32_t ENT_FORCE_D   = 1u << 18;  // trail D[q] unconditionally (first of several entries on q)
constexpr uint32_t ENT_FORCE_F   = 1u << 19;
constexpr uint32_t ENT_NOTRAIL_D = 1u << 20;  // later entry on the same q: the first one already trailed it
constexpr uint32_t ENT_NOTRAIL_F = 1u << 21;
constexpr uint32_t ENT_SKIP      = 1u << 22;  // padding so that same-q entries land in different 32-lane passes
constexpr uint32_t ENT_FIRST     = 1u << 23;  // K_AND on a value list with duplicates: mask[b] = the positions that hold the
                                              // excluded value, and only the FIRST one still present goes
                                              // (Domain::Exclude erases the first match, dequan.h:989-996, SURVEY.md Q2)
constexpr uint32_t ENT_FLAGS     = ENT_FORCE_D | ENT_FORCE_F | ENT_NOTRAIL_D | ENT_NOTRAIL_F | ENT_SKIP | ENT_FIRST;

enum ModelClass : int32_t {
    CLASS_GENERIC = 0,     // anything the entry table can express
    CLASS_NE_SAME = 1,     // only K_NE_SAME entries (Sudoku, graph colouring): no mask table needed
    CLASS_QUEENS  = 2,     // N-Queens structure: dense NotEqual with offsets {0, +-(j-i)} on [0,N)
    CLASS_SUDOKU9 = 3      // 81 variables on 1..9, pairwise different over the 27 rows / columns / boxes
};

struct CompiledModel {
    int nv = 0;
    int kmax = 0;                              // largest domain size
    bool wide() const { return kmax > 32; }    // 64-bit domain words on the device (generic tree engine only)
    std::vector<std::vector<int32_t>> values;  // [nv][k_v]
    std::vector<Mask> dom0;                    // [nv] initial domain bits
    std::vector<int32_t> order;                // [nv] position -> var id (Reset order, or the caller's assign_order)
    std::vector<int32_t> pos_of;               // [nv] var id -> position
    bool caller_order = false;                 // `order` is the caller's assign_order: batches keep it for every instance
    std::vector<uint32_t> ent_off;             // [nv+1]
    std::vector<uint32_t> ent;                 // [n_ent]
    std::vector<uint32_t> ent_moff;            // [n_ent] index into masks (kinds != K_NE_SAME)
    std::vector<Mask> masks;                   // mask tables, kmax words per entry that needs one
    bool has_f = false;                        // any K_WEQ / K_CHK entry
    bool has_table = false;                    // any entry other than K_NE_SAME
    int trail_bound = 0;                       // max live trail entries along one DFS path
    int model_class = CLASS_GENERIC;
    int queens_n = 0;
    std::vector<int32_t> distinct_sizes;       // sorted distinct initial domain sizes (batch re-ordering)
    // Small-model tables for the register-resident tree engine (nv <= 32, every pair at most AND -> WEQ -> CHK):
    // position space, [pos(x)][value index][pos(q)]: what x = value does to q.  Empty when the model does not qualify.
    bool small_ok = false;
    std::vector<uint32_t> small_and;           // AND mask (all ones: q untouched)
    std::vector<uint32_t> small_weq;           // weak-equal mask, valid where the bit of pos(q) is set in small_weq_on[pos(x)][value]
    std::vector<uint32_t> small_weq_on;        // [pos(x)][value index]
    std::vector<uint32_t> small_chk;           // values of q that will fail validation
};

// Returns DQ_OK or a negative dq_status; on failure `err` says why.
int compile_model(const dq_model_desc* desc, CompiledModel& out, std::string& err);

}  // namespace dq
