// Flat SSA program: what the Expr tree is lowered to before either GPU back end sees it.
//
// One program serves all three colour channels.  Structurally equal sub-expressions are one value
// (hash-consing), which subsumes the reference's `Let` + `Cache` sharing (reference
// src/cache.rs:23-42) and its var_fixer pre-pass (reference src/var_fixer.rs:74-82); constants are
// folded on the host with the same IEEE operations and the host libm the reference would call.
// No algebraic rewriting is done: every remaining operation is one the reference performs, on the
// same operand values, so results are bit-identical wherever the device operation is IEEE-exact.
#pragma once
#include <cmath>
#include <cstdint>
#include <string>
#include <vector>

#include "expr.hpp"

namespace maray {

enum Op : uint8_t {
    OP_CONST = 0, OP_X, OP_Y,
    OP_NEG, OP_ABS, OP_RECIP, OP_SQRT, OP_STEP, OP_SIN, OP_EXP, OP_LN,
    OP_ADD, OP_MUL, OP_MAX, OP_MIN,
    OP_TEX,          // a = x coordinate, b = y coordinate, imm = texture*4 + channel
    OP_APP,          // custom runtime: maray_app(ctx, ctx_bytes, imm, a, b), imm = the App id (never folded)
    OP_COUNT
};

inline bool op_is_unary(Op o) { return o >= OP_NEG && o <= OP_LN; }
inline bool op_is_binary(Op o) { return o >= OP_ADD && o <= OP_APP; }
const char* op_name(Op o);

enum Dep : uint8_t { DEP_CONST = 0, DEP_X = 1, DEP_Y = 2, DEP_XY = 3 };

struct Node {
    Op op;
    uint8_t dep;       // Dep bits
    uint32_t a, b;     // operand value ids (unused: 0)
    uint32_t imm;      // OP_TEX, OP_APP only
    double k;          // OP_CONST only
};

struct TextureDim { uint32_t w, h; };

// What `App(id, a, b)` calls (reference src/lib.rs:72-98, 664-668): the default texture runtime (textures::functions,
// five functions per texture, width and height folded on the host), or a custom runtime of n_functions functions that
// the host supplies as CUDA source (maray_cuda_set_functions): every App is an OP_APP value, evaluated at run time.
struct RuntimeDesc {
    std::vector<TextureDim> textures;
    bool custom = false;
    uint32_t n_functions = 0;
};

// Programs with at least this many sin/exp/ln values evaluate them out of line (the NVRTC back end
// calls batched helper functions instead of inlining every body) and get their schedule batched.
constexpr uint32_t kOutOfLineTranscendentals = 2048;

struct ProgramStats {
    uint64_t tree_nodes = 0;        // nodes of the three channel trees as stored
    uint64_t dag_nodes = 0;         // values after hash-consing, reachable from the channel roots
    uint64_t n_const = 0, n_x = 0, n_y = 0, n_xy = 0;
    uint64_t op_count[OP_COUNT] = {0};   // per op, non-constant values only
    uint32_t depth = 0;             // longest operand chain
    uint32_t max_live = 0;          // most values simultaneously live under the chosen schedule
    uint32_t n_batches = 0, n_batched = 0;   // transcendental batches formed / values in them
    uint32_t schedule_kind = 0;     // 0 depth-first, 1 the scene's own order, 2/3 greedy list schedule (newest/oldest first)
};

struct Program {
    std::vector<Node> nodes;        // topological: operands precede users; every node is reachable
    uint32_t root[3] = {0, 0, 0};   // R, G, B
    std::vector<uint32_t> order;    // evaluation order of the non-constant values (a schedule)
    // batch[i] for order[i]: 0 = not batched; otherwise consecutive entries with the same non-zero id
    // are sin/exp/ln values of one kind that are mutually independent and whose operands all precede
    // the first of them -- they may be evaluated together (instruction-level parallelism, one call).
    std::vector<uint32_t> batch;
    uint32_t n_textures = 0;        // textures the program was lowered against
    ProgramStats stats;
};

// Lowers the three channels of `scene`.  `Let` binds lexically (inner scopes see outer ones; a
// definition is lowered on first use in the scope of its own `Let`, so definition order does not
// matter, like the reference interpreter's by-name lookup, reference src/cache.rs:30-38).
// Errors (returned as false + message) instead of the reference's silent NaN / panic:
//   unbound variable (reference src/cache.rs:40 yields NaN), cyclic definitions,
//   App id >= the runtime's function count: 5 * textures.size(), or n_functions of a custom runtime
//   (reference src/lib.rs:665 panics on the index).
bool lower_scene(const Scene& scene, const RuntimeDesc& rt, Program* out, std::string* err);

// ---- operation semantics shared by host constant folding (reference src/lib.rs:632-669) --------
// f64::max / f64::min: NaN-ignoring; on an equal-compare tie (incl. +0/-0) the first operand wins
// (x86-64 lowering of llvm.maxnum: select(isnan(a), b, MAXSD(b, a)); see DESIGN.md "Semantics").
inline double sem_max(double a, double b) { return (a != a) ? b : ((b > a) ? b : a); }
inline double sem_min(double a, double b) { return (a != a) ? b : ((b < a) ? b : a); }
inline double sem_step(double v) { return (v >= 0.0) ? 1.0 : 0.0; }

}  // namespace maray
