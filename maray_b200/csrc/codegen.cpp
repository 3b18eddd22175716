// SSA program -> CUDA C++ source for NVRTC.  See codegen.hpp.
#include "codegen.hpp"

#include <algorithm>
#include <cinttypes>
#include <functional>
#include <cmath>
#include <cstdio>
#include <cstring>

namespace maray {

const char* const kJitKernelName = "maray_jit";

namespace {

// The text of device_sem.cuh, embedded by the build (csrc/Makefile: device_sem_text.inc).
const char* const kDeviceSemText =
#include "device_sem_text.inc"
    ;

void append_const(std::string& s, double v) {
    char buf[64];
    uint64_t bits;
    std::memcpy(&bits, &v, 8);
    if (v != v || v - v != 0.0) {
        // NaN / infinity: no literal form; rebuild from the bit pattern.
        std::snprintf(buf, sizeof buf, "__longlong_as_double(0x%016" PRIx64 "LL)", bits);
    } else {
        std::snprintf(buf, sizeof buf, "%a", v);   // hex float: exact
        if (buf[0] == '-') { s += "(" ; s += buf; s += ")"; return; }
    }
    s += buf;
}

constexpr uint32_t kScratchRows = 8;   // argument rows of the batched sin/exp/ln scratch (as many result rows follow)

struct Emitter {
    const Program& P;
    bool inline_trans;
    const std::vector<int32_t>* bank_index;   // value id -> index in the __constant__ table, or -1
    std::string helper_suffix;      // which instance of the batch helpers this function calls ("" or "_sK")
    // Values that are exactly +0.0 or 1.0 at every pixel (see find_booleans): kind 1 = boolean,
    // kind 2 = the NOT pattern `1 + -(b)`.  Emitted as `bool` logic plus a double shadow.
    const std::vector<uint8_t>* boolean = nullptr;
    // Sines that are only ever asked for their sign (see find_sign_only_sines): never materialised.
    const std::vector<uint8_t>* sign_only = nullptr;
    bool is_sign_only(uint32_t id) const { return sign_only && (*sign_only)[id]; }

    bool is_bool(uint32_t id) const { return boolean && (*boolean)[id]; }
    void bool_operand(std::string& s, uint32_t id) const {
        const Node& n = P.nodes[id];
        if (n.op == OP_CONST) { s += (n.k != 0.0) ? "true" : "false"; return; }
        char buf[16];
        std::snprintf(buf, sizeof buf, "b%u", id);
        s += buf;
    }
    // `const bool bN = vN != 0.0;` after a boolean value arrived as a double (frame import)
    void bool_from_double(std::string& s, uint32_t id) const {
        if (!is_bool(id)) return;
        char buf[64];
        std::snprintf(buf, sizeof buf, "  const bool b%u = v%u != 0.0;\n", id, id);
        s += buf;
    }

    void operand(std::string& s, uint32_t id) const {
        const Node& n = P.nodes[id];
        if (n.op == OP_CONST) {
            if (bank_index && (*bank_index)[id] >= 0) {
                char kb[24];
                std::snprintf(kb, sizeof kb, "MRK(%d)", (*bank_index)[id]);
                s += kb;
            } else append_const(s, n.k);
            return;
        }
        if (n.op == OP_X) { s += "X"; return; }
        if (n.op == OP_Y) { s += "Y"; return; }
        char buf[16];
        std::snprintf(buf, sizeof buf, "v%u", id);
        s += buf;
    }

    // Emits order[i..j) -- one batch of same-kind transcendentals -- as out-of-line batch calls: arguments
    // -> this thread's scratch rows, one leaf call for the whole batch, results back (rows: kScratchRows;
    // lower.cpp's kBatchMax never exceeds it).  The evaluations inside a call are independent, which is where
    // the FP64 pipe gets its instruction-level parallelism in transcendental-heavy programs.
    void batch_calls(std::string& s, const std::vector<uint32_t>& order, size_t i, size_t j) const {
        const char* fn = P.nodes[order[i]].op == OP_SIN ? "sin" : (P.nodes[order[i]].op == OP_EXP ? "exp" : "log");
        char buf[96];
        while (i < j) {
            const size_t k = std::min<size_t>(j - i, kScratchRows);
            if (k == 1) { statement(s, order[i]); i++; continue; }
            for (size_t m = 0; m < k; m++) {
                std::snprintf(buf, sizeof buf, "  MR_S(%zu) = ", m);
                s += buf; operand(s, P.nodes[order[i + m]].a); s += ";\n";
            }
            std::snprintf(buf, sizeof buf, "  if (mr_%s_batch%s(%zuu)) mr_%s_fix%s(%zuu);\n", fn, helper_suffix.c_str(), k, fn,
                          helper_suffix.c_str(), k);
            s += buf;
            for (size_t m = 0; m < k; m++) {
                std::snprintf(buf, sizeof buf, "  const double v%u = MR_R(%zu);\n", order[i + m], m);
                s += buf;
            }
            i += k;
        }
    }

    void statement(std::string& s, uint32_t id) const {
        const Node& n = P.nodes[id];
        if (n.op == OP_X || n.op == OP_Y) return;   // kernel arguments
        if (is_sign_only(id)) return;               // its one consumer, a step, evaluates mr_sin_ge0 of the argument
        char buf[160];
        if (is_bool(id)) {
            // 0/1-valued: compares and bit logic instead of FP64 multiplies, min/max and selects.  The
            // double shadow is what every non-boolean consumer reads; unused shadows are dead code.
            std::snprintf(buf, sizeof buf, "  const bool b%u = ", id);
            s += buf;
            switch (n.op) {
            case OP_STEP:
                if (is_sign_only(n.a) && P.nodes[n.a].op == OP_SIN) {
                    s += "mr_sin_ge0("; operand(s, P.nodes[n.a].a); s += ")";         // step(sin(u)): the sign is enough
                } else if (is_sign_only(n.a)) {                                       // step(v + c)  ==  v >= -c  ==  -v <= c  (finite constant c)
                    const Node& ad = P.nodes[n.a];
                    const bool ca = P.nodes[ad.a].op == OP_CONST;
                    s += "(-("; operand(s, ca ? ad.b : ad.a); s += ") <= "; operand(s, ca ? ad.a : ad.b); s += ")";   // -v <= c: c stays a bank operand
                } else { s += "("; operand(s, n.a); s += " >= 0.0)"; }                // NaN -> false, -0.0 -> true
                break;
            case OP_ADD: {                                                           // 1 + -(b)  ==  !b
                const uint32_t neg = P.nodes[n.a].op == OP_NEG ? n.a : n.b;
                s += "!"; bool_operand(s, P.nodes[neg].a);
            } break;
            case OP_MUL: case OP_MIN: s += "("; bool_operand(s, n.a); s += " && "; bool_operand(s, n.b); s += ")"; break;
            case OP_MAX: s += "("; bool_operand(s, n.a); s += " || "; bool_operand(s, n.b); s += ")"; break;
            default: s += "false"; break;
            }
            std::snprintf(buf, sizeof buf, ";\n  const double v%u = b%u ? 1.0 : 0.0;\n", id, id);
            s += buf;
            return;
        }
        std::snprintf(buf, sizeof buf, "  const double v%u = ", id);
        s += buf;
        auto un = [&](const char* pre, const char* post) { s += pre; operand(s, n.a); s += post; };
        auto bin = [&](const char* pre, const char* mid, const char* post) {
            s += pre; operand(s, n.a); s += mid; operand(s, n.b); s += post;
        };
        switch (n.op) {
        case OP_NEG: un("-", ""); break;
        case OP_ABS: un("fabs(", ")"); break;
        case OP_RECIP: un("mr_recip(", ")"); break;
        case OP_SQRT: un("mr_sqrt(", ")"); break;
        case OP_STEP: un("mr_step(", ")"); break;
        case OP_SIN: un(inline_trans ? "mr_sin(" : "mr_sin_call(", ")"); break;
        case OP_EXP: un(inline_trans ? "mr_exp(" : "mr_exp_call(", ")"); break;
        case OP_LN: un(inline_trans ? "mr_log(" : "mr_log_call(", ")"); break;
        case OP_ADD: bin("", " + ", ""); break;
        case OP_MUL: bin("", " * ", ""); break;
        case OP_MAX: bin("mr_max(", ", ", ")"); break;
        case OP_MIN: bin("mr_min(", ", ", ")"); break;
        case OP_TEX: {
            uint32_t img = n.imm / 4, k = n.imm % 4;
            std::snprintf(buf, sizeof buf, "mr_tex(T[%u].data, T[%u].w, T[%u].h, %uu, ", img, img, img, k);
            bin(buf, ", ", ")");
            break;
        }
        default: s += "0.0"; break;
        }
        s += ";\n";
    }
};

}  // namespace

namespace {
// Values that are exactly +0.0 or 1.0 whatever the pixel: step(..), the constants 0 and 1, products /
// min / max of two such values (AND, AND, OR), and `1 + -(b)` (NOT).  All of these identities are exact
// in IEEE arithmetic (0*1 = +0, 1 + -1 = +0 under round-to-nearest, min/max of {+0, 1} never see a NaN
// or a -0), so evaluating them as boolean logic changes no bit of any channel.  Scenes built from
// Maray's set algebra (range, set_and/or/xor/inv, inside_triangle; reference src/lib.rs:869-913,
// 1094-1097) are mostly made of them: chess has 1 482 steps, 768 min, 256 max.
std::vector<uint8_t> find_booleans(const Program& prog) {
    const size_t n = prog.nodes.size();
    std::vector<uint8_t> kind(n, 0);
    auto is_one = [&](uint32_t v) { return prog.nodes[v].op == OP_CONST && prog.nodes[v].k == 1.0; };
    auto neg_of_bool = [&](uint32_t v) { return prog.nodes[v].op == OP_NEG && kind[prog.nodes[v].a]; };
    for (size_t i = 0; i < n; i++) {
        const Node& nd = prog.nodes[i];
        switch (nd.op) {
        case OP_CONST: {
            uint64_t bits;
            std::memcpy(&bits, &nd.k, 8);
            kind[i] = (bits == 0 || nd.k == 1.0) ? 1 : 0;          // +0.0 only: -0.0 is not a boolean
        } break;
        case OP_STEP: kind[i] = 1; break;
        case OP_MUL: case OP_MIN: case OP_MAX: kind[i] = (kind[nd.a] && kind[nd.b]) ? 1 : 0; break;
        case OP_ADD: kind[i] = ((is_one(nd.a) && neg_of_bool(nd.b)) || (neg_of_bool(nd.a) && is_one(nd.b))) ? 2 : 0; break;
        default: break;
        }
    }
    return kind;
}

// Values that are only ever asked for their sign, by one step, and are therefore never materialised.
// step(sin(u)) where nothing else reads the sine -- Maray's `chess` is made of these (reference src/lib.rs:969-973) --
// only needs the SIGN of the sine, which the argument reduction already decides: the polynomial, its table loads and
// the quadrant selects are skipped (device_libm.cuh mr_sin_ge0; per sine 6 FP64 instructions instead of 16).  Exact:
// mr_sin_ge0(u) == (mr_sin(u) >= 0.0) for every u, so no pixel changes.
std::vector<uint8_t> find_sign_only_sines(const Program& prog, const std::vector<uint8_t>& booleans) {
    const size_t n = prog.nodes.size();
    std::vector<uint32_t> uses(n, 0);
    for (size_t i = 0; i < n; i++) {
        const Node& nd = prog.nodes[i];
        if (op_is_unary(nd.op) || op_is_binary(nd.op)) uses[nd.a]++;
        if (op_is_binary(nd.op)) uses[nd.b]++;
    }
    for (int c = 0; c < 3; c++) uses[prog.root[c]]++;
    std::vector<uint8_t> mark(n, 0);
    for (size_t i = 0; i < n; i++) {
        const Node& nd = prog.nodes[i];
        if (nd.op != OP_STEP || !booleans[i] || uses[nd.a] != 1) continue;
        const Node& arg = prog.nodes[nd.a];
        if (arg.op == OP_SIN) mark[nd.a] = 1;
        // step(v + c) with a finite constant c is the comparison v >= -c: the rounded sum is zero exactly when v == -c
        // (sums of doubles never underflow to zero), otherwise it has the sign of the exact sum; v = +-inf and NaN give
        // the same answer both ways because c is finite.  (Two variables would not do: inf - inf is NaN, inf >= inf is true.)
        if (arg.op == OP_ADD && !booleans[nd.a]) {
            const Node& x = prog.nodes[arg.a];
            const Node& y = prog.nodes[arg.b];
            const bool cx = x.op == OP_CONST && x.k - x.k == 0.0, cy = y.op == OP_CONST && y.k - y.k == 0.0;
            if (cx != cy) mark[nd.a] = 1;
        }
    }
    return mark;
}

// Guarded regions of the straight-line kernel.  For a boolean AND G = a && b (OP_MUL or OP_MIN of two booleans),
// `false && anything == false`: when one operand (the guard) is false on every lane of a warp, the other (the body)
// need not be evaluated at all, provided every value it consists of is read only through that operand edge of G.
// Such a value is post-dominated by the edge: every path from it to the program's outputs passes through it.  With one
// pseudo-node per operand edge of each AND, the body of an edge is the edge's subtree of the post-dominator tree of
// the use graph, so bodies of different edges are nested or disjoint and the regions form a tree.  Every read counts:
// both operands, the three channel roots, and the NOT form's extra read of b (`1 + -(b)` is emitted as `!b`).
struct GuardRegion {
    uint32_t guard;    // evaluated in place, before the region
    uint32_t body;     // evaluated inside `if (mr_warp_any(guard))`
};
struct GuardRegions {
    std::vector<GuardRegion> regions;
    std::vector<int32_t> owner;       // value -> innermost region whose body holds it, or -1
    std::vector<int32_t> rooted_at;   // value -> the region whose AND it is, or -1
};

GuardRegions find_guard_regions(const Program& prog, const std::vector<uint8_t>& booleans, const std::vector<uint8_t>& sign_only,
                                const std::function<uint32_t(uint32_t)>& not_operand) {
    const uint32_t n = uint32_t(prog.nodes.size());
    auto is_value = [&](uint32_t id) { const Op o = prog.nodes[id].op; return o != OP_CONST && o != OP_X && o != OP_Y; };
    // candidates: ANDs of two booleans, neither a constant
    std::vector<int32_t> cand(n, -1);
    std::vector<uint32_t> cands;
    for (uint32_t i = 0; i < n; i++) {
        const Node& nd = prog.nodes[i];
        if ((nd.op == OP_MUL || nd.op == OP_MIN) && booleans[i] && is_value(nd.a) && is_value(nd.b)) {
            cand[i] = int32_t(cands.size());
            cands.push_back(i);
        }
    }
    GuardRegions out;
    out.owner.assign(n, -1);
    out.rooted_at.assign(n, -1);
    if (cands.empty()) return out;
    // extended nodes: values 0..n-1, EXIT = n, the pseudo-node of edge k of candidate c = n + 1 + 2c + k
    const uint32_t exit_node = n, n_ext = n + 1 + 2 * uint32_t(cands.size());
    auto edge_node = [&](uint32_t c, uint32_t k) { return n + 1 + 2 * c + k; };
    // successors (readers) of every value, in CSR form
    std::vector<uint32_t> deg(n + 1, 0), succ;
    auto for_each_read = [&](auto&& fn) {   // fn(operand, successor)
        for (uint32_t r = 0; r < n; r++) {
            const Node& nd = prog.nodes[r];
            if (!is_value(r)) continue;
            if (cand[r] >= 0) { fn(nd.a, edge_node(uint32_t(cand[r]), 0)); fn(nd.b, edge_node(uint32_t(cand[r]), 1)); continue; }
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) fn(nd.a, r);
            if (op_is_binary(nd.op)) fn(nd.b, r);
            if (uint32_t x = not_operand(r); x != UINT32_MAX) fn(x, r);
        }
        for (int c = 0; c < 3; c++) fn(prog.root[c], exit_node);
    };
    for_each_read([&](uint32_t v, uint32_t) { deg[v + 1]++; });
    for (uint32_t i = 0; i < n; i++) deg[i + 1] += deg[i];
    succ.resize(deg[n]);
    {
        std::vector<uint32_t> fill(deg.begin(), deg.end() - 1);
        for_each_read([&](uint32_t v, uint32_t s) { succ[fill[v]++] = s; });
    }
    // immediate post-dominators: readers come after their operands, so one pass from the outputs backwards suffices
    std::vector<uint32_t> ipdom(n_ext, exit_node), depth(n_ext, 0);
    auto meet = [&](uint32_t x, uint32_t y) {
        while (x != y) {
            if (depth[x] < depth[y]) std::swap(x, y);
            x = ipdom[x];
        }
        return x;
    };
    for (uint32_t v = n; v-- > 0;) {
        // A value nothing reads (none exist: every node is reachable from a root) keeps EXIT; so would its edge
        // pseudo-nodes if it were an AND, which is harmless -- only values as dead as it could fall under them.
        if (!is_value(v) || deg[v] == deg[v + 1]) continue;
        uint32_t p = succ[deg[v]];
        for (uint32_t e = deg[v] + 1; e < deg[v + 1]; e++) p = meet(p, succ[e]);
        ipdom[v] = p;
        depth[v] = depth[p] + 1;
        if (cand[v] >= 0)
            for (uint32_t k = 0; k < 2; k++) {
                ipdom[edge_node(uint32_t(cand[v]), k)] = v;
                depth[edge_node(uint32_t(cand[v]), k)] = depth[v] + 1;
            }
    }
    // weight of each post-dominator subtree: about what evaluating it costs per pixel
    auto weight = [&](uint32_t v) -> uint32_t {
        switch (prog.nodes[v].op) {
        case OP_NEG: return 0;                                   // folded into its reader's operand
        case OP_SIN: case OP_EXP: case OP_LN: return !sign_only.empty() && sign_only[v] ? 7 : 16;
        default: return 1;
        }
    };
    std::vector<uint64_t> sub(n_ext, 0);
    for (uint32_t v = 0; v < n; v++) {
        if (!is_value(v)) continue;
        if (cand[v] >= 0) sub[v] += sub[edge_node(uint32_t(cand[v]), 0)] + sub[edge_node(uint32_t(cand[v]), 1)];
        sub[v] += weight(v);
        sub[ipdom[v]] += sub[v];
    }
    // regions and their members, from the outputs backwards: a value belongs to the innermost region of its post-dominator
    std::vector<int32_t> ext_owner(n_ext, -1);
    for (uint32_t v = n; v-- > 0;) {
        if (!is_value(v)) continue;
        out.owner[v] = ext_owner[v] = ext_owner[ipdom[v]];
        if (cand[v] < 0) continue;
        const uint32_t c = uint32_t(cand[v]);
        const uint32_t kb = sub[edge_node(c, 1)] > sub[edge_node(c, 0)] ? 1 : 0;   // the dearer operand is the body
        ext_owner[edge_node(c, 0)] = ext_owner[edge_node(c, 1)] = ext_owner[v];
        if (sub[edge_node(c, kb)] >= kGuardBodyMinWeight) {
            const Node& nd = prog.nodes[v];
            out.rooted_at[v] = int32_t(out.regions.size());
            ext_owner[edge_node(c, kb)] = int32_t(out.regions.size());
            out.regions.push_back({kb ? nd.a : nd.b, kb ? nd.b : nd.a});
        }
    }
    return out;
}

// Common generator.  Three forms:
//   * one kernel (programs up to opt.segment_values values);
//   * larger programs, opt.chain: one KERNEL per segment, each its own translation unit (modules[s]); values
//     that cross a cut travel through a frame in global memory, F[slot * FS + pixel] (slot-major, so a warp's
//     accesses are coalesced).  The units share nothing, so NVRTC compiles them concurrently and nothing is
//     linked, no segment pays a call ABI, and every kernel has the whole register file;
//   * larger programs, !opt.chain: __noinline__ segment functions inside ONE unit with a per-thread frame in
//     local memory (round 1's form; what generate_cuda_source returns).
std::vector<std::string> generate(const Program& prog, const CodegenOptions& opt, CodegenInfo* info) {
    const std::vector<uint32_t>& order = prog.order;
    const std::vector<uint32_t> order_batch =
        prog.batch.size() == prog.order.size() ? prog.batch : std::vector<uint32_t>(prog.order.size(), 0);
    uint64_t n_trans = prog.stats.op_count[OP_SIN] + prog.stats.op_count[OP_EXP] + prog.stats.op_count[OP_LN];

    const uint32_t cut_off = opt.segment_values ? opt.segment_values : 4096;
    bool segmented = order.size() > cut_off;
    bool chain = segmented && opt.chain;
    const uint32_t seg_len = chain ? std::max(256u, std::min(cut_off, opt.chain_segment_values)) : cut_off;
    if (chain && order.size() <= seg_len) segmented = chain = false;      // a chain of one kernel is a plain kernel
    // chain: cut into equal parts (the last kernel is not a stub)
    const uint32_t n_seg = segmented ? uint32_t((order.size() + seg_len - 1) / seg_len) : 1;
    const uint32_t seg_size = segmented ? uint32_t((order.size() + n_seg - 1) / n_seg) : uint32_t(order.size());
    auto seg_lo = [&](uint32_t s) { return std::min(order.size(), size_t(s) * (chain ? seg_size : seg_len)); };
    auto seg_hi = [&](uint32_t s) { return std::min(order.size(), size_t(s + 1) * (chain ? seg_size : seg_len)); };

    // __constant__ table of the constants a translation unit uses (64 KiB bank: at most 8000 entries; the
    // rest stay literals).  Stored as bit patterns so NaN/infinity need no special spelling.
    struct Bank { std::vector<int32_t> index; std::vector<uint64_t> bits; };
    auto make_bank = [&](size_t lo, size_t hi, bool everything) {
        Bank bk;
        bk.index.assign(prog.nodes.size(), -1);
        if (!opt.constants_in_bank) return bk;
        auto want = [&](uint32_t id) {
            if (prog.nodes[id].op != OP_CONST || bk.index[id] >= 0 || bk.bits.size() >= 8000) return;
            // Small integers and halves stay literals: the compiler folds them exactly (x*1, 0+x as
            // a select, compares against 0) and encodes them as 32-bit immediates.
            double kv = prog.nodes[id].k;
            if (kv == kv && std::fabs(kv) <= 256.0 && kv * 2.0 == std::floor(kv * 2.0)) return;
            uint64_t bits;
            std::memcpy(&bits, &prog.nodes[id].k, 8);
            bk.index[id] = int32_t(bk.bits.size());
            bk.bits.push_back(bits);
        };
        if (everything) {
            for (size_t i = 0; i < prog.nodes.size(); i++) want(uint32_t(i));
        } else {
            for (size_t i = lo; i < hi; i++) {
                const Node& n = prog.nodes[order[i]];
                if (op_is_unary(n.op) || op_is_binary(n.op)) want(n.a);
                if (op_is_binary(n.op)) want(n.b);
            }
            for (int c = 0; c < 3; c++) want(prog.root[c]);
        }
        return bk;
    };
    auto bank_text = [&](const Bank& bk) {
        std::string t;
        if (bk.bits.empty()) return t;
        t += "__constant__ unsigned long long MRK_BITS[" + std::to_string(bk.bits.size()) + "] = {\n";
        char kb[32];
        for (size_t i = 0; i < bk.bits.size(); i++) {
            std::snprintf(kb, sizeof kb, "0x%016" PRIx64 "ULL,%s", bk.bits[i], (i % 4 == 3) ? "\n" : " ");
            t += kb;
        }
        t += "};\n#define MRK(i) (reinterpret_cast<const double*>(MRK_BITS)[i])\n";
        return t;
    };
    const Bank whole_bank = make_bank(0, 0, true);

    Emitter em{prog, n_trans < opt.inline_transcendentals_below, opt.constants_in_bank ? &whole_bank.index : nullptr};
    const std::vector<uint8_t> booleans = opt.boolean_logic ? find_booleans(prog) : std::vector<uint8_t>();
    if (opt.boolean_logic) em.boolean = &booleans;
    // The NOT form `1 + -(b)` reads b itself, not only its two operands: b must be visible wherever the
    // NOT is evaluated (frame slots and imports of segmented programs).
    auto not_operand = [&](uint32_t id) -> uint32_t {
        if (booleans.empty() || booleans[id] != 2) return UINT32_MAX;
        const Node& n = prog.nodes[id];
        const uint32_t neg = prog.nodes[n.a].op == OP_NEG ? n.a : n.b;
        return prog.nodes[neg].a;
    };
    // sign-only sines: unsegmented programs whose sines are not batched (the straight-line form)
    std::vector<uint8_t> sign_only;
    if (opt.boolean_logic && opt.sign_of_sine && !segmented) {
        sign_only = find_sign_only_sines(prog, booleans);
        for (size_t i = 0; i < order.size(); i++)
            if (order_batch[i] && sign_only[order[i]]) sign_only[order[i]] = 0;
        em.sign_only = &sign_only;
    }

    uint32_t block = opt.block ? ((opt.block + 31) / 32) * 32 : 256;
    uint32_t min_blocks_per_sm = opt.min_blocks_per_sm;
    if (opt.auto_shape && em.inline_trans && !segmented && order.size() >= kOneBlockPerSmValues) {
        block = 640;
        min_blocks_per_sm = 1;
        if (opt.frame_pixels_hint) {
            static const struct { uint32_t block; double cost; } kShapes[] = {{640, 1.0}, {768, 1.015}, {1024, 1.02}};
            double best = 0.0;
            for (const auto& sh : kShapes) {
                const uint64_t per_round = uint64_t(opt.sm_count_hint ? opt.sm_count_hint : 148) * sh.block;
                const double t = double((opt.frame_pixels_hint + per_round - 1) / per_round) * sh.block * sh.cost;
                if (best == 0.0 || t < best) { best = t; block = sh.block; }
            }
        }
    }
    const bool use_batches = !em.inline_trans;
    // guarded regions: the straight-line form only (one kernel, sin/exp/ln inlined), like the sign-only sines
    const GuardRegions guards = opt.boolean_logic && !segmented && !use_batches
                                    ? find_guard_regions(prog, booleans, sign_only, not_operand) : GuardRegions{};
    std::string prelude = "// generated by maray_b200 (NVRTC back end); compiled with --fmad=false\n";
    // one private instance of the batch helpers per segment function of a single-unit program
    const bool private_helpers = use_batches && segmented && !chain;
    if (use_batches) {
        if (private_helpers) prelude += "#define MR_NO_DEFAULT_BATCH_HELPERS 1\n";
        prelude += "#define MR_SCR_STRIDE " + std::to_string(block) + "\n";
    }
    prelude += kDeviceSemText;
    prelude += "\n";

    char buf[320];
    // The sampling state is the last parameter, after the chain kernels' frame arguments (whose offsets stay put), with
    // a zero default: one sample per pixel at the integer coordinate.
    auto kernel_head = [&](std::string& out, const char* extra_args) {
        if (min_blocks_per_sm)
            std::snprintf(buf, sizeof buf,
                          "extern \"C\" __global__ void __launch_bounds__(%u, %u) %s(const MrParams p%s, const MrSampling sp = MrSampling{}) {\n",
                          block, min_blocks_per_sm, kJitKernelName, extra_args);
        else
            std::snprintf(buf, sizeof buf,
                          "extern \"C\" __global__ void __launch_bounds__(%u) %s(const MrParams p%s, const MrSampling sp = MrSampling{}) {\n",
                          block, kJitKernelName, extra_args);
        out += buf;
        out += "  __shared__ unsigned int stage[3 * " + std::to_string(block) + " / 4];\n  (void)stage;\n";
        out += "  const unsigned int j = blockIdx.x * blockDim.x + threadIdx.x;\n";
        out += "  const bool active = j < p.n;\n";
        out += "  const unsigned int pix = p.p0 + (active ? j : 0u);\n";   // idle lanes redo pixel p0
        out += "  const unsigned int yi = pix / p.W;\n";
        out += "  const unsigned int xi = pix - yi * p.W;\n";
        // `x as f64`, moved by the pass's sub-pixel offset (+0.0 with one sample per pixel: the same bits)
        out += "  const double X = (double)xi + sp.ox;\n  const double Y = (double)yi + sp.oy;\n";
        out += "  const MrTexture* __restrict__ T = p.tex;\n  (void)T;\n";
        if (use_batches) out += "  mr_scratch_tables_init();\n";
    };
    auto store_call = [&](std::string& out, const std::vector<int32_t>& slot, const std::function<std::string(int32_t)>& frame_ref,
                          const Emitter& e, const std::vector<uint8_t>* in_scope) {
        std::string args;
        for (int c = 0; c < 3; c++) {
            uint32_t r = prog.root[c];
            if (slot[r] >= 0 && !(in_scope && (*in_scope)[r])) args += frame_ref(slot[r]);
            else e.operand(args, r);
            args += ", ";
        }
        out += "  if (sp.acc != nullptr) mr_store_sampled(p, sp, stage, " + args + "active, j);\n";   // a supersampling pass
        out += "  else mr_store_block(p, stage, " + args + "active, j);\n}\n";
    };

    std::vector<std::string> modules;
    uint32_t frame_slots = 0;
    std::vector<int32_t> slot(prog.nodes.size(), -1);
    std::vector<uint32_t> seg_of(prog.nodes.size(), 0), last_use(prog.nodes.size(), 0);

    if (segmented) {
        // Segment of each value, and the last segment that reads it.  The channels are read by the epilogue:
        // after the last segment function (one unit), inside the last kernel (chain).
        const uint32_t epilogue = chain ? n_seg - 1 : n_seg;
        for (uint32_t s = 0; s < n_seg; s++)
            for (size_t i = seg_lo(s); i < seg_hi(s); i++) seg_of[order[i]] = s;
        for (size_t i = 0; i < order.size(); i++) {
            const Node& n = prog.nodes[order[i]];
            uint32_t s = seg_of[order[i]];
            auto use = [&](uint32_t id) {
                Op o = prog.nodes[id].op;
                if (o == OP_CONST || o == OP_X || o == OP_Y) return;
                if (last_use[id] < s) last_use[id] = s;
            };
            if (op_is_unary(n.op) || op_is_binary(n.op)) use(n.a);
            if (op_is_binary(n.op)) use(n.b);
            if (uint32_t extra = not_operand(order[i]); extra != UINT32_MAX) use(extra);
        }
        for (int c = 0; c < 3; c++) {
            Op o = prog.nodes[prog.root[c]].op;
            if (o != OP_CONST && o != OP_X && o != OP_Y) last_use[prog.root[c]] = std::max(last_use[prog.root[c]], epilogue);
        }
        // Frame slots: a value gets one when it is read after its own segment; slots are recycled
        // once the last reading segment has finished.
        std::vector<std::vector<int32_t>> free_after(n_seg + 2);
        std::vector<int32_t> free_list;
        for (uint32_t s = 0; s < n_seg; s++) {
            if (s > 0) for (int32_t f : free_after[s - 1]) free_list.push_back(f);
            for (size_t i = seg_lo(s); i < seg_hi(s); i++) {
                uint32_t id = order[i];
                Op o = prog.nodes[id].op;
                if (o == OP_X || o == OP_Y) continue;
                if (last_use[id] > s) {
                    int32_t f;
                    if (!free_list.empty()) { f = free_list.back(); free_list.pop_back(); }
                    else f = int32_t(frame_slots++);
                    slot[id] = f;
                    if (last_use[id] <= n_seg) free_after[std::min(last_use[id], n_seg)].push_back(f);
                }
            }
        }
    }
    // values a segment reads from earlier segments
    auto imports_of = [&](uint32_t s, bool with_roots) {
        std::vector<uint32_t> tmp;
        auto use = [&](uint32_t id) {
            Op o = prog.nodes[id].op;
            if (o == OP_CONST || o == OP_X || o == OP_Y) return;
            if (seg_of[id] < s) tmp.push_back(id);
        };
        for (size_t i = seg_lo(s); i < seg_hi(s); i++) {
            const Node& n = prog.nodes[order[i]];
            if (op_is_unary(n.op) || op_is_binary(n.op)) use(n.a);
            if (op_is_binary(n.op)) use(n.b);
            if (uint32_t extra = not_operand(order[i]); extra != UINT32_MAX) use(extra);
        }
        if (with_roots) for (int c = 0; c < 3; c++) use(prog.root[c]);
        std::sort(tmp.begin(), tmp.end());
        tmp.erase(std::unique(tmp.begin(), tmp.end()), tmp.end());
        return tmp;
    };
    // the statements of order[lo, hi) with the frame stores of values that outlive the segment
    auto emit_range = [&](std::string& out, const Emitter& e, size_t lo, size_t hi, const std::function<std::string(int32_t)>& frame_ref,
                          const char* store_guard) {
        for (size_t i = lo; i < hi;) {
            size_t j = i + 1;
            if (use_batches && order_batch[i]) while (j < hi && order_batch[j] == order_batch[i]) j++;
            if (j - i > 1) e.batch_calls(out, order, i, j);
            else e.statement(out, order[i]);
            for (size_t m = i; m < j; m++) {
                uint32_t id = order[m];
                if (segmented && slot[id] >= 0) {
                    std::snprintf(buf, sizeof buf, "  %s%s = v%u;\n", store_guard, frame_ref(slot[id]).c_str(), id);
                    out += buf;
                }
            }
            i = j;
        }
    };

    if (chain) {
        // ---- one kernel per segment ------------------------------------------------------------------
        auto gref = [](int32_t f) { return "F[" + std::to_string(f) + "ull * FS + jj]"; };
        for (uint32_t s = 0; s < n_seg; s++) {
            const Bank bk = make_bank(seg_lo(s), seg_hi(s), false);
            Emitter e = em;
            e.bank_index = opt.constants_in_bank ? &bk.index : nullptr;
            e.helper_suffix.clear();
            std::string unit;
            unit.reserve((seg_hi(s) - seg_lo(s)) * 56 + prelude.size() + 4096);
            unit += prelude;
            unit += bank_text(bk);
            std::snprintf(buf, sizeof buf, "// segment %u of %u\n", s, n_seg);
            unit += buf;
            kernel_head(unit, ", double* __restrict__ F, const unsigned long long FS");
            unit += "  const unsigned long long jj = active ? j : 0ull;\n";       // idle lanes read pixel 0's frame column, write nothing
            const bool last = s + 1 == n_seg;
            std::vector<uint8_t> in_scope(prog.nodes.size(), 0);
            for (uint32_t id : imports_of(s, last)) {
                std::snprintf(buf, sizeof buf, "  const double v%u = %s;\n", id, gref(slot[id]).c_str());
                unit += buf;
                e.bool_from_double(unit, id);
                in_scope[id] = 1;
            }
            for (size_t i = seg_lo(s); i < seg_hi(s); i++) in_scope[order[i]] = 1;
            emit_range(unit, e, seg_lo(s), seg_hi(s), gref, "if (active) ");
            if (last) store_call(unit, slot, gref, e, &in_scope);
            else unit += "}\n";
            modules.push_back(std::move(unit));
        }
    } else {
        // ---- one translation unit ------------------------------------------------------------------------
        std::string src;
        src.reserve(order.size() * 40 + 8192);
        src += prelude;
        src += bank_text(whole_bank);
        auto lref = [](int32_t f) { return "F[" + std::to_string(f) + "]"; };
        if (segmented) {
            for (uint32_t s = 0; s < n_seg; s++) {
                static const char* const kSegArgs =
                    "(double* __restrict__ F, const double X, const double Y, const MrTexture* __restrict__ T)";
                if (private_helpers) {
                    std::snprintf(buf, sizeof buf, "MR_BATCH_HELPERS(_s%u)\n", s);
                    src += buf;
                    std::snprintf(buf, sizeof buf, "_s%u", s);
                    em.helper_suffix = buf;
                }
                std::snprintf(buf, sizeof buf, "__device__ __noinline__ void mr_seg%u", s);
                src += buf; src += kSegArgs; src += " {\n";
                for (uint32_t id : imports_of(s, false)) {
                    std::snprintf(buf, sizeof buf, "  const double v%u = F[%d];\n", id, slot[id]);
                    src += buf;
                    em.bool_from_double(src, id);
                }
                emit_range(src, em, seg_lo(s), seg_hi(s), lref, "");
                src += "}\n";
            }
        }
        kernel_head(src, "");
        if (segmented) {
            std::snprintf(buf, sizeof buf, "  double F[%u];\n", frame_slots ? frame_slots : 1);
            src += buf;
            for (uint32_t s = 0; s < n_seg; s++) {
                std::snprintf(buf, sizeof buf, "  mr_seg%u(F, X, Y, T);\n", s);
                src += buf;
            }
        } else if (!guards.regions.empty()) {
            // Body values leave their places in the schedule and are emitted, in schedule order, where their AND is.
            // Valid: a body value's other operands precede it and so precede the AND, and nothing outside the body reads
            // it.  All 32 lanes reach every vote: idle lanes redo pixel p0, and an inner region sits inside its outer
            // region's warp-uniform branch.
            std::vector<std::vector<uint32_t>> members(guards.regions.size() + 1);
            for (uint32_t id : order) members[size_t(guards.owner[id] + 1)].push_back(id);
            std::function<void(int32_t)> emit_members = [&](int32_t r) {
                for (uint32_t id : members[size_t(r + 1)]) {
                    const int32_t g = guards.rooted_at[id];
                    if (g < 0) { em.statement(src, id); continue; }
                    const GuardRegion& gr = guards.regions[size_t(g)];
                    std::snprintf(buf, sizeof buf, "  bool b%u = false;\n  if (mr_warp_any(", id);
                    src += buf; em.bool_operand(src, gr.guard); src += ")) {\n";
                    emit_members(g);
                    std::snprintf(buf, sizeof buf, "  b%u = ", id);
                    src += buf; em.bool_operand(src, gr.guard); src += " && "; em.bool_operand(src, gr.body); src += ";\n  }\n";
                    std::snprintf(buf, sizeof buf, "  const double v%u = b%u ? 1.0 : 0.0;\n", id, id);
                    src += buf;
                }
            };
            emit_members(-1);
        } else {
            emit_range(src, em, 0, order.size(), lref, "");
        }
        store_call(src, slot, lref, em, nullptr);
        modules.push_back(std::move(src));
    }

    if (info) {
        info->segments = n_seg;
        info->chain = chain;
        info->frame_slots = segmented ? frame_slots : 0;
        info->transcendentals_inlined = em.inline_trans;
        info->block = block;
        // argument rows + result rows, then glibc's exp and log tables
        info->dynamic_smem_bytes = use_batches ? 2 * kScratchRows * block * uint32_t(sizeof(double)) + 4096 : 0;
    }
    return modules;
}
}  // namespace

std::string generate_cuda_source(const Program& prog, const CodegenOptions& opt, CodegenInfo* info) {
    CodegenOptions one = opt;
    one.chain = false;
    return generate(prog, one, info)[0];
}

std::vector<std::string> generate_cuda_modules(const Program& prog, const CodegenOptions& opt, CodegenInfo* info) {
    return generate(prog, opt, info);
}

}  // namespace maray
