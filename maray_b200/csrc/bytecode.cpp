// SSA program -> two-accumulator bytecode (version 3).  See bytecode.hpp for the format.
//
// One linear pass over the program's schedule.  A value that does not depend on x is computed in the
// scalar shape (once per block), everything else in the wide shape (P values per thread).  The running
// value of each shape stays in that shape's accumulator; a value is written to a slot only if somebody
// reads it after the next instruction of its own shape has replaced the accumulator.  Wide slots are
// recycled as soon as their last reader has been emitted; row-uniform scalar slots are never recycled
// (every warp of a block computes and stores every such value itself, with identical bits, so a warp
// only ever reads what it has written and the kernel needs no barrier).
#include "bytecode.hpp"

#include <algorithm>

namespace maray {
namespace {

constexpr uint32_t NONE = 0xffffffffu;

class BcGen {
public:
    BcGen(const Program& p, Bytecode& b, bool row_uniform) : P(p), B(b), uniform(row_uniform) {}
    std::string err;

    void run() {
        const size_t n = P.nodes.size();
        uses_left.assign(n, 0);
        last_use.assign(n, 0);
        wslot.assign(n, -1);
        uslot.assign(n, -1);
        kidx.assign(n, -1);
        for (size_t i = 0; i < n; i++) {
            const Node& nd = P.nodes[i];
            if (nd.op == OP_CONST) {
                kidx[i] = int32_t(B.consts.size());
                B.consts.push_back(nd.k);
                continue;
            }
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) uses_left[nd.a]++;
            if (op_is_binary(nd.op)) uses_left[nd.b]++;
        }
        if (B.consts.empty()) B.consts.push_back(0.0);
        for (int c = 0; c < 3; c++) uses_left[P.root[c]]++;
        B.row_uniform = uniform;
        B.n_wide = uniform ? 1 : 2;      // X (and Y)
        B.n_uniform = uniform ? 1 : 0;   // Y
        for (size_t i = 0; i < n; i++) {
            if (P.nodes[i].op == OP_X) { wslot[i] = 0; uses_left[i] = 0x7fffffff; }
            if (P.nodes[i].op == OP_Y) {
                if (uniform) uslot[i] = 0; else wslot[i] = 1;
                uses_left[i] = 0x7fffffff;
            }
        }

        // The instructions to emit, in order, and for each the next one of the same shape.
        std::vector<uint32_t> seq;
        for (uint32_t id : P.order) {
            Op o = P.nodes[id].op;
            if (o != OP_X && o != OP_Y) seq.push_back(id);
        }
        std::vector<uint32_t> pos(n, NONE);
        for (size_t i = 0; i < seq.size(); i++) pos[seq[i]] = uint32_t(i);
        for (size_t i = 0; i < seq.size(); i++) {
            const Node& nd = P.nodes[seq[i]];
            auto use = [&](uint32_t v) { if (P.nodes[v].op != OP_CONST) last_use[v] = std::max(last_use[v], uint32_t(i)); };
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) use(nd.a);
            if (op_is_binary(nd.op)) use(nd.b);
        }
        std::vector<uint32_t> next_same(seq.size(), NONE);
        uint32_t next_of_shape[2] = {NONE, NONE};
        for (size_t i = seq.size(); i-- > 0;) {
            const int s = scalar_shape(seq[i]) ? 1 : 0;
            next_same[i] = next_of_shape[s];
            next_of_shape[s] = uint32_t(i);
        }

        seq_ = &seq;
        for (size_t i = 0; i < seq.size() && err.empty(); i++) gen(seq[i], uint32_t(i), next_same[i]);

        // channels whose value is a constant, X or Y (everything else was written when computed)
        static const BcOp outs[3] = {BC_OUT_R, BC_OUT_G, BC_OUT_B};
        for (int c = 0; c < 3 && err.empty(); c++) {
            uint32_t r = P.root[c];
            Op o = P.nodes[r].op;
            if (o != OP_CONST && o != OP_X && o != OP_Y) continue;
            uint32_t ka = 0, a = 0;
            if (!operand(r, &ka, &a)) return;
            emit(bc_handler(outs[c], false, ka, 0), ka << BC_F_KA_SHIFT, 0, a, 0);
        }
        emit(BC_H_END, 0, 0, 0, 0);
        if (B.consts.size() + B.n_uniform > 0xffff) err = "program has more than 65535 constants and row-uniform values";
        seq_ = nullptr;                      // `seq` is this call's local
    }

private:
    const Program& P;
    Bytecode& B;
    const bool uniform;
    std::vector<uint32_t> uses_left, last_use;
    std::vector<int32_t> wslot, uslot, kidx;
    std::vector<uint32_t> free_wide;
    uint32_t acc_holds = NONE, sacc_holds = NONE;
    bool acc_negated = false;        // acc_holds is a `neg` whose negation has been left to its only consumer
    const std::vector<uint32_t>* seq_ = nullptr;

    // `neg` of the accumulator, read once, by the next wide instruction, which is a binary operation with the
    // negated value as exactly one operand: the negation rides on that instruction (BC_H_BINN) and this one
    // is not emitted.  Same arithmetic, one dispatch less (14 % of the shipped chess scene's instructions).
    bool neg_can_ride(uint32_t id, uint32_t next_same_shape) const {
        const Node& n = P.nodes[id];
        if (n.op != OP_NEG || scalar_shape(id) || acc_holds != n.a || acc_negated) return false;
        if (next_same_shape == NONE || uses_left[id] != 1 || last_use[id] != next_same_shape) return false;
        for (int c = 0; c < 3; c++) if (P.root[c] == id) return false;
        const Node& u = P.nodes[(*seq_)[next_same_shape]];
        if (u.op != OP_ADD && u.op != OP_MUL && u.op != OP_MAX && u.op != OP_MIN) return false;
        return (u.a == id) != (u.b == id);
    }

    bool is_const(uint32_t id) const { return P.nodes[id].op == OP_CONST; }
    // Values that do not depend on x are one number per block (every block lies inside one row).
    bool scalar_shape(uint32_t id) const { return uniform && !(P.nodes[id].dep & DEP_X); }

    void emit(uint32_t handler, uint32_t flags, uint32_t dst, uint32_t a, uint32_t b) {
        B.code.push_back(bc_encode(handler, flags, dst, a, b));
    }
    uint32_t alloc_wide() {
        if (!free_wide.empty()) { uint32_t s = free_wide.back(); free_wide.pop_back(); return s; }
        if (B.n_wide >= 65535) { err = "program needs more than 65535 live values"; return 0; }
        return B.n_wide++;
    }
    void consume(uint32_t id) {
        if (is_const(id)) return;
        if (uses_left[id] == 0) { err = "internal: value consumed more often than it is used"; return; }
        if (--uses_left[id] == 0 && wslot[id] >= 0 && P.nodes[id].op != OP_X && P.nodes[id].op != OP_Y) {
            free_wide.push_back(uint32_t(wslot[id]));
            wslot[id] = -1;
        }
    }

    // Where an operand comes from: kind + index.
    bool operand(uint32_t v, uint32_t* kind, uint32_t* idx) {
        *idx = 0;
        if (is_const(v)) { *kind = BC_K_S; *idx = uint32_t(kidx[v]); return true; }
        if (scalar_shape(v)) {
            if (sacc_holds == v) { *kind = BC_K_T; return true; }
            if (uslot[v] >= 0) { *kind = BC_K_S; *idx = uint32_t(B.consts.size()) + uint32_t(uslot[v]); return true; }
            err = "internal: scalar operand is neither in the scalar accumulator nor in a slot";
            return false;
        }
        if (acc_holds == v) { *kind = BC_K_A; return true; }
        if (wslot[v] >= 0) { *kind = BC_K_W; *idx = uint32_t(wslot[v]); return true; }
        err = "internal: wide operand is neither in the accumulator nor in a slot";
        return false;
    }

    void gen(uint32_t id, uint32_t at, uint32_t next_same_shape) {
        const Node& n = P.nodes[id];
        const bool sc = scalar_shape(id);
        uint32_t ka = 0, kb = 0, a = 0, b = 0, dst = 0;
        BcOp op = BC_END;
        if (neg_can_ride(id, next_same_shape)) {
            consume(n.a);
            acc_holds = id;
            acc_negated = true;
            return;
        }
        const bool neg_acc = acc_negated;      // this instruction is the consumer the negation was left to
        if (op_is_unary(n.op)) {
            op = BcOp(BC_NEG + (n.op - OP_NEG));
            if (!operand(n.a, &ka, &a)) return;
        } else {
            switch (n.op) {
            case OP_ADD: op = BC_ADD; break;
            case OP_MUL: op = BC_MUL; break;
            case OP_MAX: op = BC_MAX; break;
            case OP_MIN: op = BC_MIN; break;
            case OP_TEX:
                if (n.imm > 0xffff) { err = "texture index too large for the interpreter back end"; return; }
                op = BC_TEX; dst = n.imm;
                break;
            default: err = "internal: unexpected op"; return;
            }
            if (!operand(n.a, &ka, &a) || !operand(n.b, &kb, &b)) return;
        }
        if (sc && ((ka != BC_K_S && ka != BC_K_T) || (op_is_binary(n.op) && kb != BC_K_S && kb != BC_K_T))) {
            err = "internal: scalar instruction with a wide operand";
            return;
        }
        if (neg_acc && (sc || !(op >= BC_ADD && op <= BC_MIN) || (ka == BC_K_A) == (kb == BC_K_A))) {
            err = "internal: a deferred negation met an instruction that cannot carry it";
            return;
        }
        acc_negated = false;
        emit(bc_handler(op, sc, ka, kb, neg_acc), (ka << BC_F_KA_SHIFT) | (kb << BC_F_KB_SHIFT) | (neg_acc ? BC_F_NEG_ACC : 0u), dst, a, b);
        consume(n.a);
        if (op_is_binary(n.op)) consume(n.b);
        if (!err.empty()) return;
        (sc ? sacc_holds : acc_holds) = id;

        // A slot is needed when somebody reads the value after the next instruction of this shape has
        // replaced the accumulator (that instruction itself still reads the accumulator).
        uint32_t root_refs = 0;
        for (int c = 0; c < 3; c++) if (P.root[c] == id) root_refs++;
        const bool read_later = uses_left[id] > root_refs && next_same_shape != NONE && last_use[id] > next_same_shape;
        if (uses_left[id] > root_refs && last_use[id] <= at) { err = "internal: value is used before it is defined"; return; }
        if (read_later) {
            if (n.op == OP_TEX)   // TEX keeps its texture id in the dst field: store with a MOV
                emit(bc_handler(BC_MOV, sc, sc ? BC_K_T : BC_K_A, 0), (sc ? BC_K_T : BC_K_A) << BC_F_KA_SHIFT, 0, 0, 0);
            uint32_t s;
            if (sc) {
                s = B.n_uniform++;
                uslot[id] = int32_t(s);
                s += uint32_t(B.consts.size());            // scalar file index
            } else {
                s = alloc_wide();
                wslot[id] = int32_t(s);
            }
            B.code.back() |= (uint64_t(BC_F_STORE) << 8) | (uint64_t(s & 0xffff) << 16);
        }
        // channel outputs are written the moment their value exists
        static const BcOp outs[3] = {BC_OUT_R, BC_OUT_G, BC_OUT_B};
        for (int c = 0; c < 3; c++) {
            if (P.root[c] != id) continue;
            const uint32_t k = sc ? BC_K_T : BC_K_A;
            emit(bc_handler(outs[c], false, k, 0), k << BC_F_KA_SHIFT, 0, 0, 0);
            consume(id);
        }
    }
};

}  // namespace

std::vector<uint64_t> bytecode_for_launch(const Bytecode& bc, uint32_t slot16, std::string* err) {
    if (uint64_t(bc.n_wide + 3) * slot16 > 0xffff) {
        if (err) *err = "slot file too large for this launch shape (16-bit operand fields)";
        return {};
    }
    std::vector<uint64_t> out;
    out.reserve(bc.code.size() + bc.code.size() / (kBcChunk - 1) + kBcChunk);
    for (uint64_t w : bc.code) {
        const uint32_t h = uint32_t(w) & 0xff, fl = uint32_t(w >> 8) & 0xff;
        if (h == BC_H_END) break;                      // the padding below ends the stream
        if (h < BC_H_SCALAR || h >= BC_H_BINN) {
            uint64_t dst = (w >> 16) & 0xffff, a = (w >> 32) & 0xffff, b = (w >> 48) & 0xffff;
            if (((fl >> BC_F_KA_SHIFT) & 3u) == BC_K_W) a *= slot16;
            const bool binary = (h >= BC_H_BIN && h < BC_H_UN) || h == BC_H_TEX || h >= BC_H_BINN;
            if (binary && ((fl >> BC_F_KB_SHIFT) & 3u) == BC_K_W) b *= slot16;
            if ((fl & BC_F_STORE) && h != BC_H_TEX) dst *= slot16;
            w = (w & 0xffffull) | (dst << 16) | (a << 32) | (b << 48);
        }
        if (out.size() % kBcChunk == kBcChunk - 1) out.push_back(bc_encode(BC_H_YIELD, 0, 0, 0, 0));
        out.push_back(w);
    }
    do out.push_back(bc_encode(BC_H_END, 0, 0, 0, 0)); while (out.size() % kBcChunk != 0);
    return out;
}

bool compile_bytecode(const Program& prog, Bytecode* out, std::string* err, bool row_uniform) {
    out->code.clear();
    out->consts.clear();
    if (prog.stats.op_count[OP_APP]) {   // the interpreter is a prebuilt kernel: it cannot call a custom runtime's code
        if (err) *err = "the interpreter back end cannot call a custom runtime's maray_app (use the NVRTC back end)";
        return false;
    }
    BcGen g(prog, *out, row_uniform);
    g.run();
    if (!g.err.empty()) { if (err) *err = g.err; return false; }
    return true;
}

}  // namespace maray
