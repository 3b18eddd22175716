// Expr tree -> hash-consed SSA program.  See program.hpp for the contract.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <new>
#include <unordered_map>

#include "program.hpp"

namespace maray {

const char* op_name(Op o) {
    static const char* names[OP_COUNT] = {"const", "x", "y", "neg", "abs", "recip", "sqrt", "step", "sin", "exp",
                                          "ln", "add", "mul", "max", "min", "tex"};
    return o < OP_COUNT ? names[o] : "?";
}

namespace {

struct Key {
    uint32_t op, a, b, imm;
    uint64_t kbits;
    bool operator==(const Key& o) const { return op == o.op && a == o.a && b == o.b && imm == o.imm && kbits == o.kbits; }
};
struct KeyHash {
    size_t operator()(const Key& k) const {
        uint64_t h = k.kbits * 0x9e3779b97f4a7c15ull;
        h ^= (uint64_t(k.op) << 56) ^ (uint64_t(k.a) << 28) ^ uint64_t(k.b) ^ (uint64_t(k.imm) << 40);
        h *= 0xff51afd7ed558ccdull;
        return size_t(h ^ (h >> 31));
    }
};

constexpr uint32_t NONE = 0xffffffffu;

struct Binding { const Expr* def; uint32_t value; uint8_t state; };   // state: 0 new, 1 lowering, 2 done

struct Scope {
    const Expr* let;
    std::vector<Binding> vars;
    std::unordered_map<uint64_t, uint32_t> index;   // id -> first definition with that id
    Scope* up;
};

uint64_t bits_of(double v) { uint64_t b; std::memcpy(&b, &v, 8); return b; }

class Lowering {
public:
    Lowering(const std::vector<TextureDim>& tex) : tex_(tex) {}

    std::vector<Node> nodes;
    std::string err;

    uint32_t konst(double v) {
        Key k{OP_CONST, 0, 0, 0, bits_of(v)};
        auto it = table_.find(k);
        if (it != table_.end()) return it->second;
        Node n{OP_CONST, DEP_CONST, 0, 0, 0, v};
        nodes.push_back(n);
        uint32_t id = uint32_t(nodes.size() - 1);
        table_.emplace(k, id);
        return id;
    }

    uint32_t leaf(Op op) {
        Key k{op, 0, 0, 0, 0};
        auto it = table_.find(k);
        if (it != table_.end()) return it->second;
        Node n{op, uint8_t(op == OP_X ? DEP_X : DEP_Y), 0, 0, 0, 0.0};
        nodes.push_back(n);
        uint32_t id = uint32_t(nodes.size() - 1);
        table_.emplace(k, id);
        return id;
    }

    uint32_t unary(Op op, uint32_t a) {
        if (nodes[a].op == OP_CONST) {
            // Host folding: the same IEEE operation, and for sin/exp/ln the host libm -- which is
            // what the reference itself calls (reference src/lib.rs:648-650).
            double v = nodes[a].k, r = 0.0;
            switch (op) {
            case OP_NEG: r = -v; break;
            case OP_ABS: r = std::fabs(v); break;
            case OP_RECIP: r = 1.0 / v; break;
            case OP_SQRT: r = std::sqrt(v); break;
            case OP_STEP: r = sem_step(v); break;
            case OP_SIN: r = std::sin(v); break;
            case OP_EXP: r = std::exp(v); break;
            case OP_LN: r = std::log(v); break;
            default: break;
            }
            return konst(r);
        }
        return intern(op, a, 0, 0);
    }

    uint32_t binary(Op op, uint32_t a, uint32_t b) {
        if (nodes[a].op == OP_CONST && nodes[b].op == OP_CONST) {
            double x = nodes[a].k, y = nodes[b].k, r = 0.0;
            switch (op) {
            case OP_ADD: r = x + y; break;
            case OP_MUL: r = x * y; break;
            case OP_MAX: r = sem_max(x, y); break;
            case OP_MIN: r = sem_min(x, y); break;
            default: break;
            }
            return konst(r);
        }
        return intern(op, a, b, 0);
    }

    // App(id, a, b) with the default texture runtime (reference src/textures.rs:14-65).
    uint32_t app(uint32_t id, uint32_t a, uint32_t b) {
        uint32_t img = id / 5, k = id % 5;
        if (img >= tex_.size()) {
            err = "App id " + std::to_string(id) + " is outside the texture runtime's function table (" +
                  std::to_string(tex_.size() * 5) + " functions for " + std::to_string(tex_.size()) + " textures)";
            return NONE;
        }
        if (k == 3) return konst(double(tex_[img].w));    // fun_image_width  (arguments ignored)
        if (k == 4) return konst(double(tex_[img].h));    // fun_image_height
        return intern(OP_TEX, a, b, img * 4 + k);
    }

    uint32_t lower(const Expr* e, Scope* sc) {
        if (!err.empty()) return NONE;
        switch (e->tag) {
        case T_ARC: case T_DECOR: return lower(e->a, sc);
        case T_X: return leaf(OP_X);
        case T_Y: return leaf(OP_Y);
        case T_TAU: return konst(6.283185307179586);
        case T_E: return konst(2.718281828459045);
        case T_NAT: return konst(double(e->n));
        case T_VAR: return var(e->n, sc);
        case T_NEG: case T_ABS: case T_RECIP: case T_SQRT:
        case T_STEP: case T_SIN: case T_EXP: case T_LN: {
            uint32_t a = lower(e->a, sc);
            if (a == NONE) return NONE;
            return unary(Op(OP_NEG + (e->tag - T_NEG)), a);
        }
        case T_ADD: case T_MUL: case T_MAX: case T_MIN: {
            uint32_t a = lower(e->a, sc);
            uint32_t b = lower(e->b, sc);
            if (a == NONE || b == NONE) return NONE;
            return binary(Op(OP_ADD + (e->tag - T_ADD)), a, b);
        }
        case T_APP: {
            uint32_t a = lower(e->a, sc);
            uint32_t b = lower(e->b, sc);
            if (a == NONE || b == NONE) return NONE;
            return app(e->app_id, a, b);
        }
        case T_LET: {
            Scope in;
            in.let = e; in.up = sc;
            in.vars.resize(e->n_vars);
            for (uint64_t i = 0; i < e->n_vars; i++) {
                in.vars[i] = Binding{e->vars[i].def, NONE, 0};
                in.index.emplace(e->vars[i].id, uint32_t(i));   // keeps the FIRST definition of an id
            }
            // Lower the definitions in file order (keeps recursion shallow for the usual
            // dependency-ordered contexts); forward references are resolved on demand by var().
            for (uint64_t i = 0; i < e->n_vars; i++) {
                auto first = in.index.find(e->vars[i].id);
                if (first->second != i) continue;               // shadowed duplicate id: never visible
                if (force(&in, uint32_t(i)) == NONE) return NONE;
            }
            return lower(e->a, &in);
        }
        default: break;
        }
        err = "unsupported expression variant";
        return NONE;
    }

private:
    uint32_t intern(Op op, uint32_t a, uint32_t b, uint32_t imm) {
        Key k{op, a, b, imm, 0};
        auto it = table_.find(k);
        if (it != table_.end()) return it->second;
        uint8_t dep = uint8_t(nodes[a].dep | (op_is_binary(op) ? nodes[b].dep : 0));
        Node n{op, dep, a, op_is_binary(op) ? b : 0, imm, 0.0};
        nodes.push_back(n);
        uint32_t id = uint32_t(nodes.size() - 1);
        table_.emplace(k, id);
        return id;
    }

    uint32_t force(Scope* s, uint32_t i) {
        Binding& bnd = s->vars[i];
        if (bnd.state == 2) return bnd.value;
        if (bnd.state == 1) {
            err = "cyclic Let definitions (variable $" + std::to_string(s->let->vars[i].id) + ")";
            return NONE;
        }
        bnd.state = 1;
        uint32_t v = lower(bnd.def, s);
        s->vars[i].value = v;
        s->vars[i].state = 2;
        return v;
    }

    uint32_t var(uint64_t name, Scope* sc) {
        for (Scope* s = sc; s; s = s->up) {
            auto it = s->index.find(name);
            if (it != s->index.end()) return force(s, it->second);
        }
        err = "unbound variable $" + std::to_string(name);
        return NONE;
    }

    const std::vector<TextureDim>& tex_;
    std::unordered_map<Key, uint32_t, KeyHash> table_;
};

struct LowerJob {
    const Scene* scene;
    const std::vector<TextureDim>* tex;
    Program* out;
    std::string* err;
    bool ok;
};

void lower_job_body(LowerJob* j);

// Runs on its own (big-stack) thread: nothing may escape it -- an exception that leaves a thread's
// start routine ends the process, it never reaches the caller of run_with_big_stack.
void lower_job(void* arg) {
    LowerJob* j = static_cast<LowerJob*>(arg);
    try {
        lower_job_body(j);
    } catch (const std::bad_alloc&) {
        *j->err = "out of memory while lowering";
        j->ok = false;
    } catch (const std::exception& e) {
        *j->err = std::string("lowering failed: ") + e.what();
        j->ok = false;
    } catch (...) {
        *j->err = "lowering failed";
        j->ok = false;
    }
}

void lower_job_body(LowerJob* j) {
    Lowering L(*j->tex);
    uint32_t roots[3];
    for (int c = 0; c < 3; c++) {
        roots[c] = L.lower(j->scene->color[c], nullptr);
        if (roots[c] == NONE) { *j->err = L.err.empty() ? "lowering failed" : L.err; j->ok = false; return; }
    }
    const std::vector<Node>& all = L.nodes;   // creation order is already topological

    // Register-need estimate (Sethi-Ullman on the tree view) to pick operand evaluation order:
    // visiting the needier operand first keeps fewer values live.  Order does not affect values.
    std::vector<uint32_t> need(all.size(), 0);
    for (size_t i = 0; i < all.size(); i++) {
        const Node& n = all[i];
        if (n.op == OP_CONST) need[i] = 0;
        else if (n.op == OP_X || n.op == OP_Y) need[i] = 1;
        else if (op_is_unary(n.op)) need[i] = std::max(need[n.a], 1u);
        else {
            uint32_t na = need[n.a], nb = need[n.b];
            need[i] = std::max(1u, na == nb ? na + 1 : std::max(na, nb));
        }
    }

    // Depth-first post-order from R, G, B: prunes unreachable values and fixes the schedule.
    std::vector<uint32_t> remap(all.size(), NONE);
    std::vector<Node> out_nodes;
    out_nodes.reserve(all.size());
    struct Frame { uint32_t id; uint8_t stage; };
    std::vector<Frame> stack;
    for (int c = 0; c < 3; c++) {
        stack.push_back({roots[c], 0});
        while (!stack.empty()) {
            Frame& f = stack.back();
            uint32_t id = f.id;
            if (remap[id] != NONE) { stack.pop_back(); continue; }
            const Node& n = all[id];
            bool un = op_is_unary(n.op), bin = op_is_binary(n.op);
            uint32_t first = n.a, second = n.b;
            if (bin && need[n.b] > need[n.a]) std::swap(first, second);
            if (f.stage == 0) {
                f.stage = 1;
                if (un || bin) { stack.push_back({first, 0}); continue; }
            }
            if (f.stage == 1) {
                f.stage = 2;
                if (bin) { stack.push_back({second, 0}); continue; }
            }
            Node m = n;
            if (un || bin) m.a = remap[n.a];
            if (bin) m.b = remap[n.b];
            out_nodes.push_back(m);
            remap[id] = uint32_t(out_nodes.size() - 1);
            stack.pop_back();
        }
    }

    Program* P = j->out;
    P->nodes.swap(out_nodes);
    for (int c = 0; c < 3; c++) P->root[c] = remap[roots[c]];
    P->n_textures = uint32_t(j->tex->size());
    P->order.clear();
    // Two candidate schedules: (a) the depth-first order above, (b) the order in which the scene
    // itself introduces values (Let definitions in file order, then the bodies).  Depth-first keeps
    // tree-shaped scenes short-lived; authored order wins on wide DAGs whose roots gather values
    // from everywhere.  Keep whichever needs fewer simultaneously live values.
    std::vector<uint32_t> dfs_order, authored;
    for (size_t i = 0; i < P->nodes.size(); i++)
        if (P->nodes[i].op != OP_CONST) dfs_order.push_back(uint32_t(i));
    for (size_t i = 0; i < all.size(); i++)
        if (remap[i] != NONE && all[i].op != OP_CONST) authored.push_back(remap[i]);
    auto max_live = [&](const std::vector<uint32_t>& ord) {
        std::vector<uint32_t> uses(P->nodes.size(), 0);
        for (uint32_t id : ord) {
            const Node& n = P->nodes[id];
            if (op_is_unary(n.op) || op_is_binary(n.op)) uses[n.a]++;
            if (op_is_binary(n.op)) uses[n.b]++;
        }
        for (int c = 0; c < 3; c++) uses[P->root[c]]++;
        uint32_t live = 0, peak = 0;
        for (uint32_t id : ord) {
            const Node& n = P->nodes[id];
            live++;
            peak = std::max(peak, live);
            auto done = [&](uint32_t v) {
                if (P->nodes[v].op == OP_CONST) return;
                if (--uses[v] == 0) live--;
            };
            if (op_is_unary(n.op) || op_is_binary(n.op)) done(n.a);
            if (op_is_binary(n.op)) done(n.b);
        }
        return peak;
    };
    // (c) greedy list scheduling: among the values whose operands are ready, take the one that
    // shrinks the live set most (frees the most operands), preferring the most recently enabled one
    // so that chains stay chains.  Myopic, but it handles DAGs where both fixed orders blow up.
    // position of every value in the authored order (tie-break for the "oldest first" variant)
    std::vector<uint32_t> authored_pos(P->nodes.size(), 0);
    for (size_t i = 0; i < authored.size(); i++) authored_pos[authored[i]] = uint32_t(i);
    auto greedy_schedule = [&](bool oldest_first) {
        std::vector<uint32_t> greedy;
        const size_t n = P->nodes.size();
        std::vector<uint32_t> uses(n, 0), pending(n, 0), stamp(n, 0);
        std::vector<std::vector<uint32_t>> users(n);
        auto is_k = [&](uint32_t v) { return P->nodes[v].op == OP_CONST; };
        for (uint32_t id : dfs_order) {
            const Node& nd = P->nodes[id];
            auto dep = [&](uint32_t v) {
                if (is_k(v)) return;
                uses[v]++;
                users[v].push_back(id);
                pending[id]++;
            };
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) dep(nd.a);
            if (op_is_binary(nd.op) && nd.b != nd.a) dep(nd.b);
            else if (op_is_binary(nd.op) && !is_k(nd.b)) uses[nd.b]++;   // a == b: one edge, two reads
        }
        for (int c = 0; c < 3; c++) uses[P->root[c]]++;
        auto score = [&](uint32_t id) {
            const Node& nd = P->nodes[id];
            int freed = 0;
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) {
                uint32_t reads_a = 1 + ((op_is_binary(nd.op) && nd.b == nd.a) ? 1 : 0);
                if (!is_k(nd.a) && uses[nd.a] == reads_a) freed++;
                if (op_is_binary(nd.op) && nd.b != nd.a && !is_k(nd.b) && uses[nd.b] == 1) freed++;
            }
            return freed;
        };
        struct Item { int score; uint32_t stamp; uint32_t id; };
        auto worse = [](const Item& x, const Item& y) { return x.score != y.score ? x.score < y.score : x.stamp < y.stamp; };
        std::vector<Item> heap;
        uint32_t clock = 0;
        auto push = [&](uint32_t id) {
            // newest first: chains stay chains (depth-first flavour); oldest first: follow the order
            // in which the scene introduced the values (breadth never runs far ahead)
            stamp[id] = oldest_first ? (0xffffffffu - authored_pos[id]) : ++clock;
            heap.push_back(Item{score(id), stamp[id], id});
            std::push_heap(heap.begin(), heap.end(), worse);
        };
        std::vector<uint8_t> done(n, 0);
        for (uint32_t id : dfs_order) if (pending[id] == 0) push(id);
        while (!heap.empty()) {
            std::pop_heap(heap.begin(), heap.end(), worse);
            Item it = heap.back();
            heap.pop_back();
            if (done[it.id] || it.stamp != stamp[it.id]) continue;   // superseded entry
            int sc = score(it.id);
            if (sc != it.score) { heap.push_back(Item{sc, it.stamp, it.id}); std::push_heap(heap.begin(), heap.end(), worse); continue; }
            done[it.id] = 1;
            greedy.push_back(it.id);
            const Node& nd = P->nodes[it.id];
            auto read = [&](uint32_t v) { if (!is_k(v)) uses[v]--; };
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) read(nd.a);
            if (op_is_binary(nd.op)) read(nd.b);
            for (uint32_t u : users[it.id]) if (--pending[u] == 0) push(u);
            // users of my operands may now free them: refresh the ready ones lazily (their score is
            // recomputed when popped; bump the stamp of ready co-users so they are reconsidered early)
            auto refresh = [&](uint32_t v) {
                if (is_k(v) || uses[v] != 1) return;
                for (uint32_t u : users[v]) if (!done[u] && pending[u] == 0) push(u);
            };
            if (op_is_unary(nd.op) || op_is_binary(nd.op)) refresh(nd.a);
            if (op_is_binary(nd.op)) refresh(nd.b);
        }
        if (greedy.size() != dfs_order.size()) greedy.clear();   // cannot happen for a DAG; be safe
        return greedy;
    };
    std::vector<uint32_t> greedy_new = greedy_schedule(false), greedy_old = greedy_schedule(true);
    const std::vector<uint32_t>* cand[4] = {&dfs_order, &authored, &greedy_new, &greedy_old};
    uint32_t live[4];
    int best = 0;
    for (int i = 0; i < 4; i++) {
        live[i] = cand[i]->size() == dfs_order.size() ? max_live(*cand[i]) : 0xffffffffu;
        if (live[i] < live[best]) best = i;
    }
    // tooling: MARAY_SCHEDULE=0..3 forces a candidate (order never changes a value, only live ranges)
    if (const char* e = std::getenv("MARAY_SCHEDULE")) {
        int k = std::atoi(e);
        if (k >= 0 && k < 4 && live[k] != 0xffffffffu) best = k;
    }
    const std::vector<uint32_t>& chosen = *cand[best];
    ProgramStats st;
    st.max_live = live[best];
    st.schedule_kind = uint32_t(best);
    if (std::getenv("MARAY_VERBOSE"))
        std::fprintf(stderr, "maray: max live values  depth-first %u  authored %u  greedy(newest) %u  greedy(oldest) %u\n",
                     live[0], live[1], live[2], live[3]);
    st.tree_nodes = j->scene->tree_nodes[0] + j->scene->tree_nodes[1] + j->scene->tree_nodes[2];
    st.dag_nodes = P->nodes.size();
    std::vector<uint32_t> depth(P->nodes.size(), 0);
    for (size_t i = 0; i < P->nodes.size(); i++) {
        const Node& n = P->nodes[i];
        if (n.op == OP_CONST) { st.n_const++; continue; }
        st.op_count[n.op]++;
        switch (n.dep) {
        case DEP_X: st.n_x++; break;
        case DEP_Y: st.n_y++; break;
        default: st.n_xy++; break;       // includes texture fetches at constant coordinates
        }
        uint32_t d = 0;
        if (op_is_unary(n.op) || op_is_binary(n.op)) d = depth[n.a];
        if (op_is_binary(n.op)) d = std::max(d, depth[n.b]);
        depth[i] = d + 1;
        st.depth = std::max(st.depth, depth[i]);
    }
    // Transcendental batching: pull later sin/exp/ln values of the same kind (and the few cheap values
    // they need) forward so that up to kBatchMax independent ones sit next to each other.  Bounded
    // look-ahead, so live ranges barely change; evaluation order never changes values.
    uint64_t n_trans_total = 0;
    for (const Node& nd : P->nodes) n_trans_total += (nd.op == OP_SIN || nd.op == OP_EXP || nd.op == OP_LN);
    if (n_trans_total < kOutOfLineTranscendentals) {
        P->order = chosen;
        P->batch.assign(chosen.size(), 0);
    } else {
        constexpr uint32_t kBatchMax = 8, kWindow = 384, kConeMax = 24;
        const size_t n = P->nodes.size();
        std::vector<uint32_t> pos(n, NONE);
        for (size_t i = 0; i < chosen.size(); i++) pos[chosen[i]] = uint32_t(i);
        std::vector<uint8_t> emitted(n, 0);
        for (size_t i = 0; i < n; i++) if (P->nodes[i].op == OP_CONST) emitted[i] = 1;
        std::vector<uint32_t> out, out_batch;
        out.reserve(chosen.size());
        out_batch.reserve(chosen.size());
        auto is_trans = [&](uint32_t v) { Op o = P->nodes[v].op; return o == OP_SIN || o == OP_EXP || o == OP_LN; };
        uint32_t next_batch = 0;
        std::vector<uint32_t> cone, stack_;
        std::vector<uint8_t> in_batch(n, 0);
        for (size_t p0 = 0; p0 < chosen.size(); p0++) {
            uint32_t id = chosen[p0];
            if (emitted[id]) continue;
            if (!is_trans(id)) { emitted[id] = 1; out.push_back(id); out_batch.push_back(0); continue; }
            std::vector<uint32_t> members{id};
            in_batch[id] = 1;
            uint32_t scanned = 0;
            for (size_t j = p0 + 1; j < chosen.size() && scanned < kWindow && members.size() < kBatchMax; j++) {
                uint32_t c = chosen[j];
                if (emitted[c]) continue;
                scanned++;
                if (P->nodes[c].op != P->nodes[id].op) continue;
                // the not-yet-evaluated values c needs: small, free of transcendentals, independent of the batch
                cone.clear();
                stack_.clear();
                bool ok = true;
                auto visit = [&](uint32_t v) {
                    if (emitted[v]) return;
                    if (in_batch[v] || is_trans(v)) { ok = false; return; }
                    if (std::find(cone.begin(), cone.end(), v) != cone.end()) return;
                    cone.push_back(v);
                    stack_.push_back(v);
                };
                visit(P->nodes[c].a);
                while (ok && !stack_.empty() && cone.size() <= kConeMax) {
                    uint32_t v = stack_.back();
                    stack_.pop_back();
                    const Node& nv = P->nodes[v];
                    if (op_is_unary(nv.op) || op_is_binary(nv.op)) visit(nv.a);
                    if (ok && op_is_binary(nv.op)) visit(nv.b);
                }
                if (!ok || cone.size() > kConeMax) continue;
                std::sort(cone.begin(), cone.end(), [&](uint32_t x, uint32_t y) { return pos[x] < pos[y]; });
                for (uint32_t v : cone) { emitted[v] = 1; out.push_back(v); out_batch.push_back(0); }
                members.push_back(c);
                in_batch[c] = 1;
            }
            uint32_t tag = members.size() > 1 ? ++next_batch : 0;
            for (uint32_t v : members) {
                emitted[v] = 1;
                in_batch[v] = 0;
                out.push_back(v);
                out_batch.push_back(tag);
            }
            if (tag) { st.n_batches++; st.n_batched += uint32_t(members.size()); }
        }
        P->order.swap(out);
        P->batch.swap(out_batch);
    }
    P->stats = st;
    j->ok = true;
}

}  // namespace

bool lower_scene(const Scene& scene, const std::vector<TextureDim>& textures, Program* out, std::string* err) {
    std::string local;
    LowerJob j{&scene, &textures, out, err ? err : &local, false};
    if (!run_with_big_stack(lower_job, &j)) {
        if (err) *err = "cannot start the lowering thread (1 GiB stack unavailable)";
        return false;
    }
    return j.ok;
}

}  // namespace maray
