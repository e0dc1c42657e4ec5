// Host-side schedule compiler (C++, no CUDA): FactorGraph.initialize / has_loops / get_message_schedule /
// treelike_inference (LBP.py:155-245) for a batch of sentence graphs, lowered to dependency levels.
//
// The reference executes the BFS schedule sequentially and in place (Gauss-Seidel), one Python call per message.
// Results after 3 sweeps depend on that order, so it is reproduced literally: the same FIFO BFS with pop-time
// `seen` marking (duplicate edges included), UP pass over reversed(S), DOWN pass over S, one root per sweep.
// Each update is then given the earliest level at which all messages it reads have their sequential value
// (RAW) and nothing it overwrites is still to be read (WAR / WAW).  Updates of one level are independent, so a
// level of the whole batch is ONE leave-one-out launch (K3) plus ONE GEMM launch per potential table (K4).
//
// Unary factors never appear here: their messages are constants (LBP.py:492-498) folded into the per-variable
// unary product U (K1), var->unary-factor messages do not exist (LBP.py:237), and as leaves of the BFS they do
// not change the relative order of the other nodes.
//
// Storage: every message VERSION gets fresh rows, so there are no physical hazards:
//   - a factor->variable update is one GEMM row: it reads row i of its (level, table) block of A and writes row i
//     of the matching block of D;
//   - a variable->factor update writes its result into the A-block row of every later GEMM row that reads that
//     version (0..n destinations; versions nobody reads are dead code and dropped, as are their producers);
//   - messages still at their initial uniform value are filled by mlbp_fill_uniform_rows / read as "row -1";
//   - a factor->variable update that READS an initial uniform message is constant-folded: its result is the
//     table's row / column sums (D rows 1..4, written once per theta), so sweep 1's first level costs no GEMM.
//   - gradient stage: the normaliser Z = c'Tr of a pairwise belief (LBP.py:566-569) needs the row T r (or T'c) of
//     the FINAL messages c, r.  The last factor->variable update of the factor usually read exactly that final
//     version (its producer ran earlier in the same sweep), so its D row is reused and no extra GEMM row is spent.
//
// Blob layout (int32 words), header first:
//   [H_*] fixed header, then per-level records (LEV_WORDS each), then the index arrays they point to.
#include <algorithm>
#include <atomic>
#include <deque>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>
#include <chrono>
#include <cstdio>
#include <memory>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "../../include/mlbp.h"

namespace mlbp {
void set_error(const char *fmt, ...);
}

namespace {

enum {
    H_NLEVELS = 0, H_LEVELS_OFF, H_INIT_N, H_INIT_OFF, H_NPAIR, H_PAIR_C, H_PAIR_U0, H_PAIR_U1, H_PAIR_U2, H_PAIR_GAP1,
    H_PAIR_V0, H_PAIR_V1, H_NGRAD_GEMM, H_GRAD_GEMM_OFF, H_MARG_N, H_MARG_U, H_MARG_OFF, H_MARG_IN, H_NGRAPHS,
    H_A_ROWS, H_D_ROWS, H_MAX_IN, H_NVARS, H_PAIR_R, H_PAIR_Z, H_MSG_BLK_N, H_MSG_BLK_OFF, H_MSG_ROWS, H_SPK_BLK_N, H_PAIR_M0,
    H_PAIR_M1, H_WORDS = 32
};
enum { LEV_NGROUPS = 0, LEV_GRP_U, LEV_GRP_OFF, LEV_IN_ROW, LEV_DEST_OFF, LEV_DEST, LEV_NGEMM, LEV_GEMM, LEV_FIRST, LEV_SECOND, LEV_WORDS = 10 };
enum { GEMM_TABLE = 0, GEMM_A0, GEMM_D0, GEMM_N, GEMM_WORDS = 4 };

struct Op {
    int32_t kind;      // 0: variable -> factor, 1: factor -> variable
    int32_t f, side;   // pairwise factor (local) and which of its variables the message leaves from / goes to
    int32_t level;
    int32_t live;
    int32_t in0, in1;  // range in Graph::inputs (producer op indices, -1 = initial uniform message)
    int32_t row;       // kind 1: index inside its (level, table) block; global A / D row after assignment
    int32_t folded;    // kind 1 reading the initial uniform message: result is a per-table constant row, no GEMM row
    int32_t table;
};

struct Graph {
    int nv = 0, np = 0;
    bool fold = true;                           // constant-fold updates that read the initial uniform message
    std::vector<int32_t> v0, v1, gap1;
    std::vector<std::vector<int32_t>> facset;   // incident pairwise factors per variable, attach order
    std::vector<Op> ops;
    std::vector<int32_t> lvl;                   // ops[i].level, kept densely: the level lookups dominate build_sequence
    std::vector<int32_t> inputs;                // flat producer lists
    std::vector<int32_t> in_edge;               // parallel to inputs: edge id (f * 2 + side) of the message read
    std::vector<int32_t> fin_v2f, fin_f2v;      // producer op of the final version per edge (f * 2 + side)
    std::vector<int32_t> slot;                  // edge (f * 2 + side) -> position of f in facset[variable of that side]
    std::vector<int8_t> zmode;                  // gradient stage, per factor: where Z = c'Tr comes from (see phase A)
    int n_levels = 0;
};

struct Plan {
    std::vector<int32_t> blob;
    int64_t sizes[16];
};

inline int var_of(const Graph &g, int f, int side) { return side == 0 ? g.v0[f] : g.v1[f]; }

bool has_loops(const Graph &g, int root) {                       // LBP.py:174-190
    std::vector<char> seenV(g.nv, 0), seenF(g.np, 0);
    struct It { int node; bool is_var; int parent; };
    std::vector<It> st;
    st.push_back({root, true, -1});
    while (!st.empty()) {
        It n = st.back();
        st.pop_back();
        char &s = n.is_var ? seenV[n.node] : seenF[n.node];
        if (s) return true;
        s = 1;
        if (n.is_var) {
            for (int f : g.facset[n.node])
                if (f != n.parent) st.push_back({f, false, n.node});
        } else {
            const int vs[2] = {g.v0[n.node], g.v1[n.node]};
            for (int v : vs)
                if (v != n.parent) st.push_back({v, true, n.node});
        }
    }
    return false;
}

struct Edge { int child; bool child_is_var; int parent; };     // (child, parent) of LBP.py:165,168

void schedule(const Graph &g, int root, std::vector<Edge> &S) {  // LBP.py:155-172
    S.clear();
    std::vector<char> seenV(g.nv, 0), seenF(g.np, 0);
    struct Nd { int node; bool is_var; };
    std::vector<Nd> q;
    size_t head = 0;
    q.push_back({root, true});
    while (head < q.size()) {
        Nd n = q[head++];
        char &s = n.is_var ? seenV[n.node] : seenF[n.node];
        if (s) continue;
        s = 1;
        if (n.is_var) {
            for (int f : g.facset[n.node])
                if (!seenF[f]) { S.push_back({f, false, n.node}); q.push_back({f, false}); }
        } else {
            const int vs[2] = {g.v0[n.node], g.v1[n.node]};
            for (int v : vs)
                if (!seenV[v]) { S.push_back({v, true, n.node}); q.push_back({v, true}); }
        }
    }
}

// append one update to the sequence, computing its level from the versions it touches
struct Tracker {
    std::vector<int32_t> cur_v2f, cur_f2v;     // producer op per edge, -1 = init
    std::vector<int32_t> rd_v2f, rd_f2v;       // highest level that read the current version
};

inline int lvl_of(const Graph &g, int op) { return op < 0 ? 0 : g.lvl[op]; }

void add_f2v(Graph &g, Tracker &t, int f, int side) {           // FactorNode.update_message_to, LBP.py:499-526
    const int e_out = 2 * f + side, e_in = 2 * f + (1 - side);
    Op op{};
    op.kind = 1; op.f = f; op.side = side; op.live = 0; op.row = -1;
    op.folded = (g.fold && t.cur_v2f[e_in] < 0) ? 1 : 0;
    op.table = g.gap1[f] ? (side == 0 ? MLBP_TABLE_T1 : MLBP_TABLE_T1T) : (side == 0 ? MLBP_TABLE_T : MLBP_TABLE_TT);
    op.in0 = (int32_t)g.inputs.size();
    g.inputs.push_back(t.cur_v2f[e_in]);
    g.in_edge.push_back(e_in);
    op.in1 = (int32_t)g.inputs.size();
    int lv = std::max(lvl_of(g, t.cur_v2f[e_in]), std::max(t.rd_f2v[e_out], lvl_of(g, t.cur_f2v[e_out])));
    op.level = lv + 1;
    t.rd_v2f[e_in] = std::max(t.rd_v2f[e_in], op.level);
    t.cur_f2v[e_out] = (int32_t)g.ops.size();
    t.rd_f2v[e_out] = 0;
    g.ops.push_back(op);
    g.lvl.push_back(op.level);
}

void add_v2f(Graph &g, Tracker &t, int v, int f) {              // VariableNode.update_message_to, LBP.py:377-389
    const int side = (g.v0[f] == v) ? 0 : 1;
    const int e_out = 2 * f + side;
    Op op{};
    op.kind = 0; op.f = f; op.side = side; op.live = 0; op.row = -1; op.table = -1;
    op.in0 = (int32_t)g.inputs.size();
    int lv = std::max(t.rd_v2f[e_out], lvl_of(g, t.cur_v2f[e_out]));
    for (int of : g.facset[v]) {
        if (of == f) continue;
        const int e = 2 * of + ((g.v0[of] == v) ? 0 : 1);
        g.inputs.push_back(t.cur_f2v[e]);
        g.in_edge.push_back(e);
        lv = std::max(lv, lvl_of(g, t.cur_f2v[e]));
    }
    op.in1 = (int32_t)g.inputs.size();
    op.level = lv + 1;
    for (int i = op.in0; i < op.in1; ++i) t.rd_f2v[g.in_edge[i]] = std::max(t.rd_f2v[g.in_edge[i]], op.level);
    t.cur_v2f[e_out] = (int32_t)g.ops.size();
    t.rd_v2f[e_out] = 0;
    g.ops.push_back(op);
    g.lvl.push_back(op.level);
}

void build_sequence(Graph &g, const int32_t *roots, int sweeps) {
    Tracker t;
    t.cur_v2f.assign(2 * g.np, -1); t.cur_f2v.assign(2 * g.np, -1);
    t.rd_v2f.assign(2 * g.np, 0);   t.rd_f2v.assign(2 * g.np, 0);
    const bool loopy = g.np > 0 && has_loops(g, roots[0]);
    const int n_it = sweeps == 0 ? 0 : (loopy ? sweeps : 1);    // LBP.py:219 (0: initialize() only, no treelike_inference yet)
    std::vector<Edge> S;
    for (int it = 0; it < n_it && g.np > 0; ++it) {
        schedule(g, roots[1 + it], S);
        for (size_t i = S.size(); i-- > 0;) {                    // leaves -> root: child sends to parent (LBP.py:227-233)
            const Edge &e = S[i];
            if (e.child_is_var) add_v2f(g, t, e.child, e.parent);
            else add_f2v(g, t, e.child, (g.v0[e.child] == e.parent) ? 0 : 1);
        }
        for (const Edge &e : S) {                                // root -> leaves: parent sends to child (LBP.py:236-242)
            if (e.child_is_var) add_f2v(g, t, e.parent, (g.v0[e.parent] == e.child) ? 0 : 1);
            else add_v2f(g, t, e.parent, e.child);
        }
    }
    g.fin_v2f = t.cur_v2f;
    g.fin_f2v = t.cur_f2v;
    g.n_levels = 0;
    for (const Op &o : g.ops) g.n_levels = std::max(g.n_levels, (int)o.level);
}

}  // namespace

// per-thread output of the emit phase for a contiguous range of graphs
struct ChunkOut {
    std::vector<std::vector<int32_t>> grp_u, grp_off, in_row, dest_off, dest, first, second;   // [level]
    std::vector<int32_t> init_rows, pair_c, pair_r, pair_z, pair_u0, pair_u1, pair_u2, pair_g1, pair_gv0, pair_gv1, mu, moff, min_;
    std::vector<int32_t> pair_m0, pair_m1;                      // flag bit 4: D rows of the final factor->variable messages
    void set_levels(int n_levels) {
        grp_u.resize(n_levels + 1); grp_off.resize(n_levels + 1); in_row.resize(n_levels + 1); dest_off.resize(n_levels + 1);
        dest.resize(n_levels + 1); first.resize(n_levels + 1); second.resize(n_levels + 1);
    }
};

// Where one graph's rows start.  Every row index the emit phase writes is `base + small local index`:
//   blk[level * 4 + table]  A row of the graph's first GEMM row in that (level, table) block (its D row is MLBP_D_CONST_ROWS further)
//   rz / rn [gap class]     gradient-stage copies of r: factors that need a Z GEMM row of their own / the others
//   c                       gradient-stage c rows;  u0 / u1z / u1n / u2z / u2n: the D rows of the gradient-stage GEMMs
//   var                     the graph's first variable
struct Bases {
    const int64_t *blk;
    int64_t rz[2], rn[2], c, u0[2], u1z[2], u1n[2], u2z, u2n, var;
};

struct EmitScratch {
    std::vector<int32_t> dcount, dstart, dflat, ver, tgt;
    std::vector<std::vector<int32_t>> lev_ops;
};

// phase C for ONE graph: global rows, destinations, leave-one-out groups, gradient / marginal index lists appended to `co`
static void emit_graph(const Graph &g, const Bases &B, bool want_grad, bool want_marg, bool want_joint, ChunkOut &co,
                       EmitScratch &sc) {
    auto &dcount = sc.dcount; auto &dstart = sc.dstart; auto &dflat = sc.dflat; auto &ver = sc.ver; auto &tgt = sc.tgt;
    auto &lev_ops = sc.lev_ops;
    if ((int)lev_ops.size() < g.n_levels + 1) lev_ops.resize(g.n_levels + 1);
    auto a_row = [&](const Op &o) -> int32_t { return (int32_t)(B.blk[(size_t)o.level * 4 + o.table] + o.row); };
    // destinations of every variable->factor version = A rows of the GEMM rows that read it (counting sort)
    const size_t nops = g.ops.size();
    dcount.assign(nops + 1, 0);
    // A row of the gradient-stage copy of r for factor f; advances the per-class counters
    auto r_row_of = [&](int f, int64_t *iz, int64_t *in) -> int64_t {
        const int k = g.gap1[f];
        return g.zmode[f] ? B.rn[k] + in[k]++ : B.rz[k] + iz[k]++;
    };
    auto each_consumer = [&](auto &&fn) {
        for (const Op &o : g.ops) {
            if (!o.live || o.kind != 1 || o.folded) continue;
            fn(g.inputs[o.in0], a_row(o));
        }
        if (want_grad) {
            int64_t iz[2] = {0, 0}, in[2] = {0, 0};
            for (int f = 0; f < g.np; ++f) {
                fn(g.fin_v2f[2 * f + 1], (int32_t)r_row_of(f, iz, in));
                fn(g.fin_v2f[2 * f + 0], (int32_t)(B.c + f));
            }
        }
    };
    each_consumer([&](int prod, int32_t row) { if (prod >= 0) ++dcount[prod]; else co.init_rows.push_back(row); });
    dstart.assign(nops + 1, 0);
    for (size_t i = 0; i < nops; ++i) dstart[i + 1] = dstart[i] + dcount[i];
    dflat.resize(dstart[nops]);
    std::fill(dcount.begin(), dcount.end(), 0);
    each_consumer([&](int prod, int32_t row) { if (prod >= 0) dflat[dstart[prod] + dcount[prod]++] = row; });
    if (want_grad) {
        int64_t iz[2] = {0, 0}, in[2] = {0, 0};
        for (int f = 0; f < g.np; ++f) {
            const int k = g.gap1[f];
            const bool zrow = !g.zmode[f];                       // the factor has a Z GEMM row of its own
            const int64_t li = zrow ? iz[k] : in[k];             // index inside its class before r_row_of advances it
            const int64_t rrow = r_row_of(f, iz, in);
            co.pair_c.push_back((int32_t)(B.c + f));
            co.pair_r.push_back((int32_t)rrow);
            if (!zrow) {                                         // Z from the D row of a message update
                const int side = g.zmode[f] - 1;
                co.pair_u0.push_back(MLBP_D_CONST_ROWS + a_row(g.ops[g.fin_f2v[2 * f + side]]));
                co.pair_z.push_back((int32_t)(side == 0 ? B.c + f : rrow));
            } else {
                co.pair_u0.push_back((int32_t)(B.u0[k] + li));
                co.pair_z.push_back((int32_t)(B.c + f));
            }
            co.pair_u1.push_back((int32_t)((zrow ? B.u1z[k] : B.u1n[k]) + li));
            co.pair_u2.push_back(k ? (int32_t)((zrow ? B.u2z : B.u2n) + li) : -1);
            co.pair_g1.push_back(g.gap1[f]);
            co.pair_gv0.push_back((int32_t)(B.var + g.v0[f]));
            co.pair_gv1.push_back((int32_t)(B.var + g.v1[f]));
        }
    }
    auto d_row_of = [&](int prod) -> int32_t {
        if (prod < 0) return -1;
        return g.ops[prod].folded ? 1 + g.ops[prod].table : MLBP_D_CONST_ROWS + a_row(g.ops[prod]);
    };
    // leave-one-out groups: live variable->factor updates of one (level, variable)
    for (auto &v : lev_ops) v.clear();
    for (size_t i = 0; i < nops; ++i)
        if (g.ops[i].live && g.ops[i].kind == 0) lev_ops[g.ops[i].level].push_back((int32_t)i);
    for (int L = 1; L <= g.n_levels; ++L) {
        auto &lo = lev_ops[L];
        if (lo.empty()) continue;
        std::stable_sort(lo.begin(), lo.end(), [&](int32_t x, int32_t y) {
            return var_of(g, g.ops[x].f, g.ops[x].side) < var_of(g, g.ops[y].f, g.ops[y].side);
        });
        size_t i = 0;
        while (i < lo.size()) {
            const int v = var_of(g, g.ops[lo[i]].f, g.ops[lo[i]].side);
            size_t j = i;
            while (j < lo.size() && var_of(g, g.ops[lo[j]].f, g.ops[lo[j]].side) == v) ++j;
            const auto &fs = g.facset[v];
            ver.assign(fs.size(), -2);                   // producer seen by a reader in this group; -2 = nobody reads
            tgt.assign(fs.size(), -1);                   // update that targets this edge
            for (size_t k = i; k < j; ++k) {
                const Op &o = g.ops[lo[k]];
                tgt[g.slot[2 * o.f + o.side]] = lo[k];
                for (int q = o.in0; q < o.in1; ++q) ver[g.slot[g.in_edge[q]]] = g.inputs[q];
            }
            co.grp_u[L].push_back((int32_t)(B.var + v));
            for (size_t s = 0; s < fs.size(); ++s) {
                co.in_row[L].push_back(ver[s] == -2 ? -1 : d_row_of(ver[s]));
                if (tgt[s] >= 0)
                    co.dest[L].insert(co.dest[L].end(), dflat.begin() + dstart[tgt[s]], dflat.begin() + dstart[tgt[s] + 1]);
                // first reader's row per slot (-1: none): spares the kernels one dependent index load
                co.first[L].push_back(tgt[s] >= 0 && dstart[tgt[s] + 1] > dstart[tgt[s]] ? dflat[dstart[tgt[s]]] : -1);
                co.second[L].push_back(tgt[s] >= 0 && dstart[tgt[s] + 1] > dstart[tgt[s]] + 1 ? dflat[dstart[tgt[s]] + 1] : -1);
                co.dest_off[L].push_back((int32_t)co.dest[L].size());
            }
            co.grp_off[L].push_back((int32_t)co.in_row[L].size());
            i = j;
        }
    }
    if (want_joint)                                              // mu rows of the joint log-likelihood (mlbp_joint_logp)
        for (int f = 0; f < g.np; ++f) {
            co.pair_m0.push_back(d_row_of(g.fin_f2v[2 * f + 0]));
            co.pair_m1.push_back(d_row_of(g.fin_f2v[2 * f + 1]));
        }
    if (want_marg)
        for (int v = 0; v < g.nv; ++v) {
            co.mu.push_back((int32_t)(B.var + v));
            for (int f : g.facset[v]) co.min_.push_back(d_row_of(g.fin_f2v[2 * f + ((g.v0[f] == v) ? 0 : 1)]));
            co.moff.push_back((int32_t)co.min_.size());
        }
}

template <class F>
static void parallel_for_chunks(int n_chunks, F f) {
    std::vector<std::thread> th;
    for (int c = 1; c < n_chunks; ++c) th.emplace_back([=] { f(c); });
    f(0);
    for (auto &t : th) t.join();
}

// ---- phase A for ONE graph: wiring, sequence, levels, liveness, Z sources.  Returns 0 or an error code (1 = no variables,
// 2 = bad factor variables, 3 = root out of range)
static int analyse_graph(Graph &g, int nv, int np, const int32_t *v0, const int32_t *v1, const int32_t *gap1, const int32_t *r,
                         int sweeps, int flags, std::vector<char> &needed, int64_t &n_dead) {
    const bool want_grad = flags & 1, want_marg = flags & 2, reuse_z = !(flags & 8);
    g.fold = !(flags & 4);
    g.nv = nv;
    g.np = np;
    if (g.nv <= 0) return 1;
    g.facset.assign(g.nv, {});
    g.v0.resize(g.np); g.v1.resize(g.np); g.gap1.resize(g.np);
    g.slot.resize(2 * (size_t)g.np);
    for (int f = 0; f < g.np; ++f) {
        const int a = v0[f], b = v1[f];
        if (a < 0 || b < 0 || a >= g.nv || b >= g.nv || a == b) return 2;
        g.v0[f] = a; g.v1[f] = b; g.gap1[f] = gap1[f] ? 1 : 0;
        g.slot[2 * f] = (int32_t)g.facset[a].size();
        g.facset[a].push_back(f);
        g.slot[2 * f + 1] = (int32_t)g.facset[b].size();
        g.facset[b].push_back(f);
    }
    for (int i = 0; i <= sweeps; ++i)
        if (r[i] < 0 || r[i] >= g.nv) return 3;
    {   // one allocation per vector: 4 np updates per sweep, a variable update reads deg - 1 messages
        size_t reads = 0;
        for (int v = 0; v < g.nv; ++v) reads += g.facset[v].size() * g.facset[v].size();
        g.ops.reserve((size_t)4 * g.np * sweeps + 8);
        g.lvl.reserve((size_t)4 * g.np * sweeps + 8);
        g.inputs.reserve(((size_t)2 * g.np + reads) * sweeps + 8);
        g.in_edge.reserve(((size_t)2 * g.np + reads) * sweeps + 8);
    }
    build_sequence(g, r, sweeps);
    // liveness, reverse pass: an update is live iff a live update (or a final stage) reads its result
    needed.assign(g.ops.size(), 0);
    for (int e = 0; e < 2 * g.np; ++e) {
        if (want_grad && g.fin_v2f[e] >= 0) needed[g.fin_v2f[e]] = 1;
        if (want_marg && g.fin_f2v[e] >= 0) needed[g.fin_f2v[e]] = 1;
    }
    for (size_t i = g.ops.size(); i-- > 0;) {
        Op &o = g.ops[i];
        o.live = needed[i];
        if (!o.live) { ++n_dead; continue; }
        for (int k = o.in0; k < o.in1; ++k)
            if (g.inputs[k] >= 0) needed[g.inputs[k]] = 1;
    }
    // Z source per factor: 1 = D row of the last f->v0 update (= T r, dot with c), 2 = D row of the last
    // f->v1 update (= T'c, dot with r), 0 = a GEMM row of its own
    g.zmode.assign(g.np, 0);
    if (want_grad && reuse_z)
        for (int f = 0; f < g.np; ++f)
            for (int side = 0; side < 2 && !g.zmode[f]; ++side) {
                const int o = g.fin_f2v[2 * f + side], src = g.fin_v2f[2 * f + (1 - side)];
                if (o >= 0 && src >= 0 && g.ops[o].live && !g.ops[o].folded && g.inputs[g.ops[o].in0] == src)
                    g.zmode[f] = (int8_t)(1 + side);
            }
    return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// Schedule TEMPLATES.  Everything phases A and C derive for a graph depends only on its wiring (variables of every pairwise
// factor, gap classes), its roots and the flags -- not on where its rows land in the batch: every emitted index is
// `base of one of the graph's row segments + small local index` (struct Bases).  A training corpus repeats a few wirings
// (create_factor_graph builds a clique over the predicted tokens of a sentence, train.py:255-330) and draws the roots from a
// small set, so a template is compiled once per (wiring, roots, flags) with SYMBOLIC bases -- entry = segment << 16 | local --
// and kept; an instance of it is a relocation: entry -> base[segment] + local.  The literal path below stays as the
// fallback (graphs too large for the 16-bit local index) and as the cross-check of the tests (MLBP_PLAN_TEMPLATES=0).
namespace {

enum { SEG_LIT = 0, SEG_BLK0 = 1, SEG_GRAD = 32700, SEG_RZ = SEG_GRAD, SEG_RN = SEG_GRAD + 2, SEG_C = SEG_GRAD + 4,
       SEG_U0 = SEG_GRAD + 5, SEG_U1Z = SEG_GRAD + 7, SEG_U1N = SEG_GRAD + 9, SEG_U2Z = SEG_GRAD + 11, SEG_U2N = SEG_GRAD + 12,
       SEG_VAR = SEG_GRAD + 13, SEG_N = 32768 };
constexpr int64_t LOCAL_MAX = 65536 - 16;

struct Tmpl {
    int err = 0;                                 // analyse_graph's code; -1 = valid but too large for the 16-bit local index
    int nv = 0, np = 0, n_levels = 0, max_in = 0;
    int64_t n_dead = 0, nz[2] = {0, 0}, nn[2] = {0, 0};
    std::vector<int32_t> lt, lt_rows;            // (level * 4 + table) blocks this graph has GEMM rows in, and how many
    ChunkOut co;                                 // emit_graph's output for the graph alone, symbolic bases
    size_t bytes = 0;
};

struct KeyHash {
    size_t operator()(const std::vector<int32_t> &k) const {
        uint64_t h = 1469598103934665603ull;
        for (int32_t x : k) { h ^= (uint32_t)x; h *= 1099511628211ull; }
        return (size_t)h;
    }
};

std::mutex g_tmpl_mutex;
std::unordered_map<std::vector<int32_t>, std::shared_ptr<const Tmpl>, KeyHash> g_tmpl_cache;
size_t g_tmpl_bytes = 0;
int64_t g_tmpl_hits = 0, g_tmpl_misses = 0;

size_t chunk_bytes(const ChunkOut &co) {
    size_t n = 0;
    for (auto *vv : {&co.grp_u, &co.grp_off, &co.in_row, &co.dest_off, &co.dest, &co.first, &co.second})
        for (const auto &v : *vv) n += v.capacity();
    for (auto *v : {&co.init_rows, &co.pair_c, &co.pair_r, &co.pair_z, &co.pair_u0, &co.pair_u1, &co.pair_u2, &co.pair_g1,
                    &co.pair_gv0, &co.pair_gv1, &co.mu, &co.moff, &co.min_, &co.pair_m0, &co.pair_m1})
        n += v->capacity();
    return n * sizeof(int32_t);
}

std::shared_ptr<const Tmpl> build_template(int nv, int np, const int32_t *v0, const int32_t *v1, const int32_t *gap1,
                                           const int32_t *r, int sweeps, int flags) {
    auto T = std::make_shared<Tmpl>();
    Graph g;
    std::vector<char> needed;
    T->nv = nv; T->np = np;
    T->err = analyse_graph(g, nv, np, v0, v1, gap1, r, sweeps, flags, needed, T->n_dead);
    if (T->err) return T;
    const bool want_grad = flags & 1, want_marg = flags & 2, want_joint = want_grad && want_marg && (flags & 16);
    T->n_levels = g.n_levels;
    for (int v = 0; v < g.nv; ++v) T->max_in = std::max(T->max_in, (int)g.facset[v].size());
    const size_t LT = (size_t)(g.n_levels + 1) * 4;
    if ((int64_t)LT + SEG_BLK0 >= SEG_GRAD || (int64_t)g.ops.size() >= LOCAL_MAX || nv >= LOCAL_MAX || np >= LOCAL_MAX) { T->err = -1; return T; }
    // local rows inside each (level, table) block, in op order (what phase B of the literal path assigns)
    std::vector<int32_t> cnt(LT, 0);
    for (Op &o : g.ops)
        if (o.live && o.kind == 1 && !o.folded) o.row = cnt[(size_t)o.level * 4 + o.table]++;
    for (size_t i = 0; i < LT; ++i)
        if (cnt[i]) { T->lt.push_back((int32_t)i); T->lt_rows.push_back(cnt[i]); }
    if (want_grad)
        for (int f = 0; f < g.np; ++f) (g.zmode[f] ? T->nn : T->nz)[g.gap1[f]]++;
    std::vector<int64_t> blk(LT);
    for (size_t i = 0; i < LT; ++i) blk[i] = (int64_t)(SEG_BLK0 + i) << 16;
    Bases B;
    B.blk = blk.data();
    auto S = [](int seg) { return (int64_t)seg << 16; };
    for (int k = 0; k < 2; ++k) { B.rz[k] = S(SEG_RZ + k); B.rn[k] = S(SEG_RN + k); B.u0[k] = S(SEG_U0 + k); B.u1z[k] = S(SEG_U1Z + k); B.u1n[k] = S(SEG_U1N + k); }
    B.c = S(SEG_C); B.u2z = S(SEG_U2Z); B.u2n = S(SEG_U2N); B.var = S(SEG_VAR);
    EmitScratch sc;
    T->co.set_levels(g.n_levels);
    emit_graph(g, B, want_grad, want_marg, want_joint, T->co, sc);
    T->bytes = chunk_bytes(T->co) + 256;
    return T;
}

// relocation of one template entry
inline int32_t reloc(int32_t x, const int64_t *SB) { return x < 65536 ? x : (int32_t)(SB[x >> 16] + (x & 0xffff)); }
inline void append_reloc(std::vector<int32_t> &dst, const std::vector<int32_t> &src, const int64_t *SB) {
    const size_t n0 = dst.size();
    dst.resize(n0 + src.size());
    int32_t *d = dst.data() + n0;
    for (size_t i = 0; i < src.size(); ++i) d[i] = reloc(src[i], SB);
}
inline void append_shift(std::vector<int32_t> &dst, const std::vector<int32_t> &src, int32_t shift) {
    const size_t n0 = dst.size();
    dst.resize(n0 + src.size());
    int32_t *d = dst.data() + n0;
    for (size_t i = 0; i < src.size(); ++i) d[i] = src[i] + shift;
}

}  // namespace

extern "C" int mlbp_plan_compile(int n_graphs, const int32_t *var_off, const int32_t *pair_off, const int32_t *pair_v0,
                                 const int32_t *pair_v1, const int32_t *pair_gap1, const int32_t *roots, int sweeps,
                                 int flags, mlbp_plan **out) {
    if (!out || n_graphs < 0 || sweeps < 0 || !var_off || !pair_off || !roots) {
        mlbp::set_error("plan_compile: bad argument");
        return MLBP_ERR_INVALID;
    }
    const bool want_grad = flags & 1, want_marg = flags & 2, want_joint = want_grad && want_marg && (flags & 16);
    const bool prof = std::getenv("MLBP_PLAN_PROFILE") != nullptr;
    auto tnow = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_a = tnow();
    unsigned hw = std::thread::hardware_concurrency();
    const char *env = std::getenv("MLBP_PLAN_THREADS");
    int n_chunks = env ? std::atoi(env) : (int)std::min<unsigned>(hw ? hw : 1, 32);
    n_chunks = std::max(1, std::min(n_chunks, (n_graphs + 15) / 16));
    auto chunk_lo = [&](int c) { return (int)((int64_t)n_graphs * c / n_chunks); };
    const char *env_t = std::getenv("MLBP_PLAN_TEMPLATES");
    bool templated = !(env_t && std::atoi(env_t) == 0);
    auto bad_graph = [](int code) {
        mlbp::set_error("plan_compile: invalid graph (code %d: 1 = no variables, 2 = bad factor variables, 3 = root out of range)", code);
        return MLBP_ERR_INVALID;
    };

    int n_levels = 0, max_in = 0;
    int64_t n_dead = 0;
    std::vector<int64_t> cnt, base;
    size_t LT = 0;
    int64_t n_pair = 0, n_z[2] = {0, 0}, n_n[2] = {0, 0}, n_gap0 = 0, n_gap1 = 0, n_msg_rows = 0, a_rows = 0, d_rows = 0;
    int64_t a_r0 = 0, a_r1 = 0, a_c = 0, d_u0_0 = 0, d_u1_0 = 0, d_u0_1 = 0, d_u1_1 = 0, d_u2_1 = 0;
    // block bases and the gradient-stage layout from the per-(level, table) row counts and the pair counts
    auto layout = [&]() -> bool {
        n_gap0 = n_z[0] + n_n[0]; n_gap1 = n_z[1] + n_n[1];
        base.assign(LT, 0);
        a_rows = 0;
        for (int L = 1; L <= n_levels; ++L)
            for (int t = 0; t < 4; ++t) { base[(size_t)L * 4 + t] = a_rows; a_rows += cnt[(size_t)L * 4 + t]; }
        n_msg_rows = a_rows;
        // gradient stage: r rows (gap>1 block, gap==1 block), then the c rows; D row = 1 + A row for message rows
        a_r0 = a_rows; a_r1 = a_r0 + n_gap0; a_c = a_r1 + n_gap1;
        a_rows = a_c + n_pair;
        d_rows = MLBP_D_CONST_ROWS + n_msg_rows;
        d_u0_0 = d_rows; d_u1_0 = d_u0_0 + n_z[0]; d_u0_1 = d_u1_0 + n_gap0; d_u1_1 = d_u0_1 + n_z[1]; d_u2_1 = d_u1_1 + n_gap1;
        if (want_grad) d_rows = d_u2_1 + n_gap1;
        return !(a_rows > 0x7fffff00ll || d_rows > 0x7fffff00ll);
    };
    // first rows of graph gi's segments (gradient stage and variables; the (level, table) blocks are set by the caller)
    std::vector<int64_t> g_iz[2], g_in[2], g_ip(n_graphs);
    for (int k = 0; k < 2; ++k) { g_iz[k].resize(n_graphs); g_in[k].resize(n_graphs); }
    auto grad_bases = [&](int gi, Bases &B) {
        for (int k = 0; k < 2; ++k) {
            const int64_t blk = k ? a_r1 : a_r0, du0 = k ? d_u0_1 : d_u0_0, du1 = k ? d_u1_1 : d_u1_0;
            B.rz[k] = blk + g_iz[k][gi];
            B.rn[k] = blk + n_z[k] + g_in[k][gi];
            B.u0[k] = du0 + g_iz[k][gi];
            B.u1z[k] = du1 + g_iz[k][gi];
            B.u1n[k] = du1 + n_z[k] + g_in[k][gi];
        }
        B.u2z = d_u2_1 + g_iz[1][gi];
        B.u2n = d_u2_1 + n_z[1] + g_in[1][gi];
        B.c = a_c + g_ip[gi];
        B.var = var_off[gi];
    };
    std::vector<ChunkOut> CO(n_chunks);
    double t_b = t_a, t_c = t_a;
    int64_t hits = 0, misses = 0;

    if (templated) {
        // ---- phase A (parallel): one template per distinct (wiring, roots, flags), looked up or compiled
        std::vector<std::shared_ptr<const Tmpl>> TP(n_graphs);
        std::vector<int64_t> c_hits(n_chunks, 0), c_miss(n_chunks, 0);
        size_t cache_cap = (size_t)1024 << 20;
        if (const char *e = std::getenv("MLBP_PLAN_CACHE_MB")) cache_cap = (size_t)std::max(0, std::atoi(e)) << 20;
        parallel_for_chunks(n_chunks, [&](int c) {
            std::vector<int32_t> key, uf;
            for (int gi = chunk_lo(c); gi < chunk_lo(c + 1); ++gi) {
                const int nv = var_off[gi + 1] - var_off[gi], np = pair_off[gi + 1] - pair_off[gi], po = pair_off[gi];
                const int32_t *r = roots + (size_t)gi * (1 + sweeps);
                key.clear();
                key.push_back(nv); key.push_back(np); key.push_back(sweeps); key.push_back(flags & 31);
                // r[0] only feeds has_loops (LBP.py:176), whose answer does not depend on the start node when the graph is
                // connected (create_factor_graph's cliques are): then it is left out of the key (union-find over the factors)
                int first_root = r[0];
                if (nv > 0 && nv < 65536 && r[0] >= 0 && r[0] < nv) {
                    uf.resize(nv);
                    for (int v = 0; v < nv; ++v) uf[v] = v;
                    auto find = [&](int x) { while (uf[x] != x) { uf[x] = uf[uf[x]]; x = uf[x]; } return x; };
                    int comps = nv;
                    bool ok = true;
                    for (int f = 0; f < np && ok; ++f) {
                        const int a = pair_v0[po + f], b = pair_v1[po + f];
                        if (a < 0 || b < 0 || a >= nv || b >= nv) { ok = false; break; }
                        const int ra = find(a), rb = find(b);
                        if (ra != rb) { uf[ra] = rb; --comps; }
                    }
                    if (ok && comps == 1) first_root = -1;
                }
                key.push_back(first_root);
                key.insert(key.end(), r + 1, r + 1 + sweeps);
                if (np > 0) {
                    key.insert(key.end(), pair_v0 + po, pair_v0 + po + np);
                    key.insert(key.end(), pair_v1 + po, pair_v1 + po + np);
                    for (int f = 0; f < np; ++f) key.push_back(pair_gap1[po + f] ? 1 : 0);
                }
                std::shared_ptr<const Tmpl> T;
                {
                    std::lock_guard<std::mutex> lk(g_tmpl_mutex);
                    auto it = g_tmpl_cache.find(key);
                    if (it != g_tmpl_cache.end()) T = it->second;
                }
                if (T) { ++c_hits[c]; }
                else {
                    ++c_miss[c];
                    T = build_template(nv, np, pair_v0 + po, pair_v1 + po, pair_gap1 + po, r, sweeps, flags);
                    if (T->err <= 0 && cache_cap > 0) {
                        std::lock_guard<std::mutex> lk(g_tmpl_mutex);
                        if (g_tmpl_bytes + T->bytes > cache_cap) { g_tmpl_cache.clear(); g_tmpl_bytes = 0; }   // (templates in use stay alive)
                        if (g_tmpl_cache.emplace(key, T).second) g_tmpl_bytes += T->bytes + key.size() * sizeof(int32_t);
                    }
                }
                TP[gi] = T;
            }
        });
        for (int c = 0; c < n_chunks; ++c) { hits += c_hits[c]; misses += c_miss[c]; }
        {
            std::lock_guard<std::mutex> lk(g_tmpl_mutex);
            g_tmpl_hits += hits; g_tmpl_misses += misses;
        }
        for (int gi = 0; gi < n_graphs && templated; ++gi) {
            if (TP[gi]->err > 0) return bad_graph(TP[gi]->err);
            if (TP[gi]->err < 0) templated = false;              // too large for the 16-bit local index: literal path for the batch
        }
        if (templated) {
            for (int gi = 0; gi < n_graphs; ++gi) {
                n_levels = std::max(n_levels, TP[gi]->n_levels); max_in = std::max(max_in, TP[gi]->max_in); n_dead += TP[gi]->n_dead;
            }
            t_b = tnow();
            // ---- phase B (serial, cheap): one A/D block per (level, table); rows inside a block in graph order
            LT = (size_t)(n_levels + 1) * 4;
            cnt.assign(LT, 0);
            std::vector<int64_t> gb_off(n_graphs + 1, 0);
            for (int gi = 0; gi < n_graphs; ++gi) gb_off[gi + 1] = gb_off[gi] + (int64_t)TP[gi]->lt.size();
            std::vector<int64_t> gb(gb_off[n_graphs]);            // first row (inside the block) of each graph's used blocks
            for (int gi = 0; gi < n_graphs; ++gi) {
                const Tmpl &T = *TP[gi];
                int64_t *g0 = gb.data() + gb_off[gi];
                for (size_t j = 0; j < T.lt.size(); ++j) { g0[j] = cnt[T.lt[j]]; cnt[T.lt[j]] += T.lt_rows[j]; }
                for (int k = 0; k < 2; ++k) { g_iz[k][gi] = n_z[k]; g_in[k][gi] = n_n[k]; n_z[k] += T.nz[k]; n_n[k] += T.nn[k]; }
                g_ip[gi] = n_pair;
                if (want_grad) n_pair += T.np;
            }
            if (!layout()) { mlbp::set_error("plan_compile: batch too large"); return MLBP_ERR_INVALID; }
            t_c = tnow();
            // ---- phase C (parallel): every graph's template relocated to its rows
            parallel_for_chunks(n_chunks, [&](int c) {
                ChunkOut &co = CO[c];
                co.set_levels(n_levels);
                std::vector<int64_t> SB(SEG_N, 0);
                {   // one allocation per output vector
                    std::vector<size_t> need(7 * (size_t)(n_levels + 1), 0);
                    size_t flat[13] = {0};
                    for (int gi = chunk_lo(c); gi < chunk_lo(c + 1); ++gi) {
                        const ChunkOut &t = TP[gi]->co;
                        for (int L = 1; L <= TP[gi]->n_levels; ++L) {
                            size_t *n = &need[7 * (size_t)L];
                            n[0] += t.grp_u[L].size(); n[1] += t.grp_off[L].size(); n[2] += t.in_row[L].size(); n[3] += t.dest_off[L].size();
                            n[4] += t.dest[L].size(); n[5] += t.first[L].size(); n[6] += t.second[L].size();
                        }
                        flat[0] += t.init_rows.size(); flat[1] += t.pair_c.size(); flat[2] += t.mu.size(); flat[3] += t.moff.size(); flat[4] += t.min_.size();
                    }
                    for (int L = 1; L <= n_levels; ++L) {
                        const size_t *n = &need[7 * (size_t)L];
                        co.grp_u[L].reserve(n[0]); co.grp_off[L].reserve(n[1]); co.in_row[L].reserve(n[2]); co.dest_off[L].reserve(n[3]);
                        co.dest[L].reserve(n[4]); co.first[L].reserve(n[5]); co.second[L].reserve(n[6]);
                    }
                    co.init_rows.reserve(flat[0]);
                    for (auto *v : {&co.pair_c, &co.pair_r, &co.pair_z, &co.pair_u0, &co.pair_u1, &co.pair_u2, &co.pair_g1, &co.pair_gv0, &co.pair_gv1,
                                    &co.pair_m0, &co.pair_m1})
                        v->reserve(flat[1]);
                    co.mu.reserve(flat[2]); co.moff.reserve(flat[3]); co.min_.reserve(flat[4]);
                }
                for (int gi = chunk_lo(c); gi < chunk_lo(c + 1); ++gi) {
                    const Tmpl &T = *TP[gi];
                    const int64_t *g0 = gb.data() + gb_off[gi];
                    for (size_t j = 0; j < T.lt.size(); ++j) SB[SEG_BLK0 + T.lt[j]] = base[T.lt[j]] + g0[j];
                    Bases B;
                    B.blk = nullptr;
                    grad_bases(gi, B);
                    for (int k = 0; k < 2; ++k) {
                        SB[SEG_RZ + k] = B.rz[k]; SB[SEG_RN + k] = B.rn[k]; SB[SEG_U0 + k] = B.u0[k]; SB[SEG_U1Z + k] = B.u1z[k]; SB[SEG_U1N + k] = B.u1n[k];
                    }
                    SB[SEG_C] = B.c; SB[SEG_U2Z] = B.u2z; SB[SEG_U2N] = B.u2n; SB[SEG_VAR] = B.var;
                    const int64_t *sb = SB.data();
                    const ChunkOut &t = T.co;
                    for (int L = 1; L <= T.n_levels; ++L) {
                        if (t.grp_u[L].empty()) continue;
                        append_shift(co.grp_off[L], t.grp_off[L], (int32_t)co.in_row[L].size());
                        append_shift(co.dest_off[L], t.dest_off[L], (int32_t)co.dest[L].size());
                        append_reloc(co.grp_u[L], t.grp_u[L], sb);
                        append_reloc(co.in_row[L], t.in_row[L], sb);
                        append_reloc(co.dest[L], t.dest[L], sb);
                        append_reloc(co.first[L], t.first[L], sb);
                        append_reloc(co.second[L], t.second[L], sb);
                    }
                    append_reloc(co.init_rows, t.init_rows, sb);
                    append_reloc(co.pair_c, t.pair_c, sb); append_reloc(co.pair_r, t.pair_r, sb); append_reloc(co.pair_z, t.pair_z, sb);
                    append_reloc(co.pair_u0, t.pair_u0, sb); append_reloc(co.pair_u1, t.pair_u1, sb); append_reloc(co.pair_u2, t.pair_u2, sb);
                    co.pair_g1.insert(co.pair_g1.end(), t.pair_g1.begin(), t.pair_g1.end());
                    append_reloc(co.pair_gv0, t.pair_gv0, sb); append_reloc(co.pair_gv1, t.pair_gv1, sb);
                    append_reloc(co.pair_m0, t.pair_m0, sb); append_reloc(co.pair_m1, t.pair_m1, sb);
                    append_shift(co.moff, t.moff, (int32_t)co.min_.size());
                    append_reloc(co.mu, t.mu, sb);
                    append_reloc(co.min_, t.min_, sb);
                }
            });
        }
    }

    if (!templated) {
        n_levels = max_in = 0; n_dead = 0;
        for (auto &co : CO) co = ChunkOut();
        // ---- phase A (parallel): sequence, levels, liveness per graph
        std::vector<Graph> G(n_graphs);
        std::vector<int> err(n_chunks, 0), c_levels(n_chunks, 0), c_maxin(n_chunks, 0);
        std::vector<int64_t> c_dead(n_chunks, 0);
        parallel_for_chunks(n_chunks, [&](int c) {
            std::vector<char> needed;
            for (int gi = chunk_lo(c); gi < chunk_lo(c + 1); ++gi) {
                Graph &g = G[gi];
                const int po = pair_off[gi];
                err[c] = analyse_graph(g, var_off[gi + 1] - var_off[gi], pair_off[gi + 1] - po, pair_v0 + po, pair_v1 + po, pair_gap1 + po,
                                       roots + (size_t)gi * (1 + sweeps), sweeps, flags, needed, c_dead[c]);
                if (err[c]) return;
                c_levels[c] = std::max(c_levels[c], g.n_levels);
                for (int v = 0; v < g.nv; ++v) c_maxin[c] = std::max(c_maxin[c], (int)g.facset[v].size());
            }
        });
        for (int c = 0; c < n_chunks; ++c) {
            if (err[c]) return bad_graph(err[c]);
            n_levels = std::max(n_levels, c_levels[c]); max_in = std::max(max_in, c_maxin[c]); n_dead += c_dead[c];
        }

        t_b = tnow();
        // ---- phase B (serial, cheap): one A/D block per (level, table); rows inside a block in graph order
        LT = (size_t)(n_levels + 1) * 4;
        cnt.assign(LT, 0);
        std::vector<int64_t> gbase((size_t)n_graphs * LT);            // first row index (inside the block) of each graph
        n_pair = 0; n_z[0] = n_z[1] = n_n[0] = n_n[1] = 0;
        for (int gi = 0; gi < n_graphs; ++gi) {
            Graph &g = G[gi];
            int64_t *gb = &gbase[(size_t)gi * LT];
            for (size_t i = 0; i < LT; ++i) gb[i] = cnt[i];
            for (Op &o : g.ops)
                if (o.live && o.kind == 1 && !o.folded) o.row = (int32_t)(cnt[(size_t)o.level * 4 + o.table]++ - gb[(size_t)o.level * 4 + o.table]);
            for (int k = 0; k < 2; ++k) { g_iz[k][gi] = n_z[k]; g_in[k][gi] = n_n[k]; }
            g_ip[gi] = n_pair;
            if (want_grad) { n_pair += g.np; for (int f = 0; f < g.np; ++f) (g.zmode[f] ? n_n : n_z)[g.gap1[f]]++; }
        }
        if (!layout()) { mlbp::set_error("plan_compile: batch too large"); return MLBP_ERR_INVALID; }

        t_c = tnow();
        // ---- phase C (parallel): global rows, destinations, leave-one-out groups per chunk
        parallel_for_chunks(n_chunks, [&](int c) {
            ChunkOut &co = CO[c];
            co.set_levels(n_levels);
            EmitScratch sc;
            std::vector<int64_t> blk(LT);
            for (int gi = chunk_lo(c); gi < chunk_lo(c + 1); ++gi) {
                const int64_t *gb = &gbase[(size_t)gi * LT];
                for (size_t i = 0; i < LT; ++i) blk[i] = base[i] + gb[i];
                Bases B;
                B.blk = blk.data();
                grad_bases(gi, B);
                emit_graph(G[gi], B, want_grad, want_marg, want_joint, co, sc);
            }
        });
    }

    double t_d = tnow();
    // ---- phase D: merge the chunks into the blob
    Plan *P = new (std::nothrow) Plan();
    if (!P) { mlbp::set_error("plan_compile: out of memory"); return MLBP_ERR_ALLOC; }
    std::vector<int32_t> &B = P->blob;
    // The header and the level records are written in place; every index array is only PLACED here (offset + copy job) and
    // copied by all threads once the total size is known: the merge is memory traffic, 25 MB per 512 C3 sentences.
    struct Job { size_t dst; const int32_t *src; size_t n; int32_t shift; };
    std::vector<Job> jobs;
    std::deque<std::vector<int32_t>> owned;                                   // small arrays built here (GEMM records)
    size_t pos = H_WORDS + (size_t)n_levels * LEV_WORDS;
    B.assign(pos, 0);
    auto append = [&](const std::vector<int32_t> &v) {
        owned.push_back(v);
        const int32_t o = (int32_t)pos;
        jobs.push_back({pos, owned.back().data(), v.size(), 0});
        pos += v.size();
        return o;
    };
    // concatenation of one member over the chunks; `csr` adds a running offset (CSR offsets) and prepends a 0
    auto concat = [&](auto member, bool csr) {
        const int32_t o = (int32_t)pos;
        int32_t run = 0;
        if (csr) ++pos;                                                        // the leading 0 (the blob is zero-filled)
        for (int c = 0; c < n_chunks; ++c) {
            const std::vector<int32_t> &v = member(CO[c]);
            if (v.empty()) continue;
            jobs.push_back({pos, v.data(), v.size(), csr ? run : 0});
            pos += v.size();
            if (csr) run += v.back();
        }
        return o;
    };
    B[H_NLEVELS] = n_levels; B[H_LEVELS_OFF] = H_WORDS; B[H_NGRAPHS] = n_graphs;
    B[H_A_ROWS] = (int32_t)a_rows; B[H_D_ROWS] = (int32_t)d_rows; B[H_MAX_IN] = max_in; B[H_NVARS] = var_off[n_graphs];
    std::vector<int32_t> msg_blocks;                               // every message GEMM block, ascending in A / D rows
    for (int L = 1; L <= n_levels; ++L) {
        int32_t ng = 0;
        for (int c = 0; c < n_chunks; ++c) ng += (int32_t)CO[c].grp_u[L].size();
        const int32_t o_u = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.grp_u[L]; }, false);
        const int32_t o_off = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.grp_off[L]; }, true);
        const int32_t o_in = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.in_row[L]; }, false);
        const int32_t o_doff = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.dest_off[L]; }, true);
        const int32_t o_dest = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.dest[L]; }, false);
        const int32_t o_first = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.first[L]; }, false);
        const int32_t o_second = concat([&](ChunkOut &x) -> std::vector<int32_t> & { return x.second[L]; }, false);
        std::vector<int32_t> gemm;
        for (int t = 0; t < 4; ++t)
            if (cnt[(size_t)L * 4 + t] > 0) {
                gemm.push_back(t);
                gemm.push_back((int32_t)base[(size_t)L * 4 + t]);
                gemm.push_back((int32_t)(MLBP_D_CONST_ROWS + base[(size_t)L * 4 + t]));
                gemm.push_back((int32_t)cnt[(size_t)L * 4 + t]);
            }
        const int32_t o_gemm = append(gemm);
        msg_blocks.insert(msg_blocks.end(), gemm.begin(), gemm.end());
        const size_t rec = H_WORDS + (size_t)(L - 1) * LEV_WORDS;
        B[rec + LEV_NGROUPS] = ng; B[rec + LEV_GRP_U] = o_u; B[rec + LEV_GRP_OFF] = o_off; B[rec + LEV_IN_ROW] = o_in;
        B[rec + LEV_DEST_OFF] = o_doff; B[rec + LEV_DEST] = o_dest; B[rec + LEV_NGEMM] = (int32_t)(gemm.size() / GEMM_WORDS);
        B[rec + LEV_GEMM] = o_gemm; B[rec + LEV_FIRST] = o_first; B[rec + LEV_SECOND] = o_second;
    }
    {
        int32_t n_init = 0;
        for (int c = 0; c < n_chunks; ++c) n_init += (int32_t)CO[c].init_rows.size();
        B[H_INIT_N] = n_init;
        B[H_INIT_OFF] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.init_rows; }, false);
    }
    // flat copy of the per-level GEMM records {table, A row, D row, rows}: the exact re-score (rescore.cu) finds the table of
    // a message's D row by bisection over it
    B[H_MSG_BLK_N] = (int32_t)(msg_blocks.size() / GEMM_WORDS);
    // ... followed by the two row ranges of the gradient stage's r copies (gap > 1, gap == 1): together the list of A-row
    // ranges whose spikes the var->factor kernel files per block (H_SPK_BLK_N entries)
    if (want_grad && n_gap0 > 0) { msg_blocks.push_back(MLBP_TABLE_G); msg_blocks.push_back((int32_t)a_r0); msg_blocks.push_back((int32_t)d_u1_0); msg_blocks.push_back((int32_t)n_gap0); }
    if (want_grad && n_gap1 > 0) { msg_blocks.push_back(MLBP_TABLE_G1); msg_blocks.push_back((int32_t)a_r1); msg_blocks.push_back((int32_t)d_u1_1); msg_blocks.push_back((int32_t)n_gap1); }
    B[H_SPK_BLK_N] = (int32_t)(msg_blocks.size() / GEMM_WORDS);
    B[H_MSG_BLK_OFF] = append(msg_blocks);
    B[H_MSG_ROWS] = (int32_t)n_msg_rows;
    B[H_NPAIR] = (int32_t)n_pair;
    B[H_PAIR_C] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_c; }, false);
    B[H_PAIR_R] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_r; }, false);
    B[H_PAIR_Z] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_z; }, false);
    B[H_PAIR_U0] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_u0; }, false);
    B[H_PAIR_U1] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_u1; }, false);
    B[H_PAIR_U2] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_u2; }, false);
    B[H_PAIR_GAP1] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_g1; }, false);
    B[H_PAIR_V0] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_gv0; }, false);
    B[H_PAIR_V1] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_gv1; }, false);
    {
        std::vector<int32_t> gg;
        auto call = [&](int table, int64_t a0, int64_t d0, int64_t n) {
            if (n > 0) { gg.push_back(table); gg.push_back((int32_t)a0); gg.push_back((int32_t)d0); gg.push_back((int32_t)n); }
        };
        if (want_grad) {
            call(MLBP_TABLE_T, a_r0, d_u0_0, n_z[0]);  call(MLBP_TABLE_G, a_r0, d_u1_0, n_gap0);
            call(MLBP_TABLE_T1, a_r1, d_u0_1, n_z[1]); call(MLBP_TABLE_G1, a_r1, d_u1_1, n_gap1);
            call(MLBP_TABLE_G1W, a_r1, d_u2_1, n_gap1);
        }
        B[H_NGRAD_GEMM] = (int32_t)(gg.size() / GEMM_WORDS);
        B[H_GRAD_GEMM_OFF] = append(gg);
    }
    {
        int32_t nm = 0;
        for (int c = 0; c < n_chunks; ++c) nm += (int32_t)CO[c].mu.size();
        B[H_MARG_N] = nm;
        B[H_MARG_U] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.mu; }, false);
        B[H_MARG_OFF] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.moff; }, true);
        B[H_MARG_IN] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.min_; }, false);
    }
    if (want_joint) {                                              // last, so that everything before is the blob without flag bit 4
        B[H_PAIR_M0] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_m0; }, false);
        B[H_PAIR_M1] = concat([](ChunkOut &x) -> std::vector<int32_t> & { return x.pair_m1; }, false);
    }
    if (pos > 0x7fffff00ull) { delete P; mlbp::set_error("plan_compile: batch too large"); return MLBP_ERR_INVALID; }
    B.resize(pos, 0);
    {
        std::atomic<size_t> next{0};
        int32_t *dst = B.data();
        parallel_for_chunks(n_chunks, [&](int) {
            for (size_t j = next.fetch_add(1); j < jobs.size(); j = next.fetch_add(1)) {
                const Job &jb = jobs[j];
                if (jb.shift == 0) std::memcpy(dst + jb.dst, jb.src, jb.n * sizeof(int32_t));
                else for (size_t i = 0; i < jb.n; ++i) dst[jb.dst + i] = jb.src[i] + jb.shift;
            }
        });
    }
    int64_t gemm_rows = n_msg_rows + (want_grad ? n_z[0] + n_gap0 + n_z[1] + 2 * n_gap1 : 0);
    std::memset(P->sizes, 0, sizeof(P->sizes));
    P->sizes[MLBP_PLAN_BLOB_WORDS] = (int64_t)B.size();
    P->sizes[MLBP_PLAN_A_ROWS] = a_rows;
    P->sizes[MLBP_PLAN_D_ROWS] = d_rows;
    P->sizes[MLBP_PLAN_N_LEVELS] = n_levels;
    P->sizes[MLBP_PLAN_N_PAIR] = n_pair;
    P->sizes[MLBP_PLAN_N_GEMM_ROWS] = gemm_rows;
    P->sizes[MLBP_PLAN_MAX_IN] = max_in;
    P->sizes[MLBP_PLAN_HDR_WORDS] = H_WORDS;
    P->sizes[MLBP_PLAN_N_DEAD] = n_dead;
    P->sizes[MLBP_PLAN_TMPL_HITS] = hits;
    P->sizes[MLBP_PLAN_TMPL_MISSES] = misses;
    if (prof) std::fprintf(stderr, "plan_compile: A %.1f ms  B %.1f ms  C %.1f ms  D %.1f ms (chunks %d, templates %s: %lld hits, %lld compiled)\n", 1e3 * (t_b - t_a), 1e3 * (t_c - t_b), 1e3 * (t_d - t_c), 1e3 * (tnow() - t_d), n_chunks, templated ? "on" : "off", (long long)hits, (long long)misses);
    *out = reinterpret_cast<mlbp_plan *>(P);
    return MLBP_OK;
}

extern "C" int mlbp_plan_sizes(const mlbp_plan *p, int64_t *h_sizes) {
    if (!p || !h_sizes) { mlbp::set_error("plan_sizes: null"); return MLBP_ERR_INVALID; }
    std::memcpy(h_sizes, reinterpret_cast<const Plan *>(p)->sizes, sizeof(int64_t) * 16);
    return MLBP_OK;
}

extern "C" int mlbp_plan_export(const mlbp_plan *p, int32_t *h_blob) {
    if (!p || !h_blob) { mlbp::set_error("plan_export: null"); return MLBP_ERR_INVALID; }
    const Plan *P = reinterpret_cast<const Plan *>(p);
    std::memcpy(h_blob, P->blob.data(), P->blob.size() * sizeof(int32_t));
    return MLBP_OK;
}

extern "C" void mlbp_plan_destroy(mlbp_plan *p) { delete reinterpret_cast<Plan *>(p); }
