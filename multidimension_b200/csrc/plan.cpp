// plan.cpp — host planner: C-ABI descriptor (mdim_expr) → device Program + kernel choice.
//
// This is the "expression lowering" half that the north star places in src/view.rs, restated for
// a run-time descriptor: it validates the post-order node array, canonicalises the iteration
// space (drops length-1 axes, merges jointly-contiguous neighbours — `Iso`/`Coat` regroupings
// and contiguous arrays of any rank collapse to rank 1), picks the vector width and per-leaf load
// mode, emits the postfix device program, and recognises the shapes that have a dedicated kernel
// (tiled transpose, last-axis fold).  Host-only code; no CUDA calls.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "program.hpp"

namespace mdim {

int dtype_size(int dt) {
    switch (dt) {
        case MDIM_U8: return 1;
        case MDIM_I32: case MDIM_U32: case MDIM_F32: return 4;
        case MDIM_I64: case MDIM_U64: case MDIM_F64: return 8;
    }
    return 0;
}

const char* status_string(int st) {
    switch (st) {
        case MDIM_OK: return "ok";
        case MDIM_ERR_OOB: return "index out of bounds";
        case MDIM_ERR_SIZE: return "size mismatch";
        case MDIM_ERR_UNSUPPORTED: return "expression not lowerable to the device";
        case MDIM_ERR_CUDA: return "CUDA failure or no sm_100 device";
        case MDIM_ERR_ARITH: return "integer division by zero or with overflow";
        case MDIM_ERR_INVALID: return "malformed descriptor";
        case MDIM_ERR_NOMEM: return "out of memory";
        case MDIM_ERR_NCCL: return "NCCL is missing or a collective failed";
    }
    return "unknown status";
}

static bool is_int(int dt) { return dt == MDIM_U8 || dt == MDIM_I32 || dt == MDIM_U32 || dt == MDIM_I64 || dt == MDIM_U64; }
static bool is_float(int dt) { return dt == MDIM_F32 || dt == MDIM_F64; }

static int node_arity(const mdim_node& n) {
    switch (n.kind) {
        case MDIM_NODE_LEAF: case MDIM_NODE_IOTA: case MDIM_NODE_CONST: return 0;
        case MDIM_NODE_UNARY: case MDIM_NODE_DIAG: return 1;
        case MDIM_NODE_FOLD: return n.n_comp == 2 ? 2 : 1;  // (init, body) or body alone (init = imm)
        case MDIM_NODE_BINARY: case MDIM_NODE_CONCAT: return 2;
        case MDIM_NODE_GATHER: return n.n_comp;
        case MDIM_NODE_TUPLE: return n.n_comp;
    }
    return -1;
}

namespace {

struct Why {
    char* buf; size_t len;
    int fail(int st, const char* fmt, ...) {
        if (buf && len) { va_list ap; va_start(ap, fmt); vsnprintf(buf, len, fmt, ap); va_end(ap); }
        return st;
    }
};

struct Builder {
    const mdim_expr* e;
    uint32_t flags;
    Plan* plan;
    Why why;
    int child[MDIM_MAX_NODES][kMaxRank];
    int n_child[MDIM_MAX_NODES];
    bool under_fold[MDIM_MAX_NODES];
    bool has_err_source[MDIM_MAX_NODES];  // subtree contains GATHER or integer DIV/REM
    int fold_node = -1;
    // canonical axes
    int n_axes = 0, rank = 0, red_rank = 0;
    uint64_t len[kMaxRank];
    int axis_map[kMaxRank];  // original axis -> canonical axis, -1 = dropped (coordinate is 0)
    // per original node: canonical strides (LEAF/IOTA/GATHER)
    int64_t cstride[MDIM_MAX_NODES][kMaxRank];
    int depth = 0, max_depth = 0;
    int force_vec = 0;
    // canonical axis g (out axes outermost-first, then reduction axes) -> device program axis:
    // the out axes are stored INNERMOST FIRST, so the vector axis is always program axis 0
    int pa(int g) const { return g < rank ? rank - 1 - g : g; }  // 0 = widest that divides the innermost axis

    int validate();
    void canonical_axes();
    int emit();
    int gen(int ni, int mask_first, int mask_n);
    int push_instr(const Instr& in);
    int detect_fast_paths();
    bool detect_fold_split();
};

int Builder::validate() {
    if (!e) return why.fail(MDIM_ERR_INVALID, "null expression");
    if (e->abi_version != MDIM_ABI_VERSION) return why.fail(MDIM_ERR_INVALID, "abi_version %d != %d", e->abi_version, MDIM_ABI_VERSION);
    if (e->rank < 0 || e->red_rank < 0 || e->rank + e->red_rank > MDIM_MAX_RANK) return why.fail(MDIM_ERR_INVALID, "bad rank");
    if (e->n_nodes < 1 || e->n_nodes > MDIM_MAX_NODES || !e->nodes) return why.fail(MDIM_ERR_INVALID, "bad node count");
    const int total = e->rank + e->red_rank;
    int stack[MDIM_MAX_NODES], sp = 0;
    for (int i = 0; i < e->n_nodes; ++i) {
        const mdim_node& n = e->nodes[i];
        if (n.kind < 0 || n.kind >= MDIM_NODE_KIND_COUNT) return why.fail(MDIM_ERR_INVALID, "node %d: bad kind", i);
        if (n.dtype < 0 || n.dtype >= MDIM_DTYPE_COUNT) return why.fail(MDIM_ERR_INVALID, "node %d: bad dtype", i);
        const int k = node_arity(n);
        if (k < 0 || k > sp) return why.fail(MDIM_ERR_INVALID, "node %d: arity %d with %d operands available", i, k, sp);
        if (n.kind == MDIM_NODE_GATHER && (k < 1 || k > 3)) return why.fail(k < 1 ? MDIM_ERR_INVALID : MDIM_ERR_UNSUPPORTED, "node %d: gather with %d components", i, k);
        if (n.kind == MDIM_NODE_TUPLE) {
            if (i != e->n_nodes - 1) return why.fail(MDIM_ERR_INVALID, "node %d: a TUPLE node must be the root", i);
            if (k < 1) return why.fail(MDIM_ERR_INVALID, "node %d: empty tuple", i);
            if (k > MDIM_MAX_OUTS) return why.fail(MDIM_ERR_UNSUPPORTED, "a tuple-typed element with %d scalar leaves (> %d): collect the leaves separately", k, MDIM_MAX_OUTS);
        }
        n_child[i] = k;
        for (int c = 0; c < k; ++c) child[i][c] = stack[sp - k + c];
        sp -= k;
        stack[sp++] = i;
        has_err_source[i] = false;
        for (int c = 0; c < k; ++c) has_err_source[i] = has_err_source[i] || has_err_source[child[i][c]];
        switch (n.kind) {
            case MDIM_NODE_LEAF:
                if (n.n_peers > 1) {
                    if (n.n_peers > MDIM_MAX_PEERS || n.peer_block == 0) return why.fail(MDIM_ERR_INVALID, "node %d: bad peer table", i);
                    for (int p = 0; p < n.n_peers; ++p) if (!n.peer[p]) return why.fail(MDIM_ERR_INVALID, "node %d: null peer %d", i, p);
                } else if (!n.data) return why.fail(MDIM_ERR_INVALID, "node %d: null data", i);
                break;
            case MDIM_NODE_GATHER:
                if (n.n_peers > 1) {
                    if (n.n_peers > MDIM_MAX_PEERS || n.peer_block == 0) return why.fail(MDIM_ERR_INVALID, "node %d: bad peer table", i);
                    for (int p = 0; p < n.n_peers; ++p) if (!n.peer[p]) return why.fail(MDIM_ERR_INVALID, "node %d: null peer %d", i, p);
                } else if (!n.data) return why.fail(MDIM_ERR_INVALID, "node %d: null data", i);
                for (int c = 0; c < k; ++c)
                    if (e->nodes[child[i][c]].dtype != MDIM_U64) return why.fail(MDIM_ERR_INVALID, "node %d: index component %d is not usize (U64)", i, c);
                has_err_source[i] = true;
                break;
            case MDIM_NODE_UNARY: {
                if (n.op < 0 || n.op >= MDIM_UNARY_COUNT) return why.fail(MDIM_ERR_INVALID, "node %d: bad unary op", i);
                const int cd = e->nodes[child[i][0]].dtype;
                if (n.op == MDIM_CAST) { if (n.src_dtype != cd) return why.fail(MDIM_ERR_INVALID, "node %d: cast src_dtype mismatch", i); }
                else {
                    if (cd != n.dtype) return why.fail(MDIM_ERR_INVALID, "node %d: unary dtype mismatch", i);
                    if (n.op == MDIM_NOT && !is_int(n.dtype)) return why.fail(MDIM_ERR_INVALID, "node %d: NOT on a float", i);
                    if (n.op == MDIM_SQRT && !is_float(n.dtype)) return why.fail(MDIM_ERR_INVALID, "node %d: SQRT on an integer", i);
                }
                break;
            }
            case MDIM_NODE_BINARY:
            case MDIM_NODE_FOLD: {
                if (n.op < 0 || n.op >= MDIM_BINARY_COUNT) return why.fail(MDIM_ERR_INVALID, "node %d: bad binary op", i);
                const int l = n.kind == MDIM_NODE_BINARY ? e->nodes[child[i][0]].dtype : n.dtype;
                const int r = e->nodes[child[i][k - 1]].dtype;  // BINARY: the right operand; FOLD: the body (its last child)
                if (l != n.dtype) return why.fail(MDIM_ERR_INVALID, "node %d: lhs dtype mismatch", i);
                if (n.kind == MDIM_NODE_FOLD && k == 2 && e->nodes[child[i][0]].dtype != n.dtype) return why.fail(MDIM_ERR_INVALID, "node %d: fold init dtype mismatch", i);
                if (n.op == MDIM_SHL || n.op == MDIM_SHR) { if (!is_int(l) || !is_int(r)) return why.fail(MDIM_ERR_INVALID, "node %d: shift on a float", i); }
                else if (r != n.dtype) return why.fail(MDIM_ERR_INVALID, "node %d: rhs dtype mismatch", i);
                if (is_float(n.dtype) && n.op >= MDIM_AND) return why.fail(MDIM_ERR_INVALID, "node %d: bit op on a float", i);
                if (is_int(n.dtype) && (n.op == MDIM_DIV || n.op == MDIM_REM)) has_err_source[i] = true;
                if (n.kind == MDIM_NODE_FOLD) {
                    if (fold_node >= 0) return why.fail(MDIM_ERR_UNSUPPORTED, "more than one FOLD in one expression");
                    fold_node = i;
                }
                break;
            }
            case MDIM_NODE_CONCAT:
                if (e->nodes[child[i][0]].dtype != n.dtype || e->nodes[child[i][1]].dtype != n.dtype) return why.fail(MDIM_ERR_INVALID, "node %d: concat dtype mismatch", i);
                if (n.axis_a[0] < 0 || n.axis_a[0] >= total) return why.fail(MDIM_ERR_INVALID, "node %d: bad concat axis", i);
                break;
            case MDIM_NODE_DIAG:
                if (e->nodes[child[i][0]].dtype != n.dtype) return why.fail(MDIM_ERR_INVALID, "node %d: diag dtype mismatch", i);
                if (n.n_comp < 0 || n.n_comp > kMaxRank) return why.fail(MDIM_ERR_INVALID, "node %d: bad pair count", i);
                for (int p = 0; p < n.n_comp; ++p)
                    if (n.axis_a[p] < 0 || n.axis_a[p] >= total || n.axis_b[p] >= total) return why.fail(MDIM_ERR_INVALID, "node %d: bad diag axis", i);
                break;
            default: break;
        }
    }
    if (sp != 1) return why.fail(MDIM_ERR_INVALID, "expression leaves %d values", sp);
    if (e->red_rank > 0 && fold_node < 0) return why.fail(MDIM_ERR_INVALID, "reduction axes without a FOLD node");
    // mark nodes under the fold: post-order => the fold's subtree is a contiguous range ending at it
    for (int i = 0; i < e->n_nodes; ++i) under_fold[i] = false;
    if (fold_node >= 0) {
        std::vector<int> work{child[fold_node][n_child[fold_node] - 1]};  // the body; an init view (first child) lives outside the loop
        while (!work.empty()) {
            int x = work.back(); work.pop_back();
            under_fold[x] = true;
            for (int c = 0; c < n_child[x]; ++c) work.push_back(child[x][c]);
        }
    }
    for (int i = 0; i < e->n_nodes; ++i) {
        const mdim_node& n = e->nodes[i];
        if (n.kind == MDIM_NODE_LEAF || n.kind == MDIM_NODE_IOTA || n.kind == MDIM_NODE_GATHER)
            for (int a = e->rank; a < total; ++a)
                if (n.stride[a] != 0 && !under_fold[i]) return why.fail(MDIM_ERR_INVALID, "node %d: reduction stride outside the FOLD", i);
    }
    return MDIM_OK;
}

// Drop length-1 axes and merge neighbours that every operand walks contiguously.
void Builder::canonical_axes() {
    const int total = e->rank + e->red_rank;
    bool pred_axis[kMaxRank] = {false};
    for (int i = 0; i < e->n_nodes; ++i) {
        const mdim_node& n = e->nodes[i];
        if (n.kind == MDIM_NODE_CONCAT) pred_axis[n.axis_a[0]] = true;
        if (n.kind != MDIM_NODE_DIAG) continue;
        for (int p = 0; p < n.n_comp; ++p) {
            pred_axis[n.axis_a[p]] = true;
            if (n.axis_b[p] >= 0) pred_axis[n.axis_b[p]] = true;
        }
    }
    std::vector<int> addr_nodes;
    for (int i = 0; i < e->n_nodes; ++i) {
        const int k = e->nodes[i].kind;
        if (k == MDIM_NODE_LEAF || k == MDIM_NODE_IOTA || k == MDIM_NODE_GATHER) addr_nodes.push_back(i);
    }
    // groups of original axes; each group becomes one canonical axis
    struct Group { int first, last; uint64_t len; bool red; };
    std::vector<Group> groups;
    for (int a = 0; a < total; ++a) {
        const bool red = a >= e->rank;
        const uint64_t L = e->length[a];
        if (L == 1 && !pred_axis[a]) { axis_map[a] = -1; continue; }
        bool merged = false;
        if (!groups.empty()) {
            Group& g = groups.back();
            // g.last is the previous KEPT axis (dropped length-1 axes in between always have
            // coordinate 0, so they do not break contiguity)
            if (g.red == red && !pred_axis[a] && !pred_axis[g.last]) {
                bool ok = true;
                for (int ni : addr_nodes) {
                    const mdim_node& n = e->nodes[ni];
                    // stride of the group's last axis must equal stride[a] * len[a]
                    if (n.stride[g.last] != n.stride[a] * (int64_t)L) { ok = false; break; }
                }
                if (ok) { g.last = a; g.len *= L; merged = true; }
            }
        }
        if (!merged) groups.push_back(Group{a, a, L, red});
        axis_map[a] = (int)groups.size() - 1;
    }
    n_axes = (int)groups.size();
    rank = 0; red_rank = 0;
    for (int g = 0; g < n_axes; ++g) {
        len[g] = groups[g].len;
        if (groups[g].red) red_rank++; else rank++;
        for (int ni : addr_nodes) cstride[ni][g] = e->nodes[ni].stride[groups[g].last];
    }
    for (int ni : addr_nodes)
        for (int g = n_axes; g < kMaxRank; ++g) cstride[ni][g] = 0;
}

int Builder::push_instr(const Instr& in) {
    Program& P = plan->prog;
    if (P.n_instr >= kMaxInstr) return why.fail(MDIM_ERR_UNSUPPORTED, "expression too long (> %d device instructions)", kMaxInstr);
    P.instr[P.n_instr++] = in;
    depth += in.opc == OPC_LEAF_VEC || in.opc == OPC_LEAF_BCAST || in.opc == OPC_LEAF_STRIDED || in.opc == OPC_IOTA || in.opc == OPC_CONST ||
                     (in.opc == OPC_FOLD_BEGIN && in.aux != 1) ? 1
             : in.opc == OPC_BINARY || in.opc == OPC_FOLD_STEP || in.opc == OPC_SELECT2 ? -1
             : in.opc == OPC_GATHER ? 1 - (int)in.aux
                                    : 0;
    max_depth = std::max(max_depth, depth);
    return MDIM_OK;
}

int Builder::gen(int ni, int mask_first, int mask_n) {
    const mdim_node& n = e->nodes[ni];
    Program& P = plan->prog;
    Instr in;
    memset(&in, 0, sizeof in);
    in.dtype = (uint8_t)n.dtype;
    auto new_addr = [&](int* slot) -> int {
        if (P.n_addr >= kMaxAddr) return why.fail(MDIM_ERR_UNSUPPORTED, "too many array operands (> %d)", kMaxAddr);
        Addr& A = P.addr[P.n_addr];
        memset(&A, 0, sizeof A);
        A.ptr = n.data;
        A.offset = n.offset;
        for (int g = 0; g < n_axes; ++g) A.stride[pa(g)] = cstride[ni][g];
        A.inner = rank > 0 ? A.stride[0] : 0;
        if (red_rank > 0) {  // the fastest reduction axis is walked by a dedicated counter (see exec.cuh: rk)
            A.rstride = cstride[ni][n_axes - 1];
            A.stride[pa(n_axes - 1)] = 0;
        }
        *slot = P.n_addr++;
        return MDIM_OK;
    };
    const int V = P.vec;
    switch (n.kind) {
        case MDIM_NODE_LEAF: {
            int slot; int st = new_addr(&slot); if (st) return st;
            Addr& A = P.addr[slot];
            const int es = dtype_size(n.dtype);
            const bool sharded = n.n_peers > 1;  // the Array's items live in equal blocks on the GPUs of the box
            if (sharded) {
                if (P.peers.block != 0) return why.fail(MDIM_ERR_UNSUPPORTED, "more than one peer-sharded source");
                for (int p = 0; p < n.n_peers; ++p) P.peers.peer[p] = n.peer[p];
                P.peers.block = n.peer_block;
                A.ptr = n.peer[0]; A.n_peers = n.n_peers;
            }
            // every vector must be `align`-byte aligned wherever it lands: base pointer(s), offset, outer strides
            // and, for a sharded Array, the block boundaries (so that no vector straddles two peers)
            auto aligned = [&](int64_t align) {
                bool ok = (((uintptr_t)A.ptr + (uintptr_t)(A.offset * es)) % align) == 0;
                for (int g = 0; g < n_axes && ok; ++g)
                    if (g != rank - 1 && ((cstride[ni][g] * es) % align) != 0) ok = false;
                if (sharded) {
                    ok = ok && ((int64_t)(n.peer_block * (uint64_t)es) % align) == 0 && ((A.offset * es) % align) == 0;
                    for (int p = 0; p < n.n_peers && ok; ++p) ok = ((uintptr_t)n.peer[p] % align) == 0;
                }
                return ok;
            };
            const int64_t s_in = rank > 0 ? cstride[ni][rank - 1] : 0;
            int opc;
            if (rank == 0 || s_in == 0) opc = OPC_LEAF_BCAST;
            else if (s_in == 1) {
                bool ok = aligned(std::min<int64_t>(16, (int64_t)V * es));
                if (sharded && ok) ok = aligned((int64_t)V * es);  // a whole vector inside one block
                opc = ok ? OPC_LEAF_VEC : OPC_LEAF_STRIDED;
                if (ok && !aligned(32)) plan->vec256_ok = 0;  // 256-bit accesses need every vector of this operand 32-byte aligned
            } else opc = OPC_LEAF_STRIDED;
            in.opc = (uint8_t)opc; in.slot = (uint16_t)slot;
            if (opc == OPC_LEAF_VEC)  // re-read along a broadcast output axis => worth keeping in L1
                for (int g = 0; g < rank; ++g) if (cstride[ni][g] == 0 && len[g] > 1) in.aux = 1;
            if (sharded) in.aux |= 2;  // exec.cuh: leaf_base() picks the peer
            return push_instr(in);
        }
        case MDIM_NODE_IOTA: {
            int slot; int st = new_addr(&slot); if (st) return st;
            in.opc = OPC_IOTA; in.slot = (uint16_t)slot;
            return push_instr(in);
        }
        case MDIM_NODE_CONST:
            in.opc = OPC_CONST; in.imm = n.imm.u64;
            if (dtype_size(n.dtype) == 4) in.imm &= 0xffffffffull;
            if (dtype_size(n.dtype) == 1) in.imm &= 0xffull;
            return push_instr(in);
        case MDIM_NODE_UNARY: {
            int st = gen(child[ni][0], mask_first, mask_n); if (st) return st;
            in.opc = OPC_UNARY; in.op = (uint8_t)n.op; in.aux = (uint8_t)e->nodes[child[ni][0]].dtype;
            return push_instr(in);
        }
        case MDIM_NODE_BINARY: {
            int st = gen(child[ni][0], mask_first, mask_n); if (st) return st;
            st = gen(child[ni][1], mask_first, mask_n); if (st) return st;
            in.opc = OPC_BINARY; in.op = (uint8_t)n.op; in.aux = (uint8_t)e->nodes[child[ni][1]].dtype; in.n = (uint16_t)ni;
            return push_instr(in);
        }
        case MDIM_NODE_DIAG: {
            // pred region = enclosing (cumulative) preds followed by this node's own pairs
            if (P.n_pred + mask_n + n.n_comp > kMaxPred) return why.fail(MDIM_ERR_UNSUPPORTED, "too many diagonal predicates");
            const int r0 = P.n_pred;
            for (int p = 0; p < mask_n; ++p) P.pred[P.n_pred++] = P.pred[mask_first + p];
            const int own0 = P.n_pred;
            int own_n = 0;
            for (int p = 0; p < n.n_comp; ++p) {
                Pred pr;
                memset(&pr, 0, sizeof pr);
                const int a = axis_map[n.axis_a[p]];
                const int b = n.axis_b[p] >= 0 ? axis_map[n.axis_b[p]] : -1;
                // the fastest reduction axis is counted by ThreadState::rk (its c[] entry stays 0): its coefficient is rcoef
                auto term = [&](int g, int c) { if (red_rank > 0 && g == n_axes - 1) pr.rcoef += c; else pr.coef[pa(g)] += c; };
                term(a, 1);
                if (b >= 0) { term(b, -1); pr.rhs = (int64_t)n.axis_c[p]; }  // coord[a] == coord[b] + offset
                else if (n.axis_c[p] >= len[a]) { memset(pr.coef, 0, sizeof pr.coef); pr.rcoef = 0; pr.rhs = 1; }  // never on the diagonal
                else pr.rhs = (int64_t)n.axis_c[p];
                pr.lane_coef = rank > 0 ? pr.coef[0] : 0;
                P.pred[P.n_pred++] = pr; own_n++;
            }
            const bool lazy = has_err_source[child[ni][0]];
            if (lazy) {
                Instr m; memset(&m, 0, sizeof m);
                m.opc = OPC_MASK; m.slot = (uint16_t)r0; m.n = (uint16_t)(mask_n + own_n);
                int st = push_instr(m); if (st) return st;
            }
            int st = gen(child[ni][0], r0, mask_n + own_n); if (st) return st;
            in.opc = OPC_SELECT; in.slot = (uint16_t)own0; in.n = (uint16_t)own_n; in.imm = n.imm.u64;
            if (dtype_size(n.dtype) == 4) in.imm &= 0xffffffffull;
            if (dtype_size(n.dtype) == 1) in.imm &= 0xffull;
            st = push_instr(in); if (st) return st;
            if (lazy) {
                Instr m; memset(&m, 0, sizeof m);
                m.opc = OPC_MASK; m.slot = (uint16_t)mask_first; m.n = (uint16_t)mask_n;
                return push_instr(m);
            }
            return MDIM_OK;
        }
        case MDIM_NODE_CONCAT: {
            // Each side is evaluated under a lane mask (enclosing predicates + its own range test): its loads
            // would otherwise run past the end of the other operand.  src/view.rs:938-945.
            if (P.n_pred + 2 * (mask_n + 1) > kMaxPred) return why.fail(MDIM_ERR_UNSUPPORTED, "too many predicates");
            const int caxis = axis_map[n.axis_a[0]];
            const bool on_rk = red_rank > 0 && caxis == n_axes - 1;  // concatenated along the fastest reduction axis
            const int axis = pa(caxis);
            int first[2];
            for (int side = 0; side < 2; ++side) {
                first[side] = P.n_pred;
                for (int p = 0; p < mask_n; ++p) P.pred[P.n_pred++] = P.pred[mask_first + p];
                Pred pr; memset(&pr, 0, sizeof pr);
                if (on_rk) pr.rcoef = 1; else pr.coef[axis] = 1;
                pr.rhs = (int64_t)std::min<uint64_t>(n.axis_c[0], len[axis_map[n.axis_a[0]]]); pr.cmp = side == 0 ? 1 : 2;
                pr.lane_coef = rank > 0 ? pr.coef[0] : 0;
                P.pred[P.n_pred++] = pr;
            }
            for (int side = 0; side < 2; ++side) {
                Instr m; memset(&m, 0, sizeof m);
                m.opc = OPC_MASK; m.slot = (uint16_t)first[side]; m.n = (uint16_t)(mask_n + 1);
                int st = push_instr(m); if (st) return st;
                st = gen(child[ni][side], first[side], mask_n + 1); if (st) return st;
            }
            Instr m; memset(&m, 0, sizeof m);
            m.opc = OPC_MASK; m.slot = (uint16_t)mask_first; m.n = (uint16_t)mask_n;
            int st = push_instr(m); if (st) return st;
            in.opc = OPC_SELECT2; in.slot = (uint16_t)(first[0] + mask_n);
            return push_instr(in);
        }
        case MDIM_NODE_GATHER: {
            for (int c = 0; c < n.n_comp; ++c) { int st = gen(child[ni][c], mask_first, mask_n); if (st) return st; }
            int slot; int st = new_addr(&slot); if (st) return st;
            Addr& A = P.addr[slot];
            for (int c = 0; c < n.n_comp; ++c) { A.gstride[c] = n.gstride[c]; A.bound[c] = n.bound[c]; }
            A.n_peers = n.n_peers > 1 ? n.n_peers : 0;
            if (n.n_peers > 1) {
                if (P.peers.block != 0) return why.fail(MDIM_ERR_UNSUPPORTED, "more than one peer-sharded gather source");
                for (int p = 0; p < n.n_peers; ++p) P.peers.peer[p] = n.peer[p];
                P.peers.block = n.peer_block;
            }
            in.opc = OPC_GATHER; in.slot = (uint16_t)slot; in.aux = (uint8_t)n.n_comp; in.n = (uint16_t)ni;
            return push_instr(in);
        }
        case MDIM_NODE_TUPLE:  // no instruction: the children's values are left on the stack in order, value k is output k
            for (int c = 0; c < n_child[ni]; ++c) { int st = gen(child[ni][c], mask_first, mask_n); if (st) return st; }
            return MDIM_OK;
        case MDIM_NODE_FOLD: {
            const int body = child[ni][n_child[ni] - 1];
            if (n_child[ni] == 2) {  // `let mut s = init.at(i)`: the init value is on the stack when the loop starts
                int st0 = gen(child[ni][0], mask_first, mask_n); if (st0) return st0;
                in.aux = 1;
            }
            in.opc = OPC_FOLD_BEGIN; in.imm = n.imm.u64;
            if (dtype_size(n.dtype) == 4) in.imm &= 0xffffffffull;
            if (dtype_size(n.dtype) == 1) in.imm &= 0xffull;
            int st = push_instr(in); if (st) return st;
            const int begin_pc = P.n_instr - 1;
            const int body_pc = P.n_instr;
            st = gen(body, mask_first, mask_n); if (st) return st;
            Instr s; memset(&s, 0, sizeof s);
            s.opc = OPC_FOLD_STEP; s.dtype = (uint8_t)n.dtype; s.op = (uint8_t)n.op; s.aux = (uint8_t)e->nodes[body].dtype;
            s.slot = (uint16_t)body_pc; s.n = (uint16_t)ni;
            st = push_instr(s); if (st) return st;
            P.instr[begin_pc].slot = (uint16_t)P.n_instr;
            return MDIM_OK;
        }
    }
    return why.fail(MDIM_ERR_INVALID, "node %d: bad kind", ni);
}

// magic numbers for q = umulhi(n, mul) >> shr, exact for n < 2^31 (CUTLASS FastDivmod scheme)
static void find_divisor(uint32_t d, uint32_t* mul, uint32_t* shr) {
    if (d <= 1) { *mul = 0; *shr = 0; return; }
    uint32_t l = 0;
    while ((1ull << l) < d) ++l;  // ceil(log2 d)
    const uint32_t p = 31 + l;
    const uint64_t m = ((1ull << p) + d - 1) / d;
    *mul = (uint32_t)m;
    *shr = p - 32;
}

int Builder::emit() {
    Program& P = plan->prog;
    memset(&P, 0, sizeof P);
    const int root = e->n_nodes - 1;
    P.rank = rank; P.red_rank = red_rank;
    const bool tuple_root = e->nodes[root].kind == MDIM_NODE_TUPLE;
    P.n_out = tuple_root ? n_child[root] : 1;
    for (int k = 0; k < P.n_out; ++k) P.out_dtypes[k] = tuple_root ? e->nodes[child[root][k]].dtype : e->nodes[root].dtype;
    P.out_dtype = P.out_dtypes[0];
    plan->n_out = P.n_out;
    for (int k = 0; k < P.n_out; ++k) plan->out_esizes[k] = dtype_size(P.out_dtypes[k]);
    for (int g = 0; g < n_axes; ++g) P.length[pa(g)] = len[g];
    P.red_fast_len = 1;
    if (red_rank > 0) { P.red_fast_len = len[n_axes - 1]; P.length[pa(n_axes - 1)] = 1; }
    uint64_t out_elems = 1, red_count = 1;
    for (int g = 0; g < rank; ++g) out_elems *= len[g];
    for (int g = rank; g < n_axes; ++g) red_count *= len[g];
    P.red_count = red_count;
    plan->out_elems = out_elems;
    plan->out_esize = dtype_size(P.out_dtype);

    // slot width: 8 if any value in the program is 8 bytes wide
    int slot = 4;
    for (int i = 0; i < e->n_nodes; ++i) {
        if (dtype_size(e->nodes[i].dtype) == 8) slot = 8;
        if (e->nodes[i].kind == MDIM_NODE_UNARY && e->nodes[i].op == MDIM_CAST && dtype_size(e->nodes[i].src_dtype) == 8) slot = 8;
        if (e->nodes[i].kind == MDIM_NODE_IOTA && dtype_size(e->nodes[i].dtype) == 8) slot = 8;
    }
    plan->slot_bytes = slot;
    // vector width along the innermost output axis: the widest of at most 32 bytes that divides it
    int V = 1;
    if (rank > 0) {
        const int cand32[3] = {8, 4, 1}, cand64[3] = {4, 2, 1};
        const int* cand = slot == 4 ? cand32 : cand64;
        for (int i = 0; i < 3; ++i)
            if (len[rank - 1] % (uint64_t)cand[i] == 0) { V = cand[i]; break; }
    }
    // A fold walks its reduction axes sequentially inside one thread, so the output is the only source of
    // parallelism: prefer narrower vectors until there are enough threads to fill the machine.
    if (fold_node >= 0 && rank > 0) {
        const int cand32[3] = {8, 4, 1}, cand64[3] = {4, 2, 1};
        const int* cand = slot == 4 ? cand32 : cand64;
        const uint64_t min_threads = 40000;  // measured: 64 Ki threads x 16 B beat 256 Ki x 4 B and 32 Ki x 32 B
        for (int i = 0; i < 3 && out_elems / (uint64_t)V < min_threads; ++i)
            if (cand[i] < V && len[rank - 1] % (uint64_t)cand[i] == 0) V = cand[i];
    }
    if (force_vec) V = force_vec;
    plan->vec = V; P.vec = V;
    P.n_vec = out_elems / (uint64_t)V;  // work items: one per thread trip

    // 32-bit coordinate path needs: vectors < 2^31, every axis < 2^31, every stride in int32
    bool wide = P.n_vec >= (1ull << 31);
    for (int g = 0; g < n_axes; ++g) if (len[g] >= (1ull << 31)) wide = true;
    for (int i = 0; i < e->n_nodes; ++i) {
        const int k = e->nodes[i].kind;
        if (k == MDIM_NODE_LEAF || k == MDIM_NODE_IOTA || k == MDIM_NODE_GATHER)
            for (int g = 0; g < n_axes; ++g)
                if (cstride[i][g] > INT32_MAX || cstride[i][g] < INT32_MIN) wide = true;
    }
    // ... and every operand's linear offset must fit in int32 for every coordinate
    for (int i = 0; i < e->n_nodes; ++i) {
        const int k = e->nodes[i].kind;
        if (k != MDIM_NODE_LEAF && k != MDIM_NODE_IOTA && k != MDIM_NODE_GATHER) continue;
        double reach = (double)(e->nodes[i].offset < 0 ? -e->nodes[i].offset : e->nodes[i].offset);
        for (int g = 0; g < n_axes; ++g) reach += (double)(len[g] ? len[g] - 1 : 0) * (double)(cstride[i][g] < 0 ? -cstride[i][g] : cstride[i][g]);
        if (reach >= 2147483647.0) wide = true;
    }
    plan->wide = wide ? 1 : 0;
    plan->n_axes = n_axes;
    for (int g = 0; g < kMaxRank; ++g) {
        uint64_t L = 1;
        if (g < rank) L = (g == rank - 1) ? len[g] / (uint64_t)V : len[g];
        const int a = g < n_axes ? pa(g) : g;
        P.dec_len[a] = L;
        P.dec_scale[a] = (g == rank - 1) ? (uint32_t)V : 1u;
        find_divisor((uint32_t)std::min<uint64_t>(L, 0x7fffffffull), &P.div_mul[a], &P.div_shr[a]);
    }
    depth = 0; max_depth = 0;
    plan->vec256_ok = (V * slot == 32) ? 1 : 0;
    int st = gen(root, 0, 0);
    if (st) return st;
    if (depth != P.n_out) return why.fail(MDIM_ERR_INVALID, "internal: program leaves depth %d", depth);
    if (max_depth > kMaxDepth) return why.fail(MDIM_ERR_UNSUPPORTED, "expression needs a value stack of %d (> %d)", max_depth, kMaxDepth);
    plan->max_depth = max_depth;
    // signature bytes
    plan->sig_len = 0;
    for (int i = 0; i < P.n_instr; ++i) {
        plan->sig[plan->sig_len++] = (char)P.instr[i].opc;
        plan->sig[plan->sig_len++] = (char)P.instr[i].dtype;
        plan->sig[plan->sig_len++] = (char)P.instr[i].op;
        plan->sig[plan->sig_len++] = (char)P.instr[i].aux;
    }
    if (P.n_out > 1) {  // several outputs: no pre-built signature may match, and the run-time specialisation is keyed on the count
        plan->sig[plan->sig_len++] = (char)0xFE; plan->sig[plan->sig_len++] = (char)P.n_out;
        plan->sig[plan->sig_len++] = 0; plan->sig[plan->sig_len++] = 0;
    }
    return MDIM_OK;
}

// ---- fast paths -------------------------------------------------------------------------------
int Builder::detect_fast_paths() {
    Program& P = plan->prog;
    const mdim_node* N = e->nodes;
    const int root = e->n_nodes - 1;
    if (N[root].kind == MDIM_NODE_TUPLE) return MDIM_OK;  // several outputs: the evaluator only
    // (1) tiled transpose: a single leaf whose unit-stride axis is not the output's innermost axis
    if (e->n_nodes == 1 && N[0].kind == MDIM_NODE_LEAF && red_rank == 0 && rank >= 2) {
        const int es = dtype_size(N[0].dtype);
        const int64_t* s = cstride[0];
        int axis_a = -1;
        for (int g = 0; g < rank - 1; ++g) if (s[g] == 1) axis_a = g;
        const int axis_b = rank - 1;
        if ((es == 4 || es == 8) && axis_a >= 0 && s[axis_b] != 1 && s[axis_b] != 0 && len[axis_a] >= 16 && len[axis_b] >= 16 && !plan->wide) {
            TransposePlan& T = plan->tr;
            memset(&T, 0, sizeof T);
            T.src = N[0].n_peers > 1 ? N[0].peer[0] : N[0].data; T.esize = es; T.src_offset = N[0].offset;
            if (N[0].n_peers > 1) {
                T.n_peers = N[0].n_peers; T.peer_block = N[0].peer_block; T.peer_inv = 1.0f / (float)N[0].peer_block;
                for (int p = 0; p < N[0].n_peers; ++p) T.peer[p] = N[0].peer[p];
            }
            T.len_a = len[axis_a]; T.len_b = len[axis_b];
            T.src_stride_b = s[axis_b];
            // out strides: row-major over canonical out axes
            int64_t ostride[kMaxRank]; int64_t acc = 1;
            for (int g = rank - 1; g >= 0; --g) { ostride[g] = acc; acc *= (int64_t)len[g]; }
            T.out_stride_a = ostride[axis_a];
            for (int g = 0; g < rank; ++g) {
                if (g == axis_a || g == axis_b) continue;
                T.batch_len[T.n_batch] = len[g];
                T.batch_src_stride[T.n_batch] = s[g];
                T.batch_out_stride[T.n_batch] = ostride[g];
                T.n_batch++;
            }
            const uint64_t tile_a = (uint64_t)kTrTileChunks * 16 / (uint64_t)es;
            T.tiles_a = (T.len_a + tile_a - 1) / tile_a; T.tiles_b = (T.len_b + kTrTileRows - 1) / kTrTileRows;
            uint64_t nb = 1; for (int b = 0; b < T.n_batch; ++b) nb *= T.batch_len[b];
            T.n_tiles = T.tiles_a * T.tiles_b * nb;
            plan->kind = KK_TRANSPOSE;
            snprintf(plan->describe, sizeof plan->describe, "transpose.tile%dx%d%s es%d a=%llu b=%llu batch=%llu", (int)tile_a, kTrTileRows, T.n_peers > 1 ? ".peers" : "", es,
                     (unsigned long long)T.len_a, (unsigned long long)T.len_b, (unsigned long long)nb);
            return MDIM_OK;
        }
    }
    if (detect_fold_split()) return MDIM_OK;
    // (2) last-axis sequential fold of one contiguous f32/f64/int leaf, optionally fused with
    //     `x (eop) (fold [post_op c])` broadcast back over the folded axis (config C4)
    if (fold_node >= 0 && n_child[fold_node] == 1 && red_rank == 1 && rank <= 2 && !plan->wide && !(flags & kPlanScalarOut)) {
        const mdim_node& F = N[fold_node];
        const int fc = child[fold_node][0];
        const uint64_t row_len = len[n_axes - 1];
        const int es = dtype_size(F.dtype);
        auto rows_leaf = [&](int ni, bool with_red, int out_rank_expected) -> bool {
            // contiguous (rows, row_len) leaf: red stride 1 (if with_red) and row stride row_len
            if (N[ni].kind != MDIM_NODE_LEAF || N[ni].dtype != F.dtype || N[ni].n_peers > 1) return false;
            const int64_t* s = cstride[ni];
            (void)out_rank_expected;
            if (with_red && s[n_axes - 1] != 1) return false;
            return true;
        };
        // the row kernel has no error channel: integer DIV/REM (which can panic) stay on the evaluator
        auto row_safe = [&](int op) { return op != MDIM_SHL && op != MDIM_SHR && !(is_int(F.dtype) && (op == MDIM_DIV || op == MDIM_REM)); };
        if (es == 4 && row_len >= 8 && row_len <= (1u << 24) && row_len % 4 == 0 && row_safe(F.op)) {
            FoldRowsPlan& R = plan->fr;
            memset(&R, 0, sizeof R);
            R.row_len = (uint32_t)row_len; R.op = F.op; R.dtype = F.dtype; R.init = F.imm.u64 & 0xffffffffull;
            const bool src_aligned = (((uintptr_t)N[fc].data + (uintptr_t)(N[fc].offset * es)) % 16) == 0;
            // (2a) fold only: out rank 1 (rows), leaf strides (row_len | 1)
            if (root == fold_node && rank == 1 && rows_leaf(fc, true, 1) && cstride[fc][0] == (int64_t)row_len && src_aligned) {
                R.src = N[fc].data; R.src_offset = N[fc].offset; R.n_rows = len[0]; R.epilogue = 0;
                plan->kind = KK_FOLD_ROWS;
                snprintf(plan->describe, sizeof plan->describe, "fold_rows rows=%llu len=%u op=%d", (unsigned long long)R.n_rows, R.row_len, R.op);
                return MDIM_OK;
            }
            // (2b) fused: root = BINARY(eop, LEAF x[r][k], G) with G = FOLD(LEAF x'[r][k']) or
            //      BINARY(post_op, FOLD(..), CONST); out rank 2 = (rows, row_len); x' is the same
            //      buffer addressed (row_len, 0 | 1)
            if (rank == 2 && N[root].kind == MDIM_NODE_BINARY && len[1] == row_len && row_len <= 512) {  // fused: whole rows resident in smem
                const int lx = child[root][0], g = child[root][1];
                int fnode = -1; bool has_post = false; int post_op = 0; uint64_t post_imm = 0;
                if (g == fold_node) fnode = g;
                else if (N[g].kind == MDIM_NODE_BINARY && child[g][0] == fold_node && N[child[g][1]].kind == MDIM_NODE_CONST) {
                    fnode = fold_node; has_post = true; post_op = N[g].op; post_imm = N[child[g][1]].imm.u64 & 0xffffffffull;
                }
                if (fnode >= 0 && N[lx].kind == MDIM_NODE_LEAF && N[lx].dtype == F.dtype && N[fc].kind == MDIM_NODE_LEAF && N[fc].dtype == F.dtype &&
                    N[lx].data == N[fc].data && N[lx].offset == N[fc].offset && cstride[lx][0] == (int64_t)row_len && cstride[lx][1] == 1 &&
                    cstride[lx][2] == 0 && cstride[fc][0] == (int64_t)row_len && cstride[fc][1] == 0 && cstride[fc][2] == 1 && src_aligned &&
                    row_safe(N[root].op) && row_safe(post_op)) {
                    R.src = N[lx].data; R.src_offset = N[lx].offset; R.n_rows = len[0]; R.epilogue = 1; R.eop = N[root].op;
                    R.has_post = has_post; R.post_op = post_op; R.post_imm = post_imm;
                    plan->kind = KK_FOLD_ROWS;
                    snprintf(plan->describe, sizeof plan->describe, "fold_rows.fused rows=%llu len=%u op=%d eop=%d post=%d",
                             (unsigned long long)R.n_rows, R.row_len, R.op, R.eop, has_post ? post_op : -1);
                    return MDIM_OK;
                }
            }
        }
    }
    // (3) sequential fold over an OUTER axis of one leaf, the result contiguous (out stride 1): every output column is an independent
    //     chain down the rows and all addresses are known up front -> a column walk with 256-bit loads (k_fold_cols).  This is the
    //     one-GPU form of the fold over the sharded axis (SURVEY.md 8e) and each rank's partial fold of the all-reduce route.
    if (fold_node >= 0 && root == fold_node && n_child[fold_node] == 1 && red_rank == 1 && (rank == 1 || rank == 2) && !(flags & kPlanScalarOut)) {
        // canonical axes: [batch,] columns, then the folded axis.  rank 2 = a fold over a MIDDLE axis: one column walk per outer coordinate
        const mdim_node& F = N[fold_node];
        const int fc = child[fold_node][0];
        const int es = dtype_size(F.dtype);
        const int ac = rank - 1, ar = n_axes - 1;  // columns axis, folded axis
        const bool op_ok = F.op == MDIM_ADD || F.op == MDIM_SUB || F.op == MDIM_MUL || ((F.op == MDIM_AND || F.op == MDIM_OR || F.op == MDIM_XOR) && is_int(F.dtype));
        if ((es == 4 || es == 8) && F.dtype != MDIM_U8 && op_ok && N[fc].kind == MDIM_NODE_LEAF && N[fc].dtype == F.dtype && N[fc].n_peers <= 1 && cstride[fc][ac] == 1 &&
            cstride[fc][ar] >= (int64_t)len[ac] && len[ar] >= 1 && (rank == 1 || cstride[fc][0] > 0)) {
            const uint64_t row_bytes = len[ac] * (uint64_t)es, pitch = (uint64_t)cstride[fc][ar] * (uint64_t)es;
            const uint64_t batch_pitch = rank == 2 ? (uint64_t)cstride[fc][0] * (uint64_t)es : 0;
            const uintptr_t base = (uintptr_t)N[fc].data + (uintptr_t)(N[fc].offset * es);
            if (row_bytes % 16 == 0 && pitch % 16 == 0 && batch_pitch % 16 == 0 && base % 16 == 0) {
                FoldColsPlan& C = plan->fc;
                memset(&C, 0, sizeof C);
                C.src = (const void*)base; C.n_rows = len[ar]; C.row_bytes = row_bytes; C.pitch_bytes = pitch;
                C.n_batch = rank == 2 ? len[0] : 1; C.batch_pitch_bytes = batch_pitch;
                C.op = F.op; C.dtype = F.dtype; C.init = es == 4 ? (F.imm.u64 & 0xffffffffull) : F.imm.u64;
                plan->kind = KK_FOLD_COLS;
                snprintf(plan->describe, sizeof plan->describe, "fold_cols batch=%llu rows=%llu cols=%llu es%d op=%d", (unsigned long long)C.n_batch, (unsigned long long)C.n_rows,
                         (unsigned long long)len[ac], es, C.op);
                return MDIM_OK;
            }
        }
    }
    (void)P;
    return MDIM_OK;
}

// (0) an integer fold with few outputs and a long reduction, its body one leaf or one integer cast of one leaf: k_fold_split cuts
//     the reduction into chunks spread over the whole GPU and combines the chunks' partials.  Every other route parallelises over
//     the outputs only, so one thread (or a few lanes) would walk each output's reduction.
bool Builder::detect_fold_split() {
    const mdim_node* N = e->nodes;
    const int root = e->n_nodes - 1;
    if (fold_node != root || n_child[fold_node] != 1 || red_rank < 1) return false;  // an init view keeps its route
    const mdim_node& F = N[fold_node];
    const bool op_ok = F.op == MDIM_ADD || F.op == MDIM_SUB || F.op == MDIM_MUL || F.op == MDIM_AND || F.op == MDIM_OR || F.op == MDIM_XOR;
    if (!op_ok || !is_int(F.dtype)) return false;
    int lf = child[fold_node][0];
    if (N[lf].kind == MDIM_NODE_UNARY && N[lf].op == MDIM_CAST && is_int(N[lf].src_dtype) && N[lf].dtype == F.dtype) lf = child[lf][0];
    else if (N[lf].dtype != F.dtype) return false;
    if (N[lf].kind != MDIM_NODE_LEAF || N[lf].n_peers > 1 || !is_int(N[lf].dtype)) return false;
    uint64_t n_out = 1, red = 1;
    for (int g = 0; g < rank; ++g) n_out *= len[g];
    for (int g = rank; g < n_axes; ++g) red *= len[g];
    if (n_out > kSplitMaxOuts || red < kSplitMinRed) return false;
    // The operators above are associative and commutative (Sub: init - sum), so the reduction may be walked in any order: sort
    // its axes by |stride|, flip the negative ones and merge again.  A whole transposed or reversed array then reads memory in
    // order.  No other route may do this: a float fold, or Div, must combine in index order.
    const int64_t* s = cstride[lf];
    int64_t offset = N[lf].offset;
    struct Ax { uint64_t len; int64_t stride; };
    std::vector<Ax> ra;
    for (int g = rank; g < n_axes; ++g) {
        int64_t st = s[g];
        if (st < 0) { offset += st * (int64_t)(len[g] - 1); st = -st; }
        ra.push_back(Ax{len[g], st});
    }
    std::stable_sort(ra.begin(), ra.end(), [](const Ax& a, const Ax& b) { return a.stride < b.stride; });
    std::vector<Ax> merged{ra[0]};
    for (size_t k = 1; k < ra.size(); ++k) {
        Ax& in = merged.back();
        if (ra[k].stride == in.stride * (int64_t)in.len) in.len *= ra[k].len;
        else merged.push_back(ra[k]);
    }
    if (merged.size() != 1) return false;
    const int64_t rstride = merged[0].stride;
    FoldSplitPlan& S = plan->fs;
    memset(&S, 0, sizeof S);
    const int src_es = dtype_size(N[lf].dtype);
    S.src = (const char*)N[lf].data + offset * src_es;
    S.op = F.op; S.dtype = F.dtype; S.src_dtype = N[lf].dtype;
    S.slot_bytes = dtype_size(F.dtype) == 8 ? 8 : 4;
    S.init = F.imm.u64;
    S.red = red; S.n_out = n_out;
    if (rstride == 1 && rank <= 2) {  // runs: a whole reduction, or a few rows of contiguous elements, output strides free
        S.layout = SPLIT_RUNS;
        S.out_len[0] = S.out_len[1] = 1;
        for (int g = 0; g < rank; ++g) { S.out_len[2 - rank + g] = len[g]; S.out_stride[2 - rank + g] = s[g]; }
    } else if ((rank == 1 || rank == 2) && s[rank - 1] == 1 && rstride >= (int64_t)len[rank - 1] && n_out <= kSplitMaxCols) {  // columns: the k_fold_cols layout
        S.layout = SPLIT_COLS;
        S.cols = len[rank - 1]; S.pitch = rstride;
        S.n_batch = rank == 2 ? len[0] : 1; S.batch_stride = rank == 2 ? s[0] : 0;
    } else return false;
    static const char* const dt_name[] = {"u8", "i32", "u32", "i64", "u64"};
    plan->kind = KK_FOLD_SPLIT;
    snprintf(plan->describe, sizeof plan->describe, "fold_split.%s outs=%llu red=%llu slot=s%d src=%s op=%d", S.layout == SPLIT_RUNS ? "runs" : "cols",
             (unsigned long long)n_out, (unsigned long long)red, S.slot_bytes * 8, dt_name[S.src_dtype], S.op);
    return true;
}

}  // namespace

// Byte ranges the expression reads, from the descriptor alone: offset + sum over axes of stride * [0, length) (+ the
// gathered components over [0, bound)).  Conservative by construction (a hull per operand).
static void input_ranges(const mdim_expr* e, Plan* plan) {
    plan->n_in_ranges = 0;
    auto push = [&](uint64_t lo, uint64_t hi) {
        if (plan->n_in_ranges < 0) return;
        if (plan->n_in_ranges == kMaxRanges) { plan->n_in_ranges = -1; return; }
        plan->in_range[plan->n_in_ranges++] = MemRange{lo, hi};
    };
    const int n_axes = e->rank + e->red_rank;
    for (int i = 0; i < e->n_nodes; ++i) {
        const mdim_node& n = e->nodes[i];
        if (n.kind != MDIM_NODE_LEAF && n.kind != MDIM_NODE_GATHER) continue;
        const uint64_t es = (uint64_t)dtype_size(n.dtype);
        if (n.n_peers > 1) {
            for (int p = 0; p < n.n_peers; ++p) push((uint64_t)(uintptr_t)n.peer[p], (uint64_t)(uintptr_t)n.peer[p] + n.peer_block * es);
            continue;
        }
        int64_t lo = n.offset, hi = n.offset;
        for (int a = 0; a < n_axes; ++a) {
            if (e->length[a] == 0) continue;
            const int64_t ext = n.stride[a] * (int64_t)(e->length[a] - 1);
            if (ext > 0) hi += ext; else lo += ext;
        }
        if (n.kind == MDIM_NODE_GATHER)
            for (int c = 0; c < n.n_comp; ++c) {
                if (n.bound[c] == 0) continue;
                const int64_t ext = n.gstride[c] * (int64_t)(n.bound[c] - 1);
                if (ext > 0) hi += ext; else lo += ext;
            }
        push((uint64_t)((int64_t)(uintptr_t)n.data + lo * (int64_t)es), (uint64_t)((int64_t)(uintptr_t)n.data + (hi + 1) * (int64_t)es));
    }
}

int plan_expr(const mdim_expr* e, uint32_t flags, Plan* plan, char* why_buf, size_t why_len) {
    Builder* b = new Builder();
    b->e = e; b->flags = flags; b->plan = plan; b->why = Why{why_buf, why_len};
    if (why_buf && why_len) why_buf[0] = 0;
    memset(plan, 0, sizeof *plan);
    plan->static_id = -1;
    plan->flags = flags;
    int st = b->validate();
    if (st) { delete b; return st; }
    // zero-length output: Array::new_view pushes nothing (src/array.rs:106-113)
    bool empty = false;
    for (int a = 0; a < e->rank; ++a) if (e->length[a] == 0) empty = true;
    if (empty) {
        plan->kind = KK_EMPTY; plan->out_elems = 0; plan->out_esize = dtype_size(e->nodes[e->n_nodes - 1].dtype);
        snprintf(plan->describe, sizeof plan->describe, "empty");
        delete b; return MDIM_OK;
    }
    input_ranges(e, plan);
    bool gather_big = false;
    for (int i = 0; i < e->n_nodes; ++i) {
        const mdim_node& n = e->nodes[i];
        if (n.kind != MDIM_NODE_GATHER || n.n_peers > 1) continue;
        uint64_t span = 1;
        for (int c = 0; c < n.n_comp; ++c) span += (uint64_t)(n.gstride[c] < 0 ? -n.gstride[c] : n.gstride[c]) * (n.bound[c] ? n.bound[c] - 1 : 0);
        if (span * (uint64_t)dtype_size(n.dtype) > kGatherBigBytes) gather_big = true;
    }
    if (flags & kPlanScalarOut) b->force_vec = 1;
    b->canonical_axes();
    st = b->emit();
    if (st) { delete b; return st; }
    if (plan->max_depth > 4 && plan->vec > 1) {  // deep value stacks only exist scalar (register budget)
        b->force_vec = 1;
        st = b->emit();
        if (st) { delete b; return st; }
    }
    plan->kind = (b->rank <= 1 && b->red_rank == 0) ? KK_STREAM : KK_GENERIC;
    const int need_maxr = plan->kind == KK_STREAM ? 1 : std::max(1, plan->n_axes);
    if (!(flags & MDIM_COLLECT_NO_STATIC))
        plan->static_id = find_static_signature(plan->sig, plan->sig_len, plan->slot_bytes, plan->vec, need_maxr, plan->wide);
    snprintf(plan->describe, sizeof plan->describe, "%s.%s s%d v%dx1%s rank=%d+%d depth=%d instr=%d",
             plan->kind == KK_STREAM ? "stream" : "generic", plan->static_id >= 0 ? "static" : "interp", plan->slot_bytes * 8, plan->vec,
             plan->wide ? " wide" : "", b->rank, b->red_rank, plan->max_depth, plan->prog.n_instr);
    if (!(flags & MDIM_COLLECT_NO_FASTPATH)) {
        st = b->detect_fast_paths();
        if (st) { delete b; return st; }
    }
    if (gather_big) plan->prog.flags |= PF_GATHER_BIG;
    delete b;
    return MDIM_OK;
}

}  // namespace mdim
