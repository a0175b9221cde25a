// view.hpp — C++17 host-side mirror of the reference's View / Array / Index API over the C ABI of
// include/mdim.h.  Header-only; typed like the Rust: index and element types are compile-time, so
// `a.transpose<Unit, usize, usize, Unit>()` fails to COMPILE when the Isomorphic bound of
// src/view.rs:586-592 does not hold, exactly as rustc would reject it.  Sizes and data are run-time.
//
// The reference is compiled code (Rust) and no Rust toolchain exists in the build image, so this is
// the host side "in the reference's kind of language"; multidimension_b200/view.py is the same
// lowering in Python (used by the test-suite and the bench).  Lowering rules: DESIGN.md §2.
//
//   reference                                    here
//   Array<(usize,usize), f32>                    Array<std::tuple<usize,usize>, float>
//   a.transpose::<(),usize,usize,()>()           a.transpose<Unit, usize, usize, Unit>()
//   a.zip(b).map(|(x,y)| x*y+1.0)                (a * b + Scalar<float>(1.0f))        (closures are not lowerable)
//   idx.compose(src)                             idx.compose(src)
//   a.rows::<I,J>().map(|r| fold r.each(..))     a.rows<I, J>().fold<Add>(init)       (sequential, index order)
//   v.collect::<Array<I,T>>()                    v.collect(executor)
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <tuple>
#include <type_traits>
#include <utility>
#include <vector>

#include "../mdim.h"

namespace mdim {

// ---- errors: every reference panic surfaces as Panic with the reference's message text ---------------
struct Panic : std::runtime_error {
    int status;
    mdim_error_info info;
    Panic(int st, const std::string& msg) : std::runtime_error(msg), status(st) { std::memset(&info, 0, sizeof info); info.status = st; }
    Panic(int st, const mdim_error_info& i) : std::runtime_error(i.message), status(st), info(i) {}
};
struct Unsupported : std::runtime_error { using std::runtime_error::runtime_error; };

// ---- index types (src/index.rs, src/int.rs): usize, bool, Unit = (), Fixed<N>, Reversed, Option<I>, std::tuple<I...> ------
using usize = uint64_t;
using Unit = std::tuple<>;
template <size_t N> struct Fixed { uint64_t v; };
struct Reversed { uint64_t v; };                       // src/int.rs:58-86: counts backwards, position = size - 1 - v
template <class I> struct Option { bool some; I value; };  // src/index.rs:244-276: None is position 0, Some(i) is 1 + i.to_usize()
template <class I> Option<I> None() { return Option<I>{false, I{}}; }
template <class I> Option<I> Some(const I& i) { return Option<I>{true, i}; }

template <class I> struct Ix;  // Size type, flattened leaf-type list, position-axis lengths
template <> struct Ix<usize> {
    using Size = uint64_t; using Flat = std::tuple<usize>;
    static void lengths(const Size& s, std::vector<uint64_t>& out) { out.push_back(s); }
    static void flat_size(const Size& s, std::vector<uint64_t>& out) { out.push_back(s); }
    static Size build(const uint64_t*& it) { return *it++; }
    static void positions(const usize& i, const Size& s, std::vector<uint64_t>& out) {
        if (!(i < s)) throw Panic(MDIM_ERR_OOB, "Index " + std::to_string(i) + " is out of bounds for size " + std::to_string(s));  // src/int.rs:17
        out.push_back(i);
    }
};
template <> struct Ix<bool> {  // StaticIndex, src/index.rs:236-240
    using Size = Unit; using Flat = std::tuple<bool>;
    static void lengths(const Size&, std::vector<uint64_t>& out) { out.push_back(2); }
    static void flat_size(const Size&, std::vector<uint64_t>&) {}
    static Size build(const uint64_t*&) { return {}; }
    static void positions(const bool& i, const Size&, std::vector<uint64_t>& out) { out.push_back(i ? 1 : 0); }
};
template <size_t N> struct Ix<Fixed<N>> {  // src/int.rs:33-54
    using Size = Unit; using Flat = std::tuple<Fixed<N>>;
    static void lengths(const Size&, std::vector<uint64_t>& out) { out.push_back(N); }
    static void flat_size(const Size&, std::vector<uint64_t>&) {}
    static Size build(const uint64_t*&) { return {}; }
    static void positions(const Fixed<N>& i, const Size&, std::vector<uint64_t>& out) {
        // Fixed::to_usize is unchecked (src/int.rs:44); the slice access items[to_usize] is what panics (src/array.rs:86)
        if (!(i.v < N)) throw Panic(MDIM_ERR_OOB, "Index " + std::to_string(i.v) + " is out of bounds for size " + std::to_string(N));
        out.push_back(i.v);
    }
};
template <> struct Ix<Reversed> {  // src/int.rs:58-86
    using Size = uint64_t; using Flat = std::tuple<Reversed>;
    static void lengths(const Size& s, std::vector<uint64_t>& out) { out.push_back(s); }
    static void flat_size(const Size& s, std::vector<uint64_t>& out) { out.push_back(s); }
    static Size build(const uint64_t*& it) { return *it++; }
    static void positions(const Reversed& i, const Size& s, std::vector<uint64_t>& out) {
        if (!(i.v < s)) throw Panic(MDIM_ERR_OOB, "Index " + std::to_string(i.v) + " is out of bounds for size " + std::to_string(s));
        out.push_back(s - 1 - i.v);
    }
};
template <class... Is> struct Ix<std::tuple<Is...>> {  // src/index.rs:75-154; arity <= 3 (src/tuple.rs:92-145)
    static_assert(sizeof...(Is) <= 3, "tuple index types have arity <= 3 in the reference");
    using Size = std::tuple<typename Ix<Is>::Size...>;
    using Flat = decltype(std::tuple_cat(std::declval<typename Ix<Is>::Flat>()...));
    static void lengths(const Size& s, std::vector<uint64_t>& out) { each(s, out, std::index_sequence_for<Is...>{}, 0); }
    static void flat_size(const Size& s, std::vector<uint64_t>& out) { each(s, out, std::index_sequence_for<Is...>{}, 1); }
    static Size build(const uint64_t*& it) { return Size{Ix<Is>::build(it)...}; }  // braced init: left to right
    static void positions(const std::tuple<Is...>& i, const Size& s, std::vector<uint64_t>& out) { pos(i, s, out, std::index_sequence_for<Is...>{}); }
  private:
    template <size_t... K> static void each(const Size& s, std::vector<uint64_t>& out, std::index_sequence<K...>, int what) {
        (void)s; (void)out; (void)what;
        ((what ? Ix<Is>::flat_size(std::get<K>(s), out) : Ix<Is>::lengths(std::get<K>(s), out)), ...);
    }
    template <size_t... K> static void pos(const std::tuple<Is...>& i, const Size& s, std::vector<uint64_t>& out, std::index_sequence<K...>) {
        (void)i; (void)s; (void)out;
        (Ix<Is>::positions(std::get<K>(i), std::get<K>(s), out), ...);
    }
};
template <class I> struct Ix<Option<I>> {  // one position axis: [None, Some(0), Some(1), ...] (src/index.rs:248)
    using Size = typename Ix<I>::Size; using Flat = std::tuple<Option<I>>;
    static uint64_t inner_length(const Size& s) { std::vector<uint64_t> l; Ix<I>::lengths(s, l); uint64_t n = 1; for (uint64_t x : l) n *= x; return n; }
    static void lengths(const Size& s, std::vector<uint64_t>& out) { out.push_back(1 + inner_length(s)); }
    static void flat_size(const Size& s, std::vector<uint64_t>& out) { Ix<I>::flat_size(s, out); }
    static Size build(const uint64_t*& it) { return Ix<I>::build(it); }
    static void positions(const Option<I>& i, const Size& s, std::vector<uint64_t>& out) {
        if (!i.some) { out.push_back(0); return; }
        std::vector<uint64_t> p, l; Ix<I>::positions(i.value, s, p); Ix<I>::lengths(s, l);
        uint64_t k = 0; for (size_t a = 0; a < p.size(); ++a) k = k * l[a] + p[a];
        out.push_back(1 + k);
    }
};
template <class I> using SizeOf = typename Ix<I>::Size;
template <class I> constexpr size_t n_leaves = std::tuple_size_v<typename Ix<I>::Flat>;
// Isomorphic (src/tuple.rs:166-176): same flattened leaf list
template <class A, class B> constexpr bool isomorphic = std::is_same_v<typename Ix<A>::Flat, typename Ix<B>::Flat>;
template <class From, class To> SizeOf<To> to_iso_size(const SizeOf<From>& s) {
    static_assert(isomorphic<From, To>, "index types are not Isomorphic");
    std::vector<uint64_t> flat; Ix<From>::flat_size(s, flat); flat.push_back(0);
    const uint64_t* it = flat.data();
    return Ix<To>::build(it);
}
template <class I> uint64_t length(const SizeOf<I>& s) {  // Index::length
    std::vector<uint64_t> l; Ix<I>::lengths(s, l);
    uint64_t n = 1; for (uint64_t x : l) n *= x; return n;
}

// ---- element types --------------------------------------------------------------------------------------
template <class T> struct DType;
template <> struct DType<float> { static constexpr int v = MDIM_F32; };
template <> struct DType<double> { static constexpr int v = MDIM_F64; };
template <> struct DType<int32_t> { static constexpr int v = MDIM_I32; };
template <> struct DType<uint32_t> { static constexpr int v = MDIM_U32; };
template <> struct DType<int64_t> { static constexpr int v = MDIM_I64; };
template <> struct DType<uint64_t> { static constexpr int v = MDIM_U64; };
template <> struct DType<uint8_t> { static constexpr int v = MDIM_U8; };
template <> struct DType<int8_t> { static constexpr int v = MDIM_I8; };
template <> struct DType<int16_t> { static constexpr int v = MDIM_I16; };
template <> struct DType<uint16_t> { static constexpr int v = MDIM_U16; };
template <> struct DType<bool> { static constexpr int v = MDIM_U8; };
template <class T> mdim_scalar scalar_of(T x) { mdim_scalar s; s.u64 = 0; std::memcpy(&s, &x, sizeof(T)); return s; }

// ---- the operator vocabulary (src/ops.rs:23-129) ----------------------------------------------------------
struct Add { static constexpr int code = MDIM_ADD; };   struct Sub { static constexpr int code = MDIM_SUB; };
struct Mul { static constexpr int code = MDIM_MUL; };   struct Div { static constexpr int code = MDIM_DIV; };
struct Rem { static constexpr int code = MDIM_REM; };   struct BitAnd { static constexpr int code = MDIM_AND; };
struct BitOr { static constexpr int code = MDIM_OR; };  struct BitXor { static constexpr int code = MDIM_XOR; };
struct Shl { static constexpr int code = MDIM_SHL; };   struct Shr { static constexpr int code = MDIM_SHR; };
struct Neg { static constexpr int code = MDIM_NEG; };   struct Not { static constexpr int code = MDIM_NOT; };
struct Abs { static constexpr int code = MDIM_ABS; };   struct Sqrt { static constexpr int code = MDIM_SQRT; };

// ---- lowered form: named position axes + scalar node trees (DESIGN.md §2) ---------------------------------
struct Axis { uint64_t length; };
using AxisP = std::shared_ptr<Axis>;
struct Node;
using NodeP = std::shared_ptr<const Node>;
struct Node {
    int kind = 0, dtype = 0, op = 0, src_dtype = 0;
    std::vector<NodeP> kids;
    const void* data = nullptr;
    std::shared_ptr<void> keep;
    int64_t offset = 0;
    std::vector<std::pair<AxisP, int64_t>> stride;
    std::vector<int64_t> gstride;
    std::vector<uint64_t> bound;
    struct Pair { AxisP a, b; uint64_t c; int64_t off = 0; };  // coord[a] == coord[b] + off, or == c when !b
    std::vector<Pair> pairs;
    mdim_scalar imm{};
    std::vector<AxisP> red_axes;
    std::vector<const void*> peers;  // LEAF / GATHER: the Array is cut into equal blocks of peer_block elements, block p at peers[p]
    uint64_t peer_block = 0;         // (the other GPUs' HBM, mapped with mdim_peer_table; read over NVLink inside the kernel)
};
using Groups = std::vector<std::vector<AxisP>>;
struct Sub_ { int64_t constant = 0; std::vector<std::pair<AxisP, int64_t>> terms; };
using Table = std::vector<std::pair<const Axis*, Sub_>>;
inline const Sub_* lookup(const Table& t, const AxisP& a) { for (auto& e : t) if (e.first == a.get()) return &e.second; return nullptr; }

inline NodeP substitute(const NodeP& n, const Table& t) {
    if (t.empty()) return n;
    auto out = std::make_shared<Node>(*n);
    for (auto& k : out->kids) k = substitute(k, t);
    if (n->kind == MDIM_NODE_LEAF || n->kind == MDIM_NODE_IOTA || n->kind == MDIM_NODE_GATHER) {
        std::vector<std::pair<AxisP, int64_t>> st;
        auto add = [&](const AxisP& a, int64_t s) { for (auto& e : st) if (e.first == a) { e.second += s; return; } st.push_back({a, s}); };
        for (auto& [a, s] : n->stride) {
            if (const Sub_* sub = lookup(t, a)) { out->offset += s * sub->constant; for (auto& [b, c] : sub->terms) add(b, s * c); }
            else add(a, s);
        }
        out->stride.clear();
        for (auto& e : st) if (e.second != 0) out->stride.push_back(e);
    } else if (n->kind == MDIM_NODE_DIAG) {
        // each side is (axis | none, constant): coord[a] + ca == coord[b] + cb   (lowering.py::substitute)
        auto side = [&](const AxisP& x, int64_t c, AxisP& ox, int64_t& oc) {
            ox = x; oc = c;
            if (!x) return;
            if (const Sub_* sub = lookup(t, x)) {
                if (sub->terms.empty()) { ox = nullptr; oc = c + sub->constant; }
                else if (sub->terms.size() == 1 && sub->terms[0].second == 1) { ox = sub->terms[0].first; oc = c + sub->constant; }
                else throw Unsupported("a Diagonal whose axis has been split or merged needs device div/mod");
            }
        };
        std::vector<Node::Pair> ps; bool dead = false;
        for (auto& p : n->pairs) {
            AxisP a, b; int64_t ca = 0, cb = 0;
            side(p.a, 0, a, ca);
            side(p.b, p.b ? p.off : (int64_t)p.c, b, cb);
            if (!a && !b) { if (ca != cb) dead = true; continue; }
            if (!a) { std::swap(a, b); std::swap(ca, cb); }  // constant == coord[b] + cb  ->  coord[b] == constant - cb
            if (!b) { const int64_t k = cb - ca; if (k < 0) { dead = true; continue; } ps.push_back({a, nullptr, (uint64_t)k, 0}); }
            else ps.push_back({a, b, 0, cb - ca});
        }
        if (dead) { auto c = std::make_shared<Node>(); c->kind = MDIM_NODE_CONST; c->dtype = n->dtype; c->imm = n->imm; return c; }
        if (ps.empty()) return out->kids[0];
        out->pairs = ps;
    } else if (n->kind == MDIM_NODE_CONCAT) {  // pairs[0] = {concatenated axis, -, length of V along it}
        if (const Sub_* sub = lookup(t, n->pairs[0].a)) {
            const int64_t thr = (int64_t)n->pairs[0].c;
            if (sub->terms.empty()) return sub->constant < thr ? out->kids[0] : out->kids[1];  // pinned (row/column): one side survives
            if (sub->terms.size() == 1 && sub->terms[0].second == 1)  // k = k' + c:  k < thr  <=>  k' < thr - c
                out->pairs[0] = {sub->terms[0].first, nullptr, (uint64_t)std::max<int64_t>(thr - sub->constant, 0), 0};
            else throw Unsupported("a Concat whose axis has been split needs device div/mod");
        }
    } else if (n->kind == MDIM_NODE_FOLD) {
        for (auto& a : n->red_axes) if (lookup(t, a)) throw Unsupported("substitution of a reduction axis");
    }
    return out;
}
inline Sub_ rename_to(const AxisP& b) { Sub_ s; s.terms.push_back({b, 1}); return s; }
// Row-major combination of the pieces an axis has been cut into (outermost first); unit pieces carry no term.
inline Sub_ sub_of(const std::vector<AxisP>& pieces) {
    Sub_ s; int64_t acc = 1;
    for (auto it = pieces.rbegin(); it != pieces.rend(); ++it) { if ((*it)->length != 1) s.terms.push_back({*it, acc}); acc *= (int64_t)(*it)->length; }
    return s;
}
// Common refinement of two row-major factorisations of the same run of positions (multidimension_b200/view.py::_refine):
// an axis merged by to_usize out of (2, 3) against a plain axis of 6, or (2, 6) against (4, 3).
inline void refine(const std::vector<uint64_t>& a, const std::vector<uint64_t>& b, std::vector<uint64_t>& pieces, std::vector<std::vector<size_t>>& ma,
                   std::vector<std::vector<size_t>>& mb) {
    for (uint64_t x : a) if (x == 0) throw Unsupported("re-splitting an empty axis");
    for (uint64_t x : b) if (x == 0) throw Unsupported("re-splitting an empty axis");
    pieces.clear(); ma.assign(a.size(), {}); mb.assign(b.size(), {});
    size_t i = 0, j = 0; uint64_t ra = 0, rb = 0;  // 0 = not loaded
    for (;;) {
        while (!ra && i < a.size()) { if (a[i] == 1) { ma[i].push_back(pieces.size()); pieces.push_back(1); ++i; } else ra = a[i]; }
        while (!rb && j < b.size()) { if (b[j] == 1) { mb[j].push_back(pieces.size()); pieces.push_back(1); ++j; } else rb = b[j]; }
        if (!ra || !rb) break;
        uint64_t step;
        if (ra % rb == 0) step = rb; else if (rb % ra == 0) step = ra;
        else throw Unsupported("axis groups have no common refinement: this remapping needs div/mod on the device");
        ma[i].push_back(pieces.size()); mb[j].push_back(pieces.size()); pieces.push_back(step);
        ra /= step; rb /= step;
        if (ra == 1) { ++i; ra = 0; }
        if (rb == 1) { ++j; rb = 0; }
    }
    if (ra || rb) throw Unsupported("axis groups do not describe the same run of positions");
}
// One leaf axis seen by both operands of a binary / concat as the groups a (self) and b (other): -> the group of the result.
inline std::vector<AxisP> unify_group(const std::vector<AxisP>& a, const std::vector<AxisP>& b, Table& tv, Table& tw) {
    std::vector<uint64_t> la, lb;
    for (auto& x : a) la.push_back(x->length);
    for (auto& y : b) lb.push_back(y->length);
    if (la == lb) { for (size_t k = 0; k < a.size(); ++k) tw.push_back({b[k].get(), rename_to(a[k])}); return a; }
    std::vector<uint64_t> pieces; std::vector<std::vector<size_t>> ma, mb;
    refine(la, lb, pieces, ma, mb);
    std::vector<AxisP> axes;
    for (uint64_t n : pieces) axes.push_back(std::make_shared<Axis>(Axis{n}));
    auto pick = [&](const std::vector<size_t>& idx) { std::vector<AxisP> o; for (size_t k : idx) o.push_back(axes[k]); return o; };
    for (size_t k = 0; k < a.size(); ++k) tv.push_back({a[k].get(), sub_of(pick(ma[k]))});
    for (size_t k = 0; k < b.size(); ++k) tw.push_back({b[k].get(), sub_of(pick(mb[k]))});
    return axes;
}
inline Sub_ pin_at(uint64_t c) { Sub_ s; s.constant = (int64_t)c; return s; }
inline std::vector<AxisP> flat(const Groups& g) { std::vector<AxisP> o; for (auto& x : g) o.insert(o.end(), x.begin(), x.end()); return o; }
template <class I> Groups fresh_groups(const SizeOf<I>& s) {
    std::vector<uint64_t> l; Ix<I>::lengths(s, l);
    Groups g; for (uint64_t n : l) g.push_back({std::make_shared<Axis>(Axis{n})});
    return g;
}

// ---- executors: where collect() runs -----------------------------------------------------------------------
// A function of the same shape as mdim_collect_host / the CPU oracle: operands and result in HOST memory.
using HostCollectFn = std::function<int(const mdim_expr*, void* out_host, mdim_error_info* err)>;
struct Executor {
    HostCollectFn run;
    // The product path: mdim_collect_host on a context (sm_100a kernels; uploads/downloads inside).
    static Executor device(mdim_ctx* ctx, int (*collect_host)(mdim_ctx*, const mdim_expr*, void*, uint32_t), int (*last_error)(mdim_ctx*, mdim_error_info*)) {
        return Executor{[=](const mdim_expr* e, void* out, mdim_error_info* err) {
            const int st = collect_host(ctx, e, out, 0);
            if (st != MDIM_OK && err) last_error(ctx, err);
            return st;
        }};
    }
};

inline void emit_and_run(const NodeP& root, const std::vector<AxisP>& axes, const Executor& ex, void* out_host) {
    std::vector<const Node*> order; std::vector<AxisP> red;
    std::function<void(const NodeP&)> visit = [&](const NodeP& n) {
        for (auto& k : n->kids) visit(k);
        if (n->kind == MDIM_NODE_FOLD) { if (!red.empty()) throw Unsupported("more than one fold in one expression"); red = n->red_axes; }
        order.push_back(n.get());
    };
    visit(root);
    if (order.size() > MDIM_MAX_NODES) throw Unsupported("expression has too many nodes");
    std::vector<AxisP> all = axes; all.insert(all.end(), red.begin(), red.end());
    if (all.size() > MDIM_MAX_RANK) throw Unsupported("expression has too many position axes");
    auto pos = [&](const AxisP& a) { for (size_t i = 0; i < all.size(); ++i) if (all[i] == a) return (int)i; throw Unsupported("internal: stride over an axis that is not iterated"); };
    std::vector<mdim_node> nodes(order.size());
    for (size_t i = 0; i < order.size(); ++i) {
        const Node& n = *order[i]; mdim_node& d = nodes[i];
        std::memset(&d, 0, sizeof d);
        d.kind = n.kind; d.dtype = n.dtype; d.op = n.op; d.src_dtype = n.src_dtype; d.data = n.data; d.offset = n.offset; d.imm = n.imm;
        if (!n.peers.empty()) { d.n_peers = (int)n.peers.size(); d.peer_block = n.peer_block; d.data = nullptr; for (size_t p = 0; p < n.peers.size(); ++p) d.peer[p] = n.peers[p]; }
        for (auto& [a, s] : n.stride) d.stride[pos(a)] = s;
        if (n.kind == MDIM_NODE_GATHER) { d.n_comp = (int)n.kids.size(); for (size_t c = 0; c < n.kids.size(); ++c) { d.gstride[c] = n.gstride[c]; d.bound[c] = n.bound[c]; } }
        if (n.kind == MDIM_NODE_CONCAT) { d.axis_a[0] = pos(n.pairs[0].a); d.axis_c[0] = n.pairs[0].c; }
        if (n.kind == MDIM_NODE_DIAG) {
            d.n_comp = (int)n.pairs.size();
            for (size_t p = 0; p < n.pairs.size(); ++p) {
                d.axis_a[p] = pos(n.pairs[p].a);
                if (n.pairs[p].b) { d.axis_b[p] = pos(n.pairs[p].b); d.axis_c[p] = (uint64_t)n.pairs[p].off; }
                else { d.axis_b[p] = -1; d.axis_c[p] = n.pairs[p].c; }
            }
        }
    }
    mdim_expr e; std::memset(&e, 0, sizeof e);
    e.abi_version = MDIM_ABI_VERSION; e.rank = (int)axes.size(); e.red_rank = (int)red.size(); e.n_nodes = (int)nodes.size(); e.nodes = nodes.data();
    for (size_t i = 0; i < all.size(); ++i) e.length[i] = all[i]->length;
    mdim_error_info err; std::memset(&err, 0, sizeof err);
    const int st = ex.run(&e, out_host, &err);
    if (st != MDIM_OK) throw Panic(st, err);
}

// ---- View<I, T> (src/view.rs:116-653) ------------------------------------------------------------------------
template <class I, class T> class View;
template <class I, class T> class Array;
template <class I, class T, class U> struct PairView;
template <class V, class I_, class J_> class Rows;

namespace detail {
inline NodeP make_binary(int op, const NodeP& a, const NodeP& b) {
    auto n = std::make_shared<Node>(); n->kind = MDIM_NODE_BINARY; n->dtype = a->dtype; n->op = op; n->kids = {a, b}; return n;
}
inline NodeP make_unary(int op, int dtype, const NodeP& a) {
    auto n = std::make_shared<Node>(); n->kind = MDIM_NODE_UNARY; n->dtype = dtype; n->op = op; n->src_dtype = a->dtype; n->kids = {a}; return n;
}
// Broadcast (src/broadcast.rs:22-162): result type, size, and the axis unification that replaces Broadcast::index
template <class A, class B, class = void> struct Bc;  // primary: no impl => compile error, like a missing trait impl
template <class A> struct Bc<A, A, std::enable_if_t<(n_leaves<A> == 1) && !std::is_same_v<A, Unit> && std::is_same_v<typename Ix<A>::Flat, std::tuple<A>>>> {  // NonTuple vs itself
    using R = A;
    static SizeOf<A> go(const SizeOf<A>& sa, const SizeOf<A>& sb, Groups& ga, Groups& gb, Groups& out, Table& tv, Table& tw) {
        if (!(sa == sb)) throw Panic(MDIM_ERR_SIZE, "Unequal sizes");  // src/broadcast.rs:38
        auto a = ga.front(), b = gb.front(); ga.erase(ga.begin()); gb.erase(gb.begin());
        out.push_back(unify_group(a, b, tv, tw)); return sa;  // the two sides may split this axis differently (to_usize)
    }
};
template <class B> struct Bc<Unit, B, std::enable_if_t<!std::is_same_v<B, Unit>>> {  // () expands to any Expand type
    using R = B;
    static SizeOf<B> go(const Unit&, const SizeOf<B>& sb, Groups&, Groups& gb, Groups& out, Table&, Table&) {
        for (size_t k = 0; k < n_leaves<B>; ++k) { out.push_back(gb.front()); gb.erase(gb.begin()); } return sb;
    }
};
template <class A> struct Bc<A, Unit, std::enable_if_t<!std::is_same_v<A, Unit>>> {
    using R = A;
    static SizeOf<A> go(const SizeOf<A>& sa, const Unit&, Groups& ga, Groups&, Groups& out, Table&, Table&) {
        for (size_t k = 0; k < n_leaves<A>; ++k) { out.push_back(ga.front()); ga.erase(ga.begin()); } return sa;
    }
};
template <class... As, class... Bs> struct Bc<std::tuple<As...>, std::tuple<Bs...>, std::enable_if_t<(sizeof...(As) == sizeof...(Bs)) && (sizeof...(As) > 0)>> {
    using R = std::tuple<typename Bc<As, Bs>::R...>;
    static SizeOf<R> go(const std::tuple<SizeOf<As>...>& sa, const std::tuple<SizeOf<Bs>...>& sb, Groups& ga, Groups& gb, Groups& out, Table& tv, Table& tw) {
        return go_(sa, sb, ga, gb, out, tv, tw, std::index_sequence_for<As...>{});
    }
    template <size_t... K> static SizeOf<R> go_(const std::tuple<SizeOf<As>...>& sa, const std::tuple<SizeOf<Bs>...>& sb, Groups& ga, Groups& gb, Groups& out, Table& tv, Table& tw, std::index_sequence<K...>) {
        return SizeOf<R>{Bc<As, Bs>::go(std::get<K>(sa), std::get<K>(sb), ga, gb, out, tv, tw)...};
    }
};
}  // namespace detail

template <class I, class T> class View {
  public:
    using Index = I; using Elem = T;
    View(SizeOf<I> size, Groups groups, NodeP value) : size_(std::move(size)), groups_(std::move(groups)), value_(std::move(value)) {}
    const SizeOf<I>& size() const { return size_; }
    uint64_t len() const { return length<I>(size_); }  // src/view.rs:127
    const Groups& groups() const { return groups_; }
    const NodeP& value() const { return value_; }

    // View::collect (src/view.rs:146-150): ONE fused kernel through the executor
    Array<I, T> collect(const Executor& ex) const;

    // a copy whose axes are fresh objects (two uses of one view must not alias when they are combined)
    View fresh() const {
        Table t; Groups g;
        for (auto& grp : groups_) { g.emplace_back(); for (auto& a : grp) { auto b = std::make_shared<Axis>(*a); t.push_back({a.get(), rename_to(b)}); g.back().push_back(b); } }
        return View(size_, g, substitute(value_, t));
    }

    // map over the closed unary vocabulary (src/view.rs:299-303 takes a closure; see ops above)
    template <class U> View map() const { return View(size_, groups_, detail::make_unary(U::code, DType<T>::v, value_)); }
    template <class To> View<I, To> cast() const { return View<I, To>(size_, groups_, detail::make_unary(MDIM_CAST, DType<To>::v, value_)); }

    // binary::<_, B>() (src/view.rs:507-512) with Broadcast (src/broadcast.rs)
    template <class B, class J> View<typename detail::Bc<I, J>::R, T> binary(const View<J, T>& other) const {
        using R = typename detail::Bc<I, J>::R;
        View<J, T> w = other.fresh();
        Groups ga = groups_, gb = w.groups(), out; Table tv, tw;
        SizeOf<R> s = detail::Bc<I, J>::go(size_, w.size(), ga, gb, out, tv, tw);
        return View<R, T>(s, out, detail::make_binary(B::code, substitute(value_, tv), substitute(w.value(), tw)));
    }
    // zip (src/view.rs:490-497) with ops::Pair (src/ops.rs:25-29): tuple-typed elements are kept as a structure of arrays
    template <class J, class U> PairView<typename detail::Bc<I, J>::R, T, U> zip(const View<J, U>& other) const {
        using R = typename detail::Bc<I, J>::R;
        View<J, U> w = other.fresh();
        Groups ga = groups_, gb = w.groups(), out; Table tv, tw;
        SizeOf<R> s = detail::Bc<I, J>::go(size_, w.size(), ga, gb, out, tv, tw);
        return PairView<R, T, U>{View<R, T>(s, out, substitute(value_, tv)), View<R, U>(s, out, substitute(w.value(), tw))};
    }
    // enumerate (src/view.rs:267-269) for a usize-indexed view: (index, value)
    PairView<I, usize, T> enumerate() const {
        static_assert(std::is_same_v<I, usize>, "enumerate: this header lowers usize-indexed views (compound indices: the Python mirror)");
        auto n = std::make_shared<Node>(); n->kind = MDIM_NODE_IOTA; n->dtype = MDIM_U64;
        int64_t acc = 1;
        for (auto it = groups_[0].rbegin(); it != groups_[0].rend(); ++it) { n->stride.push_back({*it, acc}); acc *= (int64_t)(*it)->length; }
        return PairView<I, usize, T>{View<I, usize>(size_, groups_, n), *this};
    }
    // The block of this view owned by `rank` when its OUTERMOST position axis is cut into `world` contiguous blocks (the north
    // star's partitioning; multidimension_b200/sharding.py::shard_view): the outer coordinate becomes lo + k.
    View shard(int rank, int world) const {
        static_assert(n_leaves<I> >= 1, "a rank-0 view has no axis to shard");
        if (groups_.empty() || groups_[0].size() != 1) throw Unsupported("the outermost axis has been re-split: shard before merging it");
        const AxisP outer = groups_[0][0];
        const uint64_t q = outer->length / (uint64_t)world, r = outer->length % (uint64_t)world;
        const uint64_t lo = (uint64_t)rank * q + std::min<uint64_t>((uint64_t)rank, r), n = q + ((uint64_t)rank < r ? 1 : 0);
        auto k = std::make_shared<Axis>(Axis{n});
        Sub_ sub; sub.constant = (int64_t)lo; sub.terms.push_back({k, 1});
        Table t{{outer.get(), sub}};
        Groups g = groups_; g[0] = {k};
        std::vector<uint64_t> flat_sz; Ix<I>::flat_size(size_, flat_sz);
        if (flat_sz.empty()) throw Unsupported("the outermost axis must be a usize axis to be sharded");
        flat_sz[0] = n; flat_sz.push_back(0);
        const uint64_t* it = flat_sz.data();
        return View(Ix<I>::build(it), g, substitute(value_, t));
    }
    template <class J> auto operator+(const View<J, T>& o) const { return binary<Add>(o); }
    template <class J> auto operator-(const View<J, T>& o) const { return binary<Sub>(o); }
    template <class J> auto operator*(const View<J, T>& o) const { return binary<Mul>(o); }
    template <class J> auto operator/(const View<J, T>& o) const { return binary<Div>(o); }
    template <class J> auto operator%(const View<J, T>& o) const { return binary<Rem>(o); }
    template <class J> auto operator&(const View<J, T>& o) const { return binary<BitAnd>(o); }
    template <class J> auto operator|(const View<J, T>& o) const { return binary<BitOr>(o); }
    template <class J> auto operator^(const View<J, T>& o) const { return binary<BitXor>(o); }

    // compose (src/view.rs:314-316): self is the INDEX view (T == W::I), other the source
    template <class U> View<I, U> compose(const View<T, U>& source) const {
        static_assert(std::is_same_v<T, usize>, "compose: only usize-indexed sources are lowered by this header (tuple indices: zip the components in Python)");
        View<T, U> w = source.fresh();
        const AxisP ax = w.groups().at(0).at(0);
        return View<I, U>(size_, groups_, gather(w.value(), ax, value_));
    }

    // diagonal (src/view.rs:285-287)
    View<std::tuple<I, I>, T> diagonal(T zero) const {
        Groups twin; auto n = std::make_shared<Node>();
        n->kind = MDIM_NODE_DIAG; n->dtype = DType<T>::v; n->kids = {value_}; n->imm = scalar_of(zero);
        for (auto& grp : groups_) { twin.emplace_back(); for (auto& a : grp) { auto b = std::make_shared<Axis>(*a); twin.back().push_back(b); n->pairs.push_back({a, b, 0, 0}); } }
        Groups g = groups_; g.insert(g.end(), twin.begin(), twin.end());
        return View<std::tuple<I, I>, T>(std::make_tuple(size_, size_), g, n->pairs.empty() ? value_ : NodeP(n));
    }

    // iso (src/view.rs:559-564): no data movement, no change in position space
    template <class J> View<J, T> iso() const { return View<J, T>(to_iso_size<I, J>(size_), groups_, value_); }

    // transpose::<I, X, Y, J>() (src/view.rs:586-592): self.I iso (I,(Y,X),J) -> (I,(X,Y),J)
    template <class I0, class X, class Y, class J0> View<std::tuple<I0, std::tuple<X, Y>, J0>, T> transpose() const {
        using In = std::tuple<I0, std::tuple<Y, X>, J0>;
        using Out = std::tuple<I0, std::tuple<X, Y>, J0>;
        auto s = to_iso_size<I, In>(size_);
        SizeOf<Out> so{std::get<0>(s), std::make_tuple(std::get<1>(std::get<1>(s)), std::get<0>(std::get<1>(s))), std::get<2>(s)};
        const size_t ni = n_leaves<I0>, ny = n_leaves<Y>, nx = n_leaves<X>;
        Groups g(groups_.begin(), groups_.begin() + ni);
        g.insert(g.end(), groups_.begin() + ni + ny, groups_.begin() + ni + ny + nx);
        g.insert(g.end(), groups_.begin() + ni, groups_.begin() + ni + ny);
        g.insert(g.end(), groups_.begin() + ni + ny + nx, groups_.end());
        return View<Out, T>(so, g, value_);
    }

    // row::<I, J>(i) / column::<I, J>(j) (src/view.rs:609-614, 639-644)
    template <class I0, class J0> View<J0, T> row(const I0& i) const {
        auto s = to_iso_size<I, std::tuple<I0, J0>>(size_);
        std::vector<uint64_t> p; Ix<I0>::positions(i, std::get<0>(s), p);
        Groups gi(groups_.begin(), groups_.begin() + n_leaves<I0>), gj(groups_.begin() + n_leaves<I0>, groups_.end());
        Table t; auto ax = flat(gi); for (size_t k = 0; k < ax.size(); ++k) t.push_back({ax[k].get(), pin_at(p[k])});
        return View<J0, T>(std::get<1>(s), gj, substitute(value_, t));
    }
    template <class I0, class J0> View<I0, T> column(const J0& j) const {
        auto s = to_iso_size<I, std::tuple<I0, J0>>(size_);
        std::vector<uint64_t> p; Ix<J0>::positions(j, std::get<1>(s), p);
        Groups gi(groups_.begin(), groups_.begin() + n_leaves<I0>), gj(groups_.begin() + n_leaves<I0>, groups_.end());
        Table t; auto ax = flat(gj); for (size_t k = 0; k < ax.size(); ++k) t.push_back({ax[k].get(), pin_at(p[k])});
        return View<I0, T>(std::get<0>(s), gi, substitute(value_, t));
    }
    // concat::<I, J>(other) (src/view.rs:327-339, 920-946): along the usize axis between I and J; only the
    // selected side is evaluated (:938-945), W addressed with k - len(V)
    template <class I0, class J0, class IW> View<std::tuple<I0, usize, J0>, T> concat(const View<IW, T>& other) const {
        using Mid = std::tuple<I0, usize, J0>;
        auto sv = to_iso_size<I, Mid>(size_);
        auto sw = to_iso_size<IW, Mid>(other.size());
        if (!(std::get<0>(sv) == std::get<0>(sw)) || !(std::get<2>(sv) == std::get<2>(sw)))  // assert_eq!(self_i, other_i) / (self_j, other_j), :336-337
            throw Panic(MDIM_ERR_SIZE, "assertion `left == right` failed");
        View<IW, T> w = other.fresh();
        const size_t ni = n_leaves<I0>;
        if (groups_[ni].size() != 1 || w.groups()[ni].size() != 1) throw Unsupported("concat along an axis that is a merged group (to_usize) needs device div/mod");
        const uint64_t nv = std::get<1>(sv), nw = std::get<1>(sw);
        auto K = std::make_shared<Axis>(Axis{nv + nw});
        Table tv{{groups_[ni][0].get(), rename_to(K)}}, tw;
        Groups g = groups_;
        for (size_t k = 0; k < groups_.size(); ++k)
            if (k != ni) g[k] = unify_group(groups_[k], w.groups()[k], tv, tw);  // the two sides may split an axis differently (to_usize)
        Sub_ shifted; shifted.constant = -(int64_t)nv; shifted.terms.push_back({K, 1});
        tw.push_back({w.groups()[ni][0].get(), shifted});
        auto n = std::make_shared<Node>();
        n->kind = MDIM_NODE_CONCAT; n->dtype = DType<T>::v; n->kids = {substitute(value_, tv), substitute(w.value(), tw)}; n->pairs.push_back({K, nullptr, nv, 0});
        g[ni] = {K};
        return View<Mid, T>(SizeOf<Mid>{std::get<0>(sv), nv + nw, std::get<2>(sv)}, g, NodeP(n));
    }
    // from_usize::<I, X, J>(size of X) (src/view.rs:352-363, 993-1021): the usize axis is re-indexed by X;
    // its coordinate becomes x.to_usize(size), row-major over X's position axes.  (The reference takes a closure
    // old_size -> X::Size; the caller evaluates it.)
    template <class I0, class X, class J0> View<std::tuple<I0, X, J0>, T> from_usize(const SizeOf<X>& xsize) const {
        using In = std::tuple<I0, usize, J0>;
        using Out = std::tuple<I0, X, J0>;
        auto s = to_iso_size<I, In>(size_);
        if (length<X>(xsize) != std::get<1>(s))  // assert_eq!(X::length(size), old_size), src/view.rs:361
            throw Panic(MDIM_ERR_SIZE, "assertion `left == right` failed\n  left: " + std::to_string(length<X>(xsize)) + "\n right: " + std::to_string(std::get<1>(s)));
        const size_t ni = n_leaves<I0>;
        // the usize axis may itself be a merged group (a to_usize further down): both factorisations are rewritten over their refinement
        std::vector<uint64_t> lold, lx, pieces; std::vector<std::vector<size_t>> mo, mx;
        for (auto& a : groups_[ni]) lold.push_back(a->length);
        Ix<X>::lengths(xsize, lx);
        refine(lold, lx, pieces, mo, mx);
        std::vector<AxisP> axes;
        for (uint64_t n : pieces) axes.push_back(std::make_shared<Axis>(Axis{n}));
        Table t;
        for (size_t k = 0; k < groups_[ni].size(); ++k) { std::vector<AxisP> pc; for (size_t q : mo[k]) pc.push_back(axes[q]); t.push_back({groups_[ni][k].get(), sub_of(pc)}); }
        Groups gx;
        for (size_t k = 0; k < lx.size(); ++k) { gx.emplace_back(); for (size_t q : mx[k]) gx.back().push_back(axes[q]); }
        Groups g(groups_.begin(), groups_.begin() + ni);
        g.insert(g.end(), gx.begin(), gx.end());
        g.insert(g.end(), groups_.begin() + ni + 1, groups_.end());
        return View<Out, T>(SizeOf<Out>{std::get<0>(s), xsize, std::get<2>(s)}, g, substitute(value_, t));
    }
    // to_usize::<I, X, J>() (src/view.rs:373-378, 1029-1059): in position space an axis indexed by X and the usize
    // axis of length X::length are the same run of positions; the merged axis is kept as ONE group of axes.
    template <class I0, class X, class J0> View<std::tuple<I0, usize, J0>, T> to_usize() const {
        using In = std::tuple<I0, X, J0>;
        using Out = std::tuple<I0, usize, J0>;
        auto s = to_iso_size<I, In>(size_);
        const size_t ni = n_leaves<I0>, nx = n_leaves<X>;
        Groups g(groups_.begin(), groups_.begin() + ni);
        std::vector<AxisP> merged;
        for (size_t k = ni; k < ni + nx; ++k) merged.insert(merged.end(), groups_[k].begin(), groups_[k].end());
        g.push_back(merged);
        g.insert(g.end(), groups_.begin() + ni + nx, groups_.end());
        return View<Out, T>(SizeOf<Out>{std::get<0>(s), length<X>(std::get<1>(s)), std::get<2>(s)}, g, value_);
    }
    // insert_one::<I, J, K>(size) (src/view.rs:391-397): a new axis of type J and length 1
    template <class I0, class J0, class K0> View<std::tuple<I0, J0, K0>, T> insert_one(const SizeOf<J0>& jsize) const {
        using In = std::tuple<I0, K0>;
        using Out = std::tuple<I0, J0, K0>;
        if (length<J0>(jsize) != 1)  // src/view.rs:395
            throw Panic(MDIM_ERR_SIZE, "assertion `left == right` failed\n  left: " + std::to_string(length<J0>(jsize)) + "\n right: 1");
        auto s = to_iso_size<I, In>(size_);
        Groups g(groups_.begin(), groups_.begin() + n_leaves<I0>);
        Groups gj = fresh_groups<J0>(jsize);
        g.insert(g.end(), gj.begin(), gj.end());
        g.insert(g.end(), groups_.begin() + n_leaves<I0>, groups_.end());
        return View<Out, T>(SizeOf<Out>{std::get<0>(s), jsize, std::get<1>(s)}, g, value_);
    }
    // remove_one::<I, J, K>() (src/view.rs:408-418): drop an axis of length 1 (its coordinate is pinned at 0)
    template <class I0, class J0, class K0> View<std::tuple<I0, K0>, T> remove_one() const {
        using In = std::tuple<I0, J0, K0>;
        using Out = std::tuple<I0, K0>;
        auto s = to_iso_size<I, In>(size_);
        if (length<J0>(std::get<1>(s)) != 1)  // src/view.rs:413
            throw Panic(MDIM_ERR_SIZE, "assertion `left == right` failed\n  left: " + std::to_string(length<J0>(std::get<1>(s))) + "\n right: 1");
        const size_t ni = n_leaves<I0>, nj = n_leaves<J0>;
        Table t;
        for (size_t k = ni; k < ni + nj; ++k) for (auto& a : groups_[k]) t.push_back({a.get(), pin_at(0)});
        Groups g(groups_.begin(), groups_.begin() + ni);
        g.insert(g.end(), groups_.begin() + ni + nj, groups_.end());
        return View<Out, T>(SizeOf<Out>{std::get<0>(s), std::get<2>(s)}, g, substitute(value_, t));
    }
    // map_axis::<I, V, J>(other) (src/view.rs:436-442, 1140-1170): at((i, x, j)) = self.at((i, other.at(x), j)) —
    // a gather along ONE axis (`take`); `other` is a view of usize indices, bounds-checked like usize::to_usize.
    template <class I0, class J0, class X> View<std::tuple<I0, X, J0>, T> map_axis(const View<X, usize>& other) const {
        using In = std::tuple<I0, usize, J0>;
        using Out = std::tuple<I0, X, J0>;
        auto s = to_iso_size<I, In>(size_);
        const size_t ni = n_leaves<I0>;
        if (groups_[ni].size() != 1) throw Unsupported("map_axis along an axis that is a merged group (to_usize) needs device div/mod");
        View<X, usize> w = other.fresh();
        Groups g(groups_.begin(), groups_.begin() + ni);
        g.insert(g.end(), w.groups().begin(), w.groups().end());
        g.insert(g.end(), groups_.begin() + ni + 1, groups_.end());
        return View<Out, T>(SizeOf<Out>{std::get<0>(s), w.size(), std::get<2>(s)}, g, gather(value_, groups_[ni][0], w.value()));
    }
    // rows::<I, J>() (src/view.rs:617-622): on the device its one use is .fold<B>(init)
    template <class I0, class J0> Rows<View, I0, J0> rows() const { return Rows<View, I0, J0>(*this); }

  protected:
    static NodeP gather(const NodeP& n, const AxisP& ax, const NodeP& comp) {
        if (n->kind == MDIM_NODE_CONST) return n;
        if (n->kind == MDIM_NODE_UNARY || n->kind == MDIM_NODE_BINARY || (n->kind == MDIM_NODE_CONCAT && n->pairs[0].a != ax)) {
            auto o = std::make_shared<Node>(*n); for (auto& k : o->kids) k = gather(k, ax, comp); return o;
        }
        if (n->kind == MDIM_NODE_LEAF || n->kind == MDIM_NODE_GATHER) {
            auto o = std::make_shared<Node>(*n);
            for (auto& k : o->kids) k = gather(k, ax, comp);
            o->stride.clear();
            bool hit = false;
            for (auto& [a, s] : n->stride) {
                if (a == ax) { o->kids.push_back(comp); o->gstride.push_back(s); o->bound.push_back(ax->length); hit = true; }
                else o->stride.push_back({a, s});
            }
            if (hit || n->kind == MDIM_NODE_GATHER) o->kind = MDIM_NODE_GATHER;
            return o;
        }
        if (n->kind == MDIM_NODE_IOTA) {
            bool hit = false; for (auto& e : n->stride) if (e.first == ax) hit = true;
            if (!hit) return n;
            if (n->stride.size() == 1 && n->stride[0].second == 1 && n->offset == 0) return comp;  // All::at(index) = index
        }
        throw Unsupported("compose onto a view containing diagonal(), a fold or a compound All");
    }
    SizeOf<I> size_;
    Groups groups_;
    NodeP value_;
};

// Rows<V, I, J>::fold<B>(init) == rows().map(|row| { let mut s = init; row.each(|x| s = B::call(s, x)); s })
template <class V, class I_, class J_> class Rows {
  public:
    explicit Rows(const V& v) : v_(v) {}
    template <class B> View<I_, typename V::Elem> fold(typename V::Elem init) const {
        using T = typename V::Elem;
        auto s = to_iso_size<typename V::Index, std::tuple<I_, J_>>(v_.size());
        Groups gi(v_.groups().begin(), v_.groups().begin() + n_leaves<I_>), gj(v_.groups().begin() + n_leaves<I_>, v_.groups().end());
        // the reduction axes become private to the fold: the same Array may also appear outside it
        Table t; std::vector<AxisP> red;
        for (auto& a : flat(gj)) { auto b = std::make_shared<Axis>(*a); t.push_back({a.get(), rename_to(b)}); red.push_back(b); }
        auto n = std::make_shared<Node>();
        n->kind = MDIM_NODE_FOLD; n->dtype = DType<T>::v; n->op = B::code; n->kids = {substitute(v_.value(), t)}; n->imm = scalar_of(init); n->red_axes = red;
        return View<I_, T>(std::get<0>(s), gi, n);
    }
  private:
    V v_;
};

// ---- Array<I, T> (src/array.rs:5-114): dense row-major items in host memory -----------------------------------
template <class I, class T> class Array : public View<I, T> {
  public:
    using Store = std::conditional_t<std::is_same_v<T, bool>, uint8_t, T>;
    // Array::new (src/array.rs:28-30); panics like Array::new_inner (:11-14) on a length mismatch
    Array(const SizeOf<I>& size, std::vector<Store> items) : Array(Shared{}, size, std::make_shared<std::vector<Store>>(std::move(items))) {}
    const std::vector<Store>& as_ref() const { return *items_; }  // AsRef<[T]> (src/array.rs:65-67)
    std::vector<Store> to_raw() const { return *items_; }         // src/array.rs:54
    template <class J> Array<J, T> iso() const { return Array<J, T>(typename Array<J, T>::Shared{}, to_iso_size<I, J>(this->size()), items_); }  // Array::iso, no data movement
    T at(const I& index) const {  // src/array.rs:81,86
        std::vector<uint64_t> p, l; Ix<I>::positions(index, this->size(), p); Ix<I>::lengths(this->size(), l);
        uint64_t k = 0; for (size_t a = 0; a < p.size(); ++a) k = k * l[a] + p[a];
        return (T)(*items_)[k];
    }
    struct Shared {};  // adopt an existing item vector (collect, iso)
    Array(Shared, const SizeOf<I>& size, std::shared_ptr<std::vector<Store>> items) : View<I, T>(size, fresh_groups<I>(size), nullptr), items_(std::move(items)) {
        if (items_->size() != length<I>(size))
            throw Panic(MDIM_ERR_SIZE, "assertion `left == right` failed\n  left: " + std::to_string(items_->size()) + "\n right: " + std::to_string(length<I>(size)));
        auto n = std::make_shared<Node>();
        n->kind = MDIM_NODE_LEAF; n->dtype = DType<T>::v; n->data = items_->data(); n->keep = items_;
        auto ax = flat(this->groups()); int64_t acc = 1;
        for (size_t k = ax.size(); k-- > 0;) { n->stride.push_back({ax[k], acc}); acc *= (int64_t)ax[k]->length; }  // row-major (src/index.rs:109-114)
        this->value_ = n;
    }
  private:
    std::shared_ptr<std::vector<Store>> items_;
};

template <class I, class T> Array<I, T> View<I, T>::collect(const Executor& ex) const {
    using Store = typename Array<I, T>::Store;
    auto out = std::make_shared<std::vector<Store>>(len());
    emit_and_run(value_, flat(groups_), ex, out->data());
    return Array<I, T>(typename Array<I, T>::Shared{}, size_, out);
}

// ---- tuple-typed elements (zip without an operator, enumerate): a structure of arrays, one View per scalar leaf -------------
template <class I, class T, class U> struct PairView {
    View<I, T> first; View<I, U> second;
    const SizeOf<I>& size() const { return first.size(); }
    // zip(..).map(|(x, y)| x (B) y): the pair consumed by an operator (what `a.zip(b).map(closure)` lowers to)
    template <class B> View<I, T> binary() const { static_assert(std::is_same_v<T, U>, "operands of different element types"); return View<I, T>(first.size(), first.groups(), detail::make_binary(B::code, first.value(), second.value())); }
    std::pair<Array<I, T>, Array<I, U>> collect(const Executor& ex) const { return {first.collect(ex), second.collect(ex)}; }
};

// ---- device-resident Arrays: the boxed buffer in HBM, optionally sharded over the GPUs of the box ------------------------------------
// The C ABI entry points, looked up in an already loaded libmdim_b200.so (this header links nothing).
struct Api {
    int (*init)(int, mdim_ctx**) = nullptr; int (*shutdown)(mdim_ctx*) = nullptr; int (*sync)(mdim_ctx*) = nullptr;
    int (*last_error)(mdim_ctx*, mdim_error_info*) = nullptr;
    int (*buf_alloc)(mdim_ctx*, size_t, void**) = nullptr; int (*buf_free)(mdim_ctx*, void*) = nullptr;
    int (*upload)(mdim_ctx*, void*, const void*, size_t) = nullptr; int (*download)(mdim_ctx*, void*, const void*, size_t) = nullptr;
    int (*collect)(mdim_ctx*, const mdim_expr*, void*, uint32_t) = nullptr; int (*collect_host)(mdim_ctx*, const mdim_expr*, void*, uint32_t) = nullptr;
    int (*comm_unique_id)(uint8_t*) = nullptr; int (*comm_init)(mdim_ctx*, int, int, const uint8_t*) = nullptr; int (*comm_destroy)(mdim_ctx*) = nullptr;
    int (*allgather)(mdim_ctx*, const void*, void*, size_t) = nullptr; int (*allreduce)(mdim_ctx*, void*, size_t, int, int) = nullptr; int (*barrier)(mdim_ctx*) = nullptr;
    int (*peer_table)(mdim_ctx*, void*, size_t, void**) = nullptr; int (*peer_table_close)(mdim_ctx*) = nullptr;
    // fold over the sharded axis as ONE fused compute + exchange kernel per GPU: the bit-exact chain through the ranks, and the blocked (all-reduce) route
    int (*fold_sharded_axis)(mdim_ctx*, const void*, uint64_t, uint64_t, int, int, mdim_scalar, void*) = nullptr;
    int (*fold_sharded_axis_blocked)(mdim_ctx*, const void*, uint64_t, uint64_t, int, int, mdim_scalar, void*) = nullptr;
    int (*fold_sharded_axis_status)(mdim_ctx*) = nullptr;
    template <class Sym> static Api load(Sym&& sym) {  // sym(name) -> void*
        Api a;
#define MDIM_API(field, name) a.field = reinterpret_cast<decltype(a.field)>(sym(name))
        MDIM_API(init, "mdim_init"); MDIM_API(shutdown, "mdim_shutdown"); MDIM_API(sync, "mdim_sync"); MDIM_API(last_error, "mdim_last_error");
        MDIM_API(buf_alloc, "mdim_buf_alloc"); MDIM_API(buf_free, "mdim_buf_free"); MDIM_API(upload, "mdim_upload"); MDIM_API(download, "mdim_download");
        MDIM_API(collect, "mdim_collect"); MDIM_API(collect_host, "mdim_collect_host");
        MDIM_API(comm_unique_id, "mdim_comm_unique_id"); MDIM_API(comm_init, "mdim_comm_init"); MDIM_API(comm_destroy, "mdim_comm_destroy");
        MDIM_API(allgather, "mdim_allgather"); MDIM_API(allreduce, "mdim_allreduce"); MDIM_API(barrier, "mdim_barrier");
        MDIM_API(peer_table, "mdim_peer_table"); MDIM_API(peer_table_close, "mdim_peer_table_close");
        MDIM_API(fold_sharded_axis, "mdim_fold_sharded_axis"); MDIM_API(fold_sharded_axis_blocked, "mdim_fold_sharded_axis_blocked");
        MDIM_API(fold_sharded_axis_status, "mdim_fold_sharded_axis_status");
#undef MDIM_API
        return a;
    }
    void check(mdim_ctx* ctx, int st) const {
        if (st == MDIM_OK) return;
        mdim_error_info info; std::memset(&info, 0, sizeof info);
        last_error(ctx, &info);
        if (info.status == st && info.message[0]) throw Panic(st, info);
        throw Panic(st, "mdim status " + std::to_string(st));
    }
    // device-resident operands and result: mdim_collect
    Executor device_resident(mdim_ctx* ctx) const {
        const Api self = *this;
        return Executor{[self, ctx](const mdim_expr* e, void* out, mdim_error_info* err) {
            const int st = self.collect(ctx, e, out, 0);
            if (st != MDIM_OK && err) self.last_error(ctx, err);
            return st;
        }};
    }
};

template <class I, class T> class DeviceArray : public View<I, T> {
  public:
    using Store = std::conditional_t<std::is_same_v<T, bool>, uint8_t, T>;
    // Array::new + upload (src/array.rs:28-30)
    DeviceArray(const Api& api, mdim_ctx* ctx, const SizeOf<I>& size, const std::vector<Store>& items) : View<I, T>(size, fresh_groups<I>(size), nullptr), buf_(alloc(api, ctx, items.size())) {
        if (items.size() != length<I>(size)) throw Panic(MDIM_ERR_SIZE, "assertion `left == right` failed");  // src/array.rs:12
        api.check(ctx, api.upload(ctx, buf_->ptr, items.data(), items.size() * sizeof(Store)));
        leaf({}, 0);
    }
    // an uninitialised result buffer (collect target)
    DeviceArray(const Api& api, mdim_ctx* ctx, const SizeOf<I>& size) : View<I, T>(size, fresh_groups<I>(size), nullptr), buf_(alloc(api, ctx, length<I>(size))) { leaf({}, 0); }
    // An Array sharded over the GPUs of the box in equal blocks of `block` elements, block p at peers[p] (mdim_peer_table):
    // every kernel reads the owning GPU's HBM over NVLink; a transpose does its all-to-all inside the tile loads.
    static DeviceArray sharded(const SizeOf<I>& size, const std::vector<const void*>& peers, uint64_t block, std::shared_ptr<void> keep = nullptr) {
        DeviceArray a(size, std::move(keep));
        a.leaf(peers, block);
        return a;
    }
    void* device_ptr() const { return buf_ ? buf_->ptr : nullptr; }
    size_t nbytes() const { return (size_t)this->len() * sizeof(Store); }
    std::vector<Store> to_raw() const {  // src/array.rs:54: downloads
        std::vector<Store> out(this->len());
        buf_->api.check(buf_->ctx, buf_->api.download(buf_->ctx, out.data(), buf_->ptr, out.size() * sizeof(Store)));
        return out;
    }
  private:
    struct Buf { Api api; mdim_ctx* ctx; void* ptr; ~Buf() { if (ptr) api.buf_free(ctx, ptr); } };
    static std::shared_ptr<Buf> alloc(const Api& api, mdim_ctx* ctx, size_t n) {
        void* p = nullptr;
        api.check(ctx, api.buf_alloc(ctx, n * sizeof(Store), &p));
        return std::shared_ptr<Buf>(new Buf{api, ctx, p});
    }
    DeviceArray(const SizeOf<I>& size, std::shared_ptr<void> keep) : View<I, T>(size, fresh_groups<I>(size), nullptr), keep_(std::move(keep)) {}
    void leaf(const std::vector<const void*>& peers, uint64_t block) {
        auto n = std::make_shared<Node>();
        n->kind = MDIM_NODE_LEAF; n->dtype = DType<T>::v; n->data = buf_ ? buf_->ptr : nullptr; n->keep = buf_ ? std::shared_ptr<void>(buf_, buf_.get()) : keep_;
        n->peers = peers; n->peer_block = block;
        auto ax = flat(this->groups()); int64_t acc = 1;
        for (size_t k = ax.size(); k-- > 0;) { n->stride.push_back({ax[k], acc}); acc *= (int64_t)ax[k]->length; }
        this->value_ = n;
    }
    std::shared_ptr<Buf> buf_;
    std::shared_ptr<void> keep_;
};
// View::collect into HBM: ONE fused kernel, operands and result device-resident
template <class I, class T> DeviceArray<I, T> collect_device(const View<I, T>& v, const Api& api, mdim_ctx* ctx) {
    DeviceArray<I, T> out(api, ctx, v.size());
    emit_and_run(v.value(), flat(v.groups()), api.device_resident(ctx), out.device_ptr());
    return out;
}

// ---- All<I> (src/index.rs:177-186) for usize, and Scalar<T> (src/view.rs:1399-1408) ------------------------------
inline View<usize, usize> all(uint64_t size) {
    Groups g = fresh_groups<usize>(size);
    auto n = std::make_shared<Node>(); n->kind = MDIM_NODE_IOTA; n->dtype = MDIM_U64; n->stride.push_back({g[0][0], 1});
    return View<usize, usize>(size, g, n);
}
// All<Reversed>: position p holds Reversed(size - 1 - p) (src/int.rs:82-84); the element is its usize payload
inline View<Reversed, usize> all_reversed(uint64_t size) {
    Groups g = fresh_groups<Reversed>(size);
    auto n = std::make_shared<Node>(); n->kind = MDIM_NODE_IOTA; n->dtype = MDIM_U64; n->offset = (int64_t)size - 1; n->stride.push_back({g[0][0], -1});
    return View<Reversed, usize>(size, g, n);
}
template <class T> View<Unit, T> Scalar(T value) {
    auto n = std::make_shared<Node>(); n->kind = MDIM_NODE_CONST; n->dtype = DType<T>::v; n->imm = scalar_of(value);
    return View<Unit, T>(Unit{}, Groups{}, n);
}

}  // namespace mdim
