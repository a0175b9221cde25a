"""Expression lowering: lazy View tree -> flattened position-space descriptor (mdim_expr).

This is the half of the north star that lives in src/view.rs in a Rust build ("expression
lowering and descriptor emission"): every reference node type is re-stated as a transformation of
a small scalar expression tree whose addressed nodes carry strides against NAMED position axes.
Index-remapping views (Transpose, Iso, Coat, Row, Column, FromUsize, ToUsize, InsertOne,
RemoveOne, broadcast in Zip) never touch data: they reorder, rename, split or pin axes, i.e. they
rewrite strides and offsets.  At `collect()` the root view's axes are numbered in to_usize order
(row-major, index.rs:109-114), the tree is written out in post-order as mdim_node[], and the
C ABI runs it as one fused kernel.
"""
from __future__ import annotations

import ctypes as C
import struct

from . import _ffi as F


class Unsupported(F.MdimError):
    """Valid in the reference, but not lowerable to the device (MDIM_ERR_UNSUPPORTED)."""

    def __init__(self, message):
        super().__init__(F.ERR_UNSUPPORTED, message)


class Axis:
    """One position-space axis (a leaf of a flattened index type) with its run-time length."""
    __slots__ = ("length", "tag")
    _count = 0

    def __init__(self, length):
        self.length = int(length)
        Axis._count += 1
        self.tag = Axis._count

    def __repr__(self):
        return f"ax{self.tag}[{self.length}]"


class Node:
    """One scalar-valued node.  `stride` maps Axis -> elements per step (absent = 0 = broadcast)."""
    __slots__ = ("kind", "dtype", "op", "children", "buf", "offset", "stride", "gstride", "bound", "pairs", "imm",
                 "src_dtype", "red_axes", "peers", "peer_block")

    def __init__(self, kind, dtype, **kw):
        self.kind = kind
        self.dtype = dtype
        self.op = kw.get("op", 0)
        self.children = kw.get("children", ())
        self.buf = kw.get("buf")            # storage object exposing .ptr (keeps the Array alive)
        self.offset = kw.get("offset", 0)
        self.stride = kw.get("stride", {})  # {Axis: int}
        self.gstride = kw.get("gstride", ())
        self.bound = kw.get("bound", ())
        self.pairs = kw.get("pairs", ())    # DIAG: ((Axis, Axis | int[, offset]), ...): coord[a] == coord[b] + offset | == int
        self.imm = kw.get("imm", 0)         # raw python value of `dtype`
        self.src_dtype = kw.get("src_dtype", 0)
        self.red_axes = kw.get("red_axes", ())  # FOLD: reduction axes, iterated last-fastest
        self.peers = kw.get("peers")
        self.peer_block = kw.get("peer_block", 0)

    def clone(self, **kw):
        n = Node(self.kind, self.dtype, op=self.op, children=self.children, buf=self.buf, offset=self.offset,
                 stride=self.stride, gstride=self.gstride, bound=self.bound, pairs=self.pairs, imm=self.imm,
                 src_dtype=self.src_dtype, red_axes=self.red_axes, peers=self.peers, peer_block=self.peer_block)
        for k, v in kw.items():
            setattr(n, k, v)
        return n


# A VALUE is a Node (scalar element) or a tuple of values (tuple-typed element, e.g. the pairs of
# `zip`, src/ops.rs:25-29, or the compound indices of `All<(I,J)>`, src/index.rs:177-186).
def map_value(value, fn):
    if isinstance(value, tuple):
        return tuple(map_value(v, fn) for v in value)
    return fn(value)


def flatten_value(value):
    if isinstance(value, tuple):
        out = []
        for v in value:
            out.extend(flatten_value(v))
        return out
    return [value]


class Sub:
    """Substitution of one old axis: coordinate = const + sum(coef * new_axis)."""
    __slots__ = ("const", "terms")

    def __init__(self, const=0, terms=()):
        self.const = const
        self.terms = tuple(terms)  # ((Axis, coef), ...)


def substitute(node, table, memo=None):
    """Rewrite every reference to the axes in `table` ({Axis: Sub}).  Linear in strides/offsets:
    stride'[n] += stride[a] * coef, offset' += stride[a] * const.  Shared subtrees stay shared."""
    if not table:
        return node
    if memo is None:
        memo = {}
    key = id(node)
    if key in memo:
        return memo[key]
    kids = tuple(substitute(c, table, memo) for c in node.children)
    out = node
    changed = any(k is not c for k, c in zip(kids, node.children))
    if node.kind in (F.LEAF, F.IOTA, F.GATHER) and any(a in table for a in node.stride):
        stride, offset = {}, node.offset
        for a, s in node.stride.items():
            sub = table.get(a)
            if sub is None:
                stride[a] = stride.get(a, 0) + s
            else:
                offset += s * sub.const
                for n, coef in sub.terms:
                    stride[n] = stride.get(n, 0) + s * coef
        out = node.clone(stride={a: s for a, s in stride.items() if s != 0}, offset=offset, children=kids)
    elif node.kind == F.DIAG and any((pr[0] in table) or (not isinstance(pr[1], int) and pr[1] in table) for pr in node.pairs):
        # each side is (axis | None, constant): coord[a] + ca == coord[b] + cb
        pairs, dead = [], False
        for pr in node.pairs:
            a, b = pr[0], pr[1]
            off = pr[2] if len(pr) > 2 else 0
            a2, ca = _sub_pred_side(a, table)
            b2, cb = _sub_pred_side(b, table)
            cb += off
            if a2 is None and b2 is None:
                if ca != cb:
                    dead = True  # statically off the diagonal
                continue
            if a2 is None:  # const == coord[b] + cb  ->  coord[b] == const - cb
                a2, b2, ca, cb = b2, None, cb, ca
            if b2 is None:
                k = cb - ca
                if k < 0:
                    dead = True
                    continue
                pairs.append((a2, int(k)))
            else:
                pairs.append((a2, b2, cb - ca))
        if dead:
            out = Node(F.CONST, node.dtype, imm=node.imm)
        elif not pairs:
            out = kids[0]
        else:
            out = node.clone(pairs=tuple(pairs), children=kids)
    elif node.kind == F.CONCAT and node.pairs[0][0] in table:
        sub, thr = table[node.pairs[0][0]], node.pairs[0][1]
        if not sub.terms:  # the concatenated axis has been pinned (row/column): one side survives
            out = kids[0] if sub.const < thr else kids[1]
        elif len(sub.terms) == 1 and sub.terms[0][1] == 1:  # k = k' + const:  k < thr  <=>  k' < thr - const
            out = node.clone(pairs=((sub.terms[0][0], max(thr - sub.const, 0)),), children=kids)
        else:
            raise Unsupported("a Concat whose axis has been split needs device div/mod")
    elif node.kind == F.FOLD and any(a in table for a in node.red_axes):
        raise Unsupported("substitution of a reduction axis")
    elif changed:
        out = node.clone(children=kids)
    memo[key] = out
    return out


def _sub_pred_side(x, table):
    """-> (axis | None, constant): the coordinate x after substitution is coord[axis] + constant."""
    if isinstance(x, int):
        return None, x
    sub = table.get(x)
    if sub is None:
        return x, 0
    if not sub.terms:
        return None, int(sub.const)
    if len(sub.terms) == 1 and sub.terms[0][1] == 1:
        return sub.terms[0][0], int(sub.const)
    raise Unsupported("a Diagonal whose axis has been split or merged needs device div/mod")


def rename(table):
    return {a: Sub(0, ((b, 1),)) for a, b in table.items()}


# ---- packing immediates -----------------------------------------------------------------------
_PACK = {F.U8: "<B", F.I32: "<i", F.U32: "<I", F.I64: "<q", F.U64: "<Q", F.F32: "<f", F.F64: "<d", F.I8: "<b", F.I16: "<h", F.U16: "<H"}


def imm_bits(dtype, value):
    if dtype in (F.F32, F.F64):
        raw = struct.pack(_PACK[dtype], float(value))
    else:
        width = F.DTYPE_SIZE[dtype] * 8
        v = int(value) & ((1 << width) - 1)
        raw = v.to_bytes(F.DTYPE_SIZE[dtype], "little")
    return int.from_bytes(raw.ljust(8, b"\0"), "little")


# ---- emission -----------------------------------------------------------------------------------
class Emitted:
    """An mdim_expr plus everything that must stay alive while it is in use."""

    def __init__(self, expr, nodes, keep, out_dtype, out_len, bufs):
        self.expr, self.nodes, self.keep, self.out_dtype, self.out_len, self.bufs = expr, nodes, keep, out_dtype, out_len, bufs


def emit(root, axes, location):
    """root: scalar Node, or a list of scalar Nodes — the scalar leaves of a tuple-typed element, written out under ONE
    MDIM_NODE_TUPLE root so that a single kernel launch fills every leaf's run (structure of arrays, include/mdim.h);
    axes: the output's position axes in to_usize order; location: 'device' | 'host' — which pointer of each storage to write."""
    order = []   # post-order, children before parents; shared subtrees are emitted per use
    red_axes = []
    if isinstance(root, (list, tuple)):
        if len(root) > F.MAX_OUTS:
            raise Unsupported(f"a tuple-typed element with {len(root)} scalar leaves (> {F.MAX_OUTS}): collect the leaves separately")
        root = Node(F.TUPLE, root[0].dtype, children=tuple(root))

    def visit(n):
        for c in n.children:
            visit(c)
        if n.kind == F.FOLD:
            if red_axes:
                raise Unsupported("more than one fold in one expression")
            red_axes.extend(n.red_axes)
        order.append(n)
    visit(root)
    if len(order) > F.MAX_NODES:
        raise Unsupported(f"expression has {len(order)} nodes (> {F.MAX_NODES})")
    all_axes = list(axes) + red_axes
    if len(all_axes) > F.MAX_RANK:
        raise Unsupported(f"expression has {len(all_axes)} position axes (> {F.MAX_RANK})")
    pos = {a: i for i, a in enumerate(all_axes)}
    arr = (F.Node * len(order))()
    bufs = []
    for i, n in enumerate(order):
        d = arr[i]
        d.kind, d.dtype, d.op = n.kind, n.dtype, n.op
        d.src_dtype = n.src_dtype
        if n.kind in (F.LEAF, F.IOTA, F.GATHER):
            d.offset = n.offset
            for a, s in n.stride.items():
                if a not in pos:
                    raise Unsupported(f"internal: node strides over an axis that is not iterated ({a!r})")
                d.stride[pos[a]] = s
        if n.kind in (F.LEAF, F.GATHER):
            if n.peers:
                d.n_peers = len(n.peers)
                for k, p in enumerate(n.peers):
                    d.peer[k] = p
                d.peer_block = n.peer_block
            else:
                d.data = n.buf.pointer(location)
            bufs.append(n.buf)
        if n.kind == F.GATHER:
            d.n_comp = len(n.children)
            for c in range(len(n.children)):
                d.gstride[c] = n.gstride[c]
                d.bound[c] = n.bound[c]
        if n.kind == F.DIAG:
            d.n_comp = len(n.pairs)
            for p, pr in enumerate(n.pairs):
                a, b = pr[0], pr[1]
                d.axis_a[p] = pos[a]
                if isinstance(b, int):
                    d.axis_b[p] = -1
                    d.axis_c[p] = b
                else:
                    d.axis_b[p] = pos[b]
                    d.axis_c[p] = (pr[2] if len(pr) > 2 else 0) & 0xFFFFFFFFFFFFFFFF
            d.imm.u64 = imm_bits(n.dtype, n.imm)
        if n.kind == F.CONCAT:
            d.axis_a[0] = pos[n.pairs[0][0]]
            d.axis_c[0] = n.pairs[0][1]
        if n.kind in (F.CONST, F.FOLD):
            d.imm.u64 = imm_bits(n.dtype, n.imm)
        if n.kind == F.FOLD and len(n.children) == 2:  # (init view, body): `let mut s = init.at(i)`
            d.n_comp = 2
        if n.kind == F.TUPLE:
            d.n_comp = len(n.children)
    e = F.Expr()
    e.abi_version = F.ABI_VERSION
    e.rank = len(axes)
    e.red_rank = len(red_axes)
    e.n_nodes = len(order)
    for i, a in enumerate(all_axes):
        e.length[i] = a.length
    e.nodes = C.cast(arr, C.POINTER(F.Node))
    out_len = 1
    for a in axes:
        out_len *= a.length
    em = Emitted(e, arr, order, root.dtype, out_len, bufs)
    em.out_dtypes = [c.dtype for c in root.children] if root.kind == F.TUPLE else [root.dtype]
    return em


# ---- splitting an expression that does not fit ONE fused kernel -----------------------------------------------------------------
# One mdim_expr is bounded (48 nodes, 56 instructions, 12 array operands, one FOLD: include/mdim.h).  The reference has no such
# bound — a View chain is as long as the user writes it — so collect() falls back to SEVERAL kernels: sub-expressions are collected
# into dense temporaries (over exactly the axes they depend on) and the rest of the tree reads them as ordinary Arrays.  Only nodes
# that the fused kernel would evaluate UNCONDITIONALLY are cut out (the spine below the root through operators and gather
# components); the inside of a Diagonal, of a Concat side and of a fold body stays in one piece, because the reference evaluates
# those lazily (src/view.rs:846-857, 920-946) and a temporary would evaluate — and possibly panic — where the reference does not.
_SPLIT_NODES, _SPLIT_OPERANDS = 20, 5    # a subtree beyond either is materialised: two such children + their parent stay under the limits


def axes_used(node, memo=None):
    """The position axes a value depends on (a fold's own reduction axes are internal to it)."""
    memo = {} if memo is None else memo
    if id(node) in memo:
        return memo[id(node)]
    used = set()
    for c in node.children:
        used |= axes_used(c, memo)
    if node.kind in (F.LEAF, F.IOTA, F.GATHER):
        used |= set(node.stride)  # zero strides too: emit() wants every named axis iterated
    if node.kind == F.DIAG:
        for pr in node.pairs:
            used.add(pr[0])
            if not isinstance(pr[1], int):
                used.add(pr[1])
    if node.kind == F.CONCAT:
        used.add(node.pairs[0][0])
    if node.kind == F.FOLD:
        used -= set(node.red_axes)
    memo[id(node)] = used
    return used


def _tree_cost(node):
    """(nodes, array operands, folds) of a subtree as emit() writes it (shared subtrees count per use)."""
    n, ops, folds = 1, int(node.kind in (F.LEAF, F.GATHER)), int(node.kind == F.FOLD)
    for c in node.children:
        cn, co, cf = _tree_cost(c)
        n, ops, folds = n + cn, ops + co, folds + cf
    return n, ops, folds


def split_for_limits(root, axes, materialise):
    """-> a tree equivalent to `root` in which every sub-expression beyond the split budget, and every fold but one, has been replaced
    by a LEAF over a dense temporary; `materialise(subtree, sub_axes) -> storage` collects one (row-major over `sub_axes`, the axes of
    `axes` the subtree depends on, in order).  -> None when nothing could be cut (the expression is too large INSIDE a lazy region)."""
    cut = [0]
    temps, seen = {}, {}   # a sub-expression used several times (a traced closure mentioning its argument twice) is collected ONCE

    def temp_leaf(node):
        if id(node) in temps:
            return temps[id(node)]
        used = axes_used(node)
        sub_axes = [a for a in axes if a in used]
        if len(sub_axes) != len(used):
            return None  # depends on an axis the root does not iterate (inside a fold body): not a spine node after all
        storage = materialise(node, sub_axes)
        stride, acc = {}, 1
        for a in reversed(sub_axes):
            stride[a] = acc
            acc *= a.length
        cut[0] += 1
        temps[id(node)] = Node(F.LEAF, node.dtype, buf=storage, stride=stride)
        return temps[id(node)]

    def visit(node, is_root):
        """-> (node', nodes, operands, folds) with every over-budget spine child already replaced."""
        if id(node) not in seen:
            seen[id(node)] = visit_once(node, is_root)
        return seen[id(node)]

    def visit_once(node, is_root):
        if node.kind == F.FOLD and len(node.children) == 2:  # a fold continued from a per-row initial VIEW (evaluated for every row): a fold in there runs first
            init, in_n, in_ops, in_folds = visit(node.children[0], False)
            if in_folds and init.kind not in (F.LEAF, F.CONST, F.IOTA):
                leaf = temp_leaf(init)
                if leaf is not None:
                    node = node.clone(children=(leaf, node.children[1]))
            elif init is not node.children[0]:
                node = node.clone(children=(init, node.children[1]))
            return (node,) + _tree_cost(node)
        if node.kind not in (F.UNARY, F.BINARY, F.GATHER, F.TUPLE):  # a unit: leaf, constant, iota, or a lazy region / fold as a whole
            return (node,) + _tree_cost(node)
        kids, costs = [], []
        folds = 0
        for c in node.children:
            c2, cn, co, cf = visit(c, False)
            over = cn > _SPLIT_NODES or co > _SPLIT_OPERANDS or (cf and folds)   # too big, or a second fold under this node
            if over and c2.kind not in (F.LEAF, F.CONST, F.IOTA):
                leaf = temp_leaf(c2)
                if leaf is not None:
                    c2, cn, co, cf = leaf, 1, 1, 0
            kids.append(c2)
            costs.append([cn, co, cf])
            folds += cf
        own_ops = int(node.kind == F.GATHER)
        while 1 + sum(c[0] for c in costs) > F.MAX_NODES - 4 or own_ops + sum(c[1] for c in costs) > 11:  # many children (gather components, a tuple)
            k = max(range(len(kids)), key=lambda i: costs[i][0] if kids[i].kind not in (F.LEAF, F.CONST, F.IOTA) else -1)
            if kids[k].kind in (F.LEAF, F.CONST, F.IOTA):
                break
            leaf = temp_leaf(kids[k])
            if leaf is None:
                break
            kids[k], costs[k] = leaf, [1, 1, 0]
        n, ops, folds = 1 + sum(c[0] for c in costs), own_ops + sum(c[1] for c in costs), sum(c[2] for c in costs)
        out = node.clone(children=tuple(kids)) if any(a is not b for a, b in zip(kids, node.children)) else node
        return out, n, ops, folds

    new_root, _, _, _ = visit(root, True)
    return new_root if cut[0] else None
