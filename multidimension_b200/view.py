"""Host-side mirror of the reference's `View` / `Array` API (src/view.rs, src/array.rs), backed by
the fused sm_100a kernels behind include/mdim.h.

Same names, argument meaning and panics as the reference: generic parameters become leading
arguments (`a.transpose::<(),usize,usize,()>()` is `a.transpose((), usize, usize, ())`).  A view
is lazy; `collect()` (src/view.rs:146-150) lowers the whole chain to one descriptor and runs it
as ONE kernel.  Nothing here computes elements on the CPU.
"""
from __future__ import annotations

import numpy as np

from . import _ffi as F
from . import index as X
from . import lowering as L
from . import ops as O
from .index import usize, Reversed, Fixed, Coated, Option
from .runtime import Storage, default_context, NP_OF

Panic = F.Panic
Unsupported = L.Unsupported

# ---- element types ------------------------------------------------------------------------------
_DT_OF_NAME = {"u8": F.U8, "i32": F.I32, "u32": F.U32, "i64": F.I64, "u64": F.U64, "f32": F.F32, "f64": F.F64,
               "i8": F.I8, "i16": F.I16, "u16": F.U16}
_NAME_OF_NP = {np.dtype(np.uint8): "u8", np.dtype(np.int32): "i32", np.dtype(np.uint32): "u32", np.dtype(np.int64): "i64",
               np.dtype(np.uint64): usize, np.dtype(np.float32): "f32", np.dtype(np.float64): "f64", np.dtype(np.bool_): bool,
               np.dtype(np.int8): "i8", np.dtype(np.int16): "i16", np.dtype(np.uint16): "u16"}


def dtype_of(T):
    """mdim_dtype of a scalar element type.  `usize` (and the other usize-like indices) is U64."""
    if T is usize or T is Reversed or isinstance(T, Fixed):
        return F.U64
    if T is bool:
        return F.U8
    if isinstance(T, str) and T in _DT_OF_NAME:
        return _DT_OF_NAME[T]
    raise TypeError(f"no device representation for element type {T!r}")


def _same_T(a, b):
    if isinstance(a, tuple) or isinstance(b, tuple):
        return isinstance(a, tuple) and isinstance(b, tuple) and len(a) == len(b) and all(_same_T(x, y) for x, y in zip(a, b))
    return dtype_of(a) == dtype_of(b) and (a is bool) == (b is bool)


def _T_leaves(T):
    if isinstance(T, tuple):
        out = []
        for t in T:
            out.extend(_T_leaves(t))
        return out
    return [T]


def _build_like(T, leaves):
    if isinstance(T, tuple):
        return tuple(_build_like(t, leaves) for t in T)
    return leaves.pop(0)


# ---- axis bookkeeping -----------------------------------------------------------------------------
def _fresh_groups(I, size):
    return [[L.Axis(n) for n in X.leaf_lengths(t, s)] for t, s in zip(X.type_leaves(I), X.size_leaves(I, size))]


def _flat(groups):
    return [a for g in groups for a in g]


def _split_groups(groups, *types):
    """Partition the per-leaf axis groups of a view indexed by something isomorphic to `types`."""
    out, k = [], 0
    for t in types:
        n = len(X.type_leaves(t))
        out.append(groups[k:k + n])
        k += n
    assert k == len(groups)
    return out


def _refine(lens_a, lens_b):
    """Common refinement of two row-major factorisations of the same run of positions (e.g. an axis merged by
    `to_usize` out of (2, 3) against a plain axis of 6, or (2, 6) against (4, 3)): -> (pieces, map_a, map_b) where
    `pieces` are the lengths of the refined axes in row-major order and map_x[i] lists the pieces that make up axis i
    of x, outermost first.  Raises Unsupported when no refinement exists (that remapping needs div/mod on the device)."""
    if 0 in lens_a or 0 in lens_b:
        raise Unsupported("re-splitting an empty axis")
    pieces, map_a, map_b = [], [[] for _ in lens_a], [[] for _ in lens_b]
    i = j = 0
    ra = rb = None  # what is left of axis i of a / axis j of b (None: not loaded yet)
    while True:
        while ra is None and i < len(lens_a):
            if lens_a[i] == 1:  # a unit axis is its own piece
                map_a[i].append(len(pieces)); pieces.append(1); i += 1
            else:
                ra = lens_a[i]
        while rb is None and j < len(lens_b):
            if lens_b[j] == 1:
                map_b[j].append(len(pieces)); pieces.append(1); j += 1
            else:
                rb = lens_b[j]
        if ra is None or rb is None:
            break
        if ra % rb == 0:
            step = rb
        elif rb % ra == 0:
            step = ra
        else:
            raise Unsupported(f"axis groups {lens_a} and {lens_b} have no common refinement: this remapping needs div/mod on the device")
        map_a[i].append(len(pieces)); map_b[j].append(len(pieces)); pieces.append(step)
        ra //= step
        rb //= step
        if ra == 1:
            i += 1; ra = None
        if rb == 1:
            j += 1; rb = None
    if ra is not None or rb is not None:
        raise Unsupported(f"axis groups {lens_a} and {lens_b} do not describe the same run of positions")
    return pieces, map_a, map_b


def _sub_of(piece_axes):
    """The coordinate of an axis cut into `piece_axes` (outermost first): row-major combination of the pieces."""
    terms, acc = [], 1
    for a in reversed(piece_axes):
        if a.length != 1:  # the coordinate along a unit axis is always 0 (and the axis may not be iterated at all)
            terms.append((a, acc))
        acc *= a.length
    return L.Sub(0, tuple(terms))


def _unify_group(a, b, table_v, table_w):
    """One leaf axis seen by both operands of a Zip / Concat as the groups `a` (self) and `b` (other): -> the group the
    result iterates.  Identical splits are renamed 1:1; different splits of the same run of positions (an axis produced
    by `to_usize`, src/view.rs:1029-1059) are both rewritten over their common refinement."""
    la, lb = [x.length for x in a], [y.length for y in b]
    if la == lb:
        for x, y in zip(a, b):
            table_w[y] = L.Sub(0, ((x, 1),))
        return a
    pieces, map_a, map_b = _refine(la, lb)
    axes = [L.Axis(n) for n in pieces]
    for x, idx in zip(a, map_a):
        table_v[x] = _sub_of([axes[k] for k in idx])
    for y, idx in zip(b, map_b):
        table_w[y] = _sub_of([axes[k] for k in idx])
    return axes


def _broadcast(I, J, si, sj, gi, gj, table_v, table_w):
    """Broadcast::{Result,size} (src/broadcast.rs:22-162) + the axis unification that replaces
    Broadcast::index: unified axes of `other` are rewritten in terms of `self`'s (table_w; table_v only when the two
    sides split an axis differently), missing ones stay absent (stride 0).  gi/gj are consumed from the front."""
    if I == () and J == ():
        raise TypeError("() does not implement Broadcast<()> (Expand excludes (), src/broadcast.rs:4-9)")
    if I == ():
        n = len(X.type_leaves(J))
        groups = [gj.pop(0) for _ in range(n)]
        return J, sj, groups
    if J == ():
        n = len(X.type_leaves(I))
        groups = [gi.pop(0) for _ in range(n)]
        return I, si, groups
    ti, tj = isinstance(I, tuple), isinstance(J, tuple)
    if not ti and not tj:
        if I != J:
            raise TypeError(f"{I!r} does not implement Broadcast<{J!r}>")
        if si != sj:
            raise Panic(F.ERR_SIZE, "Unequal sizes")  # src/broadcast.rs:38
        a, b = gi.pop(0), gj.pop(0)
        return I, si, [_unify_group(a, b, table_v, table_w)]
    if ti and tj and len(I) == len(J):
        Rs, ss, gs = [], [], []
        for a, b, x, y in zip(I, J, si, sj):
            R, s, g = _broadcast(a, b, x, y, gi, gj, table_v, table_w)
            Rs.append(R); ss.append(s); gs.extend(g)
        return tuple(Rs), tuple(ss), gs
    raise TypeError(f"{I!r} does not implement Broadcast<{J!r}>")


# ---- symbolic values for traced closures ---------------------------------------------------------------
class Sym:
    """A scalar element inside a traced `map` closure."""
    __slots__ = ("node", "T")

    def __init__(self, node, T):
        self.node, self.T = node, T

    def _lift(self, o):
        if isinstance(o, Sym):
            return o
        return Sym(L.Node(F.CONST, self.node.dtype, imm=o), self.T)

    def _bin(self, o, B, swap=False):
        o = self._lift(o)
        a, b = (o, self) if swap else (self, o)
        return Sym(_binary_node(B, a.node, b.node), a.T)

    def __add__(self, o): return self._bin(o, O.Add)
    def __radd__(self, o): return self._bin(o, O.Add, True)
    def __sub__(self, o): return self._bin(o, O.Sub)
    def __rsub__(self, o): return self._bin(o, O.Sub, True)
    def __mul__(self, o): return self._bin(o, O.Mul)
    def __rmul__(self, o): return self._bin(o, O.Mul, True)
    def __truediv__(self, o): return self._bin(o, O.Div)
    def __rtruediv__(self, o): return self._bin(o, O.Div, True)
    def __floordiv__(self, o): return self._bin(o, O.Div)
    def __mod__(self, o): return self._bin(o, O.Rem)
    def __and__(self, o): return self._bin(o, O.BitAnd)
    def __or__(self, o): return self._bin(o, O.BitOr)
    def __xor__(self, o): return self._bin(o, O.BitXor)
    def __lshift__(self, o): return self._bin(o, O.Shl)
    def __rshift__(self, o): return self._bin(o, O.Shr)
    def __neg__(self): return Sym(_unary_node(O.Neg, self.node), self.T)
    def __invert__(self): return Sym(_unary_node(O.Not, self.node, self.T is bool), self.T)
    def __abs__(self): return Sym(_unary_node(O.Abs, self.node), self.T)
    def sqrt(self): return Sym(_unary_node(O.Sqrt, self.node), self.T)

    def cast(self, T):  # Rust `as`
        return Sym(_cast_node(self.node, dtype_of(T)), T)


def _binary_node(B, a, b):
    if B.code is None:
        raise TypeError("ops::Pair has no scalar result")
    is_shift = B.code in (F.SHL, F.SHR)
    if not is_shift and a.dtype != b.dtype:
        raise TypeError(f"{B!r} on mismatched element types {F.DTYPE_NAME[a.dtype]} and {F.DTYPE_NAME[b.dtype]}")
    if a.dtype in (F.F32, F.F64) and B.code >= F.AND:
        raise TypeError(f"{B!r} is not implemented for floats")
    return L.Node(F.BINARY, a.dtype, op=B.code, children=(a, b))


def _unary_node(U, a, is_bool=False):
    if U.code == F.NOT and a.dtype in (F.F32, F.F64):
        raise TypeError("ops::Not is not implemented for floats")
    if U.code == F.NOT and is_bool:  # `!bool` is logical: the descriptor's NOT is bitwise on U8, so lower it as x ^ true
        return L.Node(F.BINARY, a.dtype, op=F.XOR, children=(a, L.Node(F.CONST, a.dtype, imm=1)))
    if U.code in (F.NEG, F.ABS, F.SQRT) and is_bool:
        raise TypeError(f"{U!r} is not implemented for bool")
    if U.code == F.SQRT and a.dtype not in (F.F32, F.F64):
        raise TypeError("sqrt is only defined for floats")
    return L.Node(F.UNARY, a.dtype, op=U.code, children=(a,), src_dtype=a.dtype)


def _cast_node(a, dtype):
    if a.dtype == dtype:
        return a
    return L.Node(F.UNARY, dtype, op=F.CAST, children=(a,), src_dtype=a.dtype)


def _to_syms(value, T):
    if isinstance(value, tuple):
        return tuple(_to_syms(v, t) for v, t in zip(value, T))
    return Sym(value, T)


def _from_syms(result):
    if isinstance(result, tuple):
        parts = [_from_syms(r) for r in result]
        return tuple(p[0] for p in parts), tuple(p[1] for p in parts)
    if not isinstance(result, Sym):
        raise Unsupported("a traced map closure must return values built from its argument")
    return result.node, result.T


# ---- the View trait (src/view.rs:116-653) ---------------------------------------------------------------------
class View:
    """`I` = index type, `T` = element type, `size()`, and every provided combinator."""
    I = None
    T = None

    def size(self):
        return self._size

    def len(self):  # src/view.rs:127
        return X.length(self.I, self._size)

    def _lower(self):
        """-> (groups, value): per type-leaf lists of position axes, and the element value tree."""
        raise NotImplementedError

    # -- collect ------------------------------------------------------------------------------------
    def collect(self, I=None, ctx=None, flags=0, location=None, out=None):
        """View::collect (src/view.rs:146-150) -> Array<I, T>.  `I` may be any index type isomorphic
        to `self.I` (`A: NewView<I=Self::I>` after an `iso`).  Operands that all live in host memory
        give a host Array through mdim_collect_host; otherwise the result is device-resident."""
        I_out = self.I if I is None else I
        size_out = self._size if I is None else X.to_iso_size(self._size, self.I, I_out)
        groups, value = self._lower()
        axes = _flat(groups)
        ctx = ctx or default_context()
        leaves_T = _T_leaves(self.T)
        storages = []
        outs = list(out) if isinstance(out, (tuple, list)) else ([out] if out is not None else [None] * len(leaves_T))
        nodes = L.flatten_value(value)

        def run_all(nodes):
            fused = _fused_sharded_axis_fold(ctx, nodes, axes, flags, outs[0]) if len(nodes) == 1 and location != "host" else None
            if fused is not None:
                return [fused]
            if 1 < len(nodes) <= F.MAX_OUTS and all(_location_of(n, location) == "device" for n in nodes):
                return _run_tuple(ctx, nodes, axes, flags, outs)  # ONE kernel launch: shared operands are read once
            # host-resident operands (mdim_collect_host is per leaf), or more leaves than one launch writes
            return [_run(ctx, node, axes, flags, location, o) for node, o in zip(nodes, outs)]
        try:
            storages = run_all(nodes)
        except F.MdimError as e:
            if e.status != F.ERR_UNSUPPORTED:
                raise
            # beyond what ONE fused kernel takes (nodes, instructions, operands, a second fold): several kernels through dense temporaries
            split = [L.split_for_limits(n, axes, lambda sub, sub_axes: _run(ctx, sub, sub_axes, flags, location, None)) for n in nodes]
            if all(n2 is None for n2 in split):
                raise
            storages = run_all([n2 if n2 is not None else n for n2, n in zip(split, nodes)])
        st = _build_like(self.T, list(storages)) if isinstance(self.T, tuple) else storages[0]
        return Array(I_out, size_out, st, self.T)

    def prepare(self, out=None, ctx=None, flags=0):
        """Lower once, run many times: returns a `Prepared` whose `run()` is a single C-ABI call (the lowering
        and descriptor emission are not repeated).  Device-resident operands and scalar element types only; ONE fused kernel:
        an expression beyond its limits raises Unsupported here (collect() splits such an expression, lowering.split_for_limits)."""
        groups, value = self._lower()
        if isinstance(value, tuple):
            raise Unsupported("prepare() of a tuple-typed view: prepare the components")
        ctx = ctx or default_context()

        def visit(n):
            for c in n.children:
                visit(c)
            if n.kind in (F.LEAF, F.GATHER) and n.buf is not None:
                n.buf.ensure_device(ctx)
        visit(value)
        em = L.emit(value, _flat(groups), "device")
        st = out if out is not None else Storage.device(ctx, em.out_dtype, em.out_len)
        if st.n != em.out_len or st.dtype != em.out_dtype:
            raise Panic(F.ERR_SIZE, "output buffer does not match the view")
        return Prepared(ctx, em, st, Array(self.I, self._size, st, self.T), flags)

    def describe(self, flags=0):
        """Which kernel the planner picks for this chain (needs the library, not a GPU)."""
        from .runtime import describe_nodevice
        groups, value = self._lower()
        out = []
        for node in L.flatten_value(value):
            em = L.emit(node, _flat(groups), "any")
            st, text = describe_nodevice(em.expr, flags)
            out.append(text if st == F.OK else f"error {st}: {text}")
        return out[0] if len(out) == 1 else out

    # -- combinators, in the order of src/view.rs ------------------------------------------------------------
    def enumerate(self):  # :267
        return Enumerate(self)

    def diagonal(self, zero):  # :285
        return Diagonal(self, zero)

    def map(self, f):  # :299
        return Map(self, f)

    def compose(self, other):  # :314
        return Compose(self, other)

    def concat(self, other, I, J):  # :327
        return Concat(self, other, I, J)

    def from_usize(self, I, Xt, J, from_length):  # :352
        return FromUsize(self, I, Xt, J, from_length)

    def to_usize(self, I, Xt, J):  # :373
        return ToUsize(self, I, Xt, J)

    def insert_one(self, I, J, K, size):  # :391
        return InsertOne(self, I, J, K, size)

    def remove_one(self, I, J, K):  # :408
        return RemoveOne(self, I, J, K)

    def map_axis(self, other, I, J):  # :436
        return MapAxis(self, I, other, J)

    def zip(self, other):  # :490
        return Zip(self, other, O.Pair)

    def binary(self, other, B):  # :507
        return Zip(self, other, B)

    def coat(self, I):  # :549
        return CoatView(self, I)

    def iso(self, J):  # :559
        return Iso(self, J)

    def transpose(self, I, Xt, Y, J):  # :586
        return Transpose(self, I, Xt, Y, J)

    def row(self, I, J, i):  # :609
        return Row(self, I, J, i)

    def rows(self, I, J):  # :617
        return Rows(self, I, J)

    def column(self, I, J, j):  # :639
        return Column(self, I, J, j)

    def columns(self, I, J):  # :647
        return Columns(self, I, J)

    # -- operator sugar of impl_ops_for_view! (src/ops.rs:159-208) ------------------------------------------------
    def __add__(self, o): return self.binary(_as_view(o, self), O.Add)
    def __sub__(self, o): return self.binary(_as_view(o, self), O.Sub)
    def __mul__(self, o): return self.binary(_as_view(o, self), O.Mul)
    def __truediv__(self, o): return self.binary(_as_view(o, self), O.Div)
    def __mod__(self, o): return self.binary(_as_view(o, self), O.Rem)
    def __and__(self, o): return self.binary(_as_view(o, self), O.BitAnd)
    def __or__(self, o): return self.binary(_as_view(o, self), O.BitOr)
    def __xor__(self, o): return self.binary(_as_view(o, self), O.BitXor)
    def __lshift__(self, o): return self.binary(_as_view(o, self), O.Shl)
    def __rshift__(self, o): return self.binary(_as_view(o, self), O.Shr)


class Prepared:
    """A lowered View chain bound to its operands and output buffer."""

    def __init__(self, ctx, em, storage, array, flags):
        import ctypes
        self.ctx, self.em, self.storage, self.array, self.flags = ctx, em, storage, array, flags
        self._collect = ctx.lib.mdim_collect
        self._args = (ctx.handle, ctypes.byref(em.expr), ctypes.c_void_p(storage.dptr))

    def run(self, flags=None):
        """View::collect into the bound buffer (one kernel launch); returns the result Array."""
        st = self._collect(*self._args, self.flags if flags is None else flags)
        if st != F.OK:
            self.ctx.check(st)
        return self.array


def _as_view(o, like):
    if isinstance(o, View):
        return o
    return Scalar(o, like.T)  # Python convenience: `a + 1.0` means `a + Scalar(1.0)`


def _location_of(node, requested):
    """'host' iff every operand lives in host memory (and nothing forces the device)."""
    homes = set()

    def visit(n):
        for c in n.children:
            visit(c)
        if n.kind in (F.LEAF, F.GATHER) and n.buf is not None:
            homes.add(n.buf.home)
        if n.kind == F.GATHER and n.peers:
            homes.add("device")
    visit(node)
    if requested:
        return requested
    return "host" if homes == {"host"} else "device"


def _run_tuple(ctx, nodes, axes, flags, outs):
    """Device-resident collect of a tuple-typed view: every scalar leaf's run from one launch (mdim_collect_tuple)."""
    def visit(n):
        for c in n.children:
            visit(c)
        if n.kind in (F.LEAF, F.GATHER) and n.buf is not None:
            n.buf.ensure_device(ctx)
    for n in nodes:
        visit(n)
    em = L.emit(list(nodes), axes, "device")
    sts = []
    for dt, o in zip(em.out_dtypes, outs):
        st = o if o is not None else Storage.device(ctx, dt, em.out_len)
        if st.n != em.out_len or st.dtype != dt:
            raise Panic(F.ERR_SIZE, "output buffer does not match the view")
        sts.append(st)
    ctx.collect_tuple(em.expr, [s.dptr for s in sts], flags)
    return sts


def _fused_sharded_axis_fold(ctx, nodes, axes, flags, out):
    """Planner rule for the one fold the evaluator serves badly: `rows().map(fold)` over the SHARDED (outermost) axis of a whole Array whose
    blocks live on the ranks of a communicator (a PeerStorage made by `sharding.peer_source`).  Read through the peer table every rank would
    pull all ranks' rows over NVLink (0.47 ms for config 4's Array on 8 GPUs); `mdim_fold_sharded_axis` hands the running values from rank
    to rank instead (0.071 ms) and gives the same bits — the reference's sequential chain — on EVERY rank.  Collective: every rank collects
    the same view.  -> the result Storage, or None when the view is anything else (then the ordinary path runs)."""
    node = nodes[0]
    if (flags & F.COLLECT_NO_FASTPATH) or node.kind != F.FOLD or len(node.children) != 1 or len(node.red_axes) != 1:
        return None
    leaf = node.children[0]
    st = leaf.buf
    comm = getattr(st, "comm", None)
    if leaf.kind != F.LEAF or comm is None or not leaf.peers or leaf.offset != 0 or leaf.dtype != node.dtype:
        return None
    if node.op not in (F.ADD, F.SUB, F.MUL, F.AND, F.OR, F.XOR) or node.dtype not in (F.F32, F.F64, F.I32, F.U32, F.I64, F.U64):
        return None
    red = node.red_axes[0]
    cols = 1
    for a in reversed(axes):  # the result walks the columns contiguously, in order
        if a.length != 1 and leaf.stride.get(a, 0) != cols:
            return None
        cols *= a.length
    if set(leaf.stride) - set(axes) - {red} or leaf.stride.get(red, 0) != cols or cols == 0:
        return None
    if red.length * cols != st.n or st.block % cols or st.block * comm.world != st.n or comm.ctx is not ctx:
        return None
    from .ops import BinaryOp
    local = Storage.wrap_device(ctx, st.dtype, st.block, st.peers[comm.rank], keep=st)
    try:
        res = comm.fold_sharded_axis(local, st.block // cols, cols, BinaryOp("fold", node.op), node.imm, out=out)
    except F.MdimError as e:
        if e.status == F.ERR_UNSUPPORTED:  # alignment / width limits of the fused kernel: the same answer on every rank
            return None
        raise
    if not (flags & F.COLLECT_ASYNC):
        comm.fold_status()
    return res


def _run(ctx, node, axes, flags, location, out):
    loc = _location_of(node, location)
    if loc == "device":  # upload any host operand (convenience for mixed expressions)
        def visit(n):
            for c in n.children:
                visit(c)
            if n.kind in (F.LEAF, F.GATHER) and n.buf is not None:
                n.buf.ensure_device(ctx)
        visit(node)
    em = L.emit(node, axes, loc)
    if loc == "host":
        st = out if out is not None else Storage.from_host(em.out_dtype, np.empty(em.out_len, dtype=NP_OF[em.out_dtype]))
        if st.n != em.out_len or st.dtype != em.out_dtype:
            raise Panic(F.ERR_SIZE, "output buffer does not match the view")  # src/array.rs:12
        ctx.collect_host(em.expr, st.host.ctypes.data, flags)
        return st
    st = out if out is not None else Storage.device(ctx, em.out_dtype, em.out_len)
    if st.n != em.out_len or st.dtype != em.out_dtype:
        raise Panic(F.ERR_SIZE, "output buffer does not match the view")
    ctx.collect(em.expr, st.dptr, flags)
    return st


# ---- Array (src/array.rs:5-114) ------------------------------------------------------------------------------
class Array(View):
    """Dense row-major `Array<I, T>`; storage in host memory or HBM (a device-resident Box<[T]>)."""

    def __init__(self, I, size, storage, T):
        X.check_type(I)
        self.I, self._size, self.storage, self.T = I, size, storage, T
        n = X.length(I, size)
        for s in L.flatten_value(storage) if isinstance(storage, tuple) else [storage]:
            if s.n != n:  # Array::new_inner, src/array.rs:11-14
                raise Panic(F.ERR_SIZE, f"assertion `left == right` failed\n  left: {s.n}\n right: {n}")

    @staticmethod
    def new(I, size, items, T=None):  # src/array.rs:28-30
        size = X.coerce_size(I, size)
        a = np.asarray(items)
        if T is None:
            if a.dtype == np.dtype(np.int64) and not isinstance(items, np.ndarray):
                T = usize  # Python ints default to usize, like the reference's doctests
            elif a.dtype in _NAME_OF_NP:
                T = _NAME_OF_NP[a.dtype]
            else:
                raise TypeError(f"no device representation for items of dtype {a.dtype}")
        return Array(I, size, Storage.from_host(dtype_of(T), a), T)

    @staticmethod
    def from_device(I, size, dptr, T, ctx=None, keep=None):
        """Wrap device memory owned by someone else (e.g. a torch tensor's data_ptr())."""
        size = X.coerce_size(I, size)
        ctx = ctx or default_context()
        return Array(I, size, Storage.wrap_device(ctx, dtype_of(T), X.length(I, size), dptr, keep), T)

    def to_device(self, ctx=None):
        ctx = ctx or default_context()
        for s in _T_leaves_storage(self.storage):
            s.ensure_device(ctx)
            s.home = "device"
        return self

    def to_raw(self):  # src/array.rs:54
        return self.as_ref()

    def as_ref(self):  # AsRef<[T]>, src/array.rs:65-67: downloads when device-resident
        if isinstance(self.storage, tuple):
            cols = [s.to_numpy() for s in _T_leaves_storage(self.storage)]
            leaves_T = _T_leaves(self.T)
            cols = [c.astype(bool) if t is bool else c for c, t in zip(cols, leaves_T)]
            return [_build_like(self.T, [c[k].item() for c in cols]) for k in range(len(cols[0]))]
        a = self.storage.to_numpy()
        return a.astype(bool) if self.T is bool else a

    def iso(self, J):  # Array::iso, src/array.rs:57-62: no data movement
        return Array(J, X.to_iso_size(self._size, self.I, J), self.storage, self.T)

    def at(self, index):  # src/array.rs:81,86 (host-side probe; downloads one element)
        pos = X.index_positions(self.I, index, self._size)
        lens = [a for t, s in zip(X.type_leaves(self.I), X.size_leaves(self.I, self._size)) for a in X.leaf_lengths(t, s)]
        k = 0
        for p, n in zip(pos, lens):
            k = k * n + p
        vals = []
        for s, t in zip(_T_leaves_storage(self.storage), _T_leaves(self.T)):
            if s.home == "host":
                v = s.host[k]
            else:
                one = np.empty(1, dtype=NP_OF[s.dtype])
                s.ctx.download(one, s.dptr + k * F.DTYPE_SIZE[s.dtype])
                v = one[0]
            vals.append(bool(v) if t is bool else v.item())
        return _build_like(self.T, vals) if isinstance(self.T, tuple) else vals[0]

    __getitem__ = at

    def _lower(self):
        groups = _fresh_groups(self.I, self._size)
        axes = _flat(groups)
        stride, acc = {}, 1
        for a in reversed(axes):  # row-major: Index::to_usize, src/index.rs:109-114
            stride[a] = acc
            acc *= a.length
        stride = {a: s for a, s in stride.items()}

        def leaf(s):
            peers = getattr(s, "peers", None)
            return L.Node(F.LEAF, s.dtype, buf=s, stride=dict(stride), peers=peers, peer_block=getattr(s, "block", 0))
        value = L.map_value(self.storage, leaf) if isinstance(self.storage, tuple) else leaf(self.storage)
        return groups, value


def _T_leaves_storage(storage):
    return L.flatten_value(storage) if isinstance(storage, tuple) else [storage]


# ---- All (src/index.rs:177-186) ---------------------------------------------------------------------------------
class All(View):
    """`I::all(size)`: the view whose element at `index` is `index`."""

    def __init__(self, I, size):
        X.check_type(I)
        self.I, self._size, self.T = I, X.coerce_size(I, size), I

    def _lower(self):
        groups = _fresh_groups(self.I, self._size)
        return groups, _iota_value(self.I, groups)


def all_(I, size):
    return All(I, size)


def _iota_value(I, groups):
    """The index VALUE at each position, shaped like I (tuple of scalar nodes)."""
    it = iter(groups)

    def build(t):
        if isinstance(t, tuple):
            return tuple(build(x) for x in t)
        g = next(it)
        if isinstance(t, (Coated, Option)):
            raise Unsupported(f"All<{t!r}> elements have no device representation")
        stride, acc = {}, 1
        for a in reversed(g):  # a leaf whose group has been re-split: its value is the row-major position
            stride[a] = acc
            acc *= a.length
        if t is Reversed:  # src/int.rs:82-84: position p holds Reversed(size-1-p)
            return L.Node(F.IOTA, F.U64, offset=acc - 1, stride={a: -v for a, v in stride.items()})
        n = L.Node(F.IOTA, F.U64, stride=stride)
        return _cast_node(n, F.U8) if t is bool else n
    return build(I)


# ---- Scalar (src/view.rs:1399-1408) -------------------------------------------------------------------------------
class Scalar(View):
    def __init__(self, value, T=None):
        if T is None:
            T = bool if isinstance(value, bool) else usize if isinstance(value, int) else "f64"
        self.I, self._size, self.T, self.value = (), (), T, value

    def _lower(self):
        return [], L.Node(F.CONST, dtype_of(self.T), imm=self.value)


# ---- Enumerate (src/view.rs:829-838) --------------------------------------------------------------------------------
class Enumerate(View):
    def __init__(self, v):
        self.v, self.I, self._size, self.T = v, v.I, v._size, (v.I, v.T)

    def _lower(self):
        groups, value = self.v._lower()
        return groups, (_iota_value(self.I, groups), value)


# ---- Diagonal (src/view.rs:846-857) -----------------------------------------------------------------------------------
class Diagonal(View):
    def __init__(self, v, zero):
        self.v, self.zero = v, zero
        self.I, self._size, self.T = (v.I, v.I), (v._size, v._size), v.T

    def _lower(self):
        groups, value = self.v._lower()
        twin = [[L.Axis(a.length) for a in g] for g in groups]
        pairs = tuple(zip(_flat(groups), _flat(twin)))
        zeros = L.flatten_value(self.zero) if isinstance(self.T, tuple) else [self.zero]
        zi = iter(zeros)

        def diag(n):
            z = next(zi)
            if not pairs:
                return n
            return L.Node(F.DIAG, n.dtype, children=(n,), pairs=pairs, imm=z)
        return groups + twin, L.map_value(value, diag)


# ---- Map (src/view.rs:880-889) ------------------------------------------------------------------------------------------
class Map(View):
    def __init__(self, v, f):
        self.v, self.f = v, f
        self.I, self._size = v.I, v._size
        if isinstance(v, Rows):
            if not isinstance(f, O.Fold):
                raise Unsupported("the only lowerable map over rows() is ops.Fold(B, init)")
            if isinstance(v.v.T, tuple):
                raise Unsupported("fold over tuple-typed elements")
            self.T = v.v.T
        elif isinstance(f, O.Fold):
            raise TypeError("ops.Fold maps rows(): write v.rows(I, J).map(Fold(B, init))")
        elif isinstance(f, O.UnaryOp):
            self.T = v.T
        elif isinstance(f, O.Cast):
            self.T = f.T
        elif callable(f):
            self.T = self._trace()[1]
        else:
            raise TypeError(f"cannot map {f!r}")

    def _trace(self, value=None):
        if value is None:  # type inference only: trace over placeholder constants
            leaves = [L.Node(F.CONST, dtype_of(t), imm=0) for t in _T_leaves(self.v.T)]
            value = _build_like(self.v.T, leaves) if isinstance(self.v.T, tuple) else leaves[0]
        return _from_syms(self.f(_to_syms(value, self.v.T)))

    def _lower(self):
        if isinstance(self.v, Rows):
            groups_i, groups_j, value = self.v._lower_rows()
            red = tuple(_flat(groups_j))
            if isinstance(self.f.init, View):  # `let mut s = init.at(i)`: the initial value is a view over the rows' index
                init = self.f.init
                if init.I != self.v.I or init._size != self.v._size:
                    raise Panic(F.ERR_SIZE, "Unequal sizes") if init.I == self.v.I else TypeError("Fold: the init view must be indexed like rows()")
                if isinstance(init.T, tuple) or dtype_of(init.T) != value.dtype:
                    raise TypeError("Fold: the init view's element type differs from the rows'")
                gi, vi = init._lower()
                tv, tw = {}, {}
                groups_i = [_unify_group(a, b, tv, tw) for a, b in zip(groups_i, gi)]
                value = _substituter(tv)(value)
                node = L.Node(F.FOLD, value.dtype, op=self.f.B.code, children=(_substituter(tw)(vi), value), imm=0, red_axes=red)
                return groups_i, node
            node = L.Node(F.FOLD, value.dtype, op=self.f.B.code, children=(value,), imm=self.f.init, red_axes=red)
            return groups_i, node
        groups, value = self.v._lower()
        f = self.f
        if isinstance(f, O.UnaryOp):
            if isinstance(self.v.T, tuple):
                raise TypeError(f"{f!r} is not implemented for tuple-typed elements")
            return groups, _unary_node(f, value, self.v.T is bool)
        if isinstance(f, O.Cast):
            return groups, L.map_value(value, lambda n: _cast_node(n, dtype_of(f.T)))
        return groups, self._trace(value)[0]


# ---- Compose (src/view.rs:897-912) and MapAxis (src/view.rs:1140-1170) ---------------------------------------------------
def _index_components(T, value, groups_w):
    """Pair each position axis of the gathered index type with the scalar node that supplies its
    coordinate: -> {Axis: (node_u64, bound)}."""
    comps = L.flatten_value(value)
    leaves = X.type_leaves(T) if T != () else []
    if len(comps) != len(leaves) or len(leaves) != len(groups_w):
        raise TypeError("compose: index view's element type does not match the source's index type")
    table = {}
    for t, node, g in zip(leaves, comps, groups_w):
        if len(g) != 1 or t is Reversed or isinstance(t, Coated):
            raise Unsupported(f"gather through an index component of type {t!r}")
        (a,) = g
        table[a] = (_cast_node(node, F.U64), a.length)
    return table


def _gather(node, table, memo):
    """Rewrite `node` (over the source's axes) so that the coordinates of the axes in `table` come
    from index values: w.at(v.at(i)).  Every Array load becomes a bounds-checked GATHER."""
    key = id(node)
    if key in memo:
        return memo[key]
    k = node.kind
    if k == F.CONST:
        out = node
    elif k in (F.UNARY, F.BINARY) or (k == F.CONCAT and node.pairs[0][0] not in table):
        out = node.clone(children=tuple(_gather(c, table, memo) for c in node.children))
    elif k in (F.LEAF, F.GATHER):
        kids = [_gather(c, table, memo) for c in node.children]
        gstride, bound, stride = list(node.gstride), list(node.bound), {}
        for a, s in node.stride.items():
            if a in table:
                comp, n = table[a]
                kids.append(comp); gstride.append(s); bound.append(n)
            else:
                stride[a] = s
        if not kids:
            out = node
        else:
            out = L.Node(F.GATHER, node.dtype, buf=node.buf, offset=node.offset, stride=stride, children=tuple(kids),
                         gstride=tuple(gstride), bound=tuple(bound), peers=node.peers, peer_block=node.peer_block)
    elif k == F.IOTA:
        hit = [a for a in node.stride if a in table]
        if not hit:
            out = node
        elif len(node.stride) == 1 and node.stride[hit[0]] == 1 and node.offset == 0:
            out = table[hit[0]][0]  # All::at(index) = index: no bounds check (src/index.rs:185)
        else:
            raise Unsupported("compose onto a compound All")
    else:
        raise Unsupported("compose onto a view containing diagonal() or a fold")
    memo[key] = out
    return out


class Compose(View):
    def __init__(self, v, w):
        if not _index_T_matches(v.T, w.I):
            raise TypeError(f"compose: V::T = {v.T!r} is not W::I = {w.I!r}")
        self.v, self.w = v, w
        self.I, self._size, self.T = v.I, v._size, w.T

    def _lower(self):
        groups_v, value_v = self.v._lower()
        groups_w, value_w = self.w._lower()
        table = _index_components(self.w.I, value_v, groups_w)
        memo = {}
        return groups_v, L.map_value(value_w, lambda n: _gather(n, table, memo))


def _index_T_matches(T, I):
    if isinstance(T, tuple) or isinstance(I, tuple):
        return isinstance(T, tuple) and isinstance(I, tuple) and len(T) == len(I) and all(_index_T_matches(t, i) for t, i in zip(T, I))
    return T == I or (T is usize and I is usize)


class MapAxis(View):
    def __init__(self, v, I, w, J):
        if not X.isomorphic(v.I, (I, w.T, J)):
            raise X.IndexError_(f"map_axis: {v.I!r} is not isomorphic to {(I, w.T, J)!r}")
        self.v, self.w, self._I, self._J = v, w, I, J
        si, _st, sj = X.to_iso_size(v._size, v.I, (I, w.T, J))
        self.I, self._size, self.T = (I, w.I, J), (si, w._size, sj), v.T

    def _lower(self):
        groups_v, value_v = self.v._lower()
        gi, gt, gj = _split_groups(groups_v, self._I, self.w.T, self._J)
        groups_w, value_w = self.w._lower()
        table = _index_components(self.w.T, value_w, gt)
        memo = {}
        return gi + groups_w + gj, L.map_value(value_v, lambda n: _gather(n, table, memo))


# ---- Zip (src/view.rs:1178-1198) --------------------------------------------------------------------------------------------
class Zip(View):
    def __init__(self, v, w, B):
        self.v, self.w, self.B = v, w, B
        # type and size now (panics with "Unequal sizes" like Zip::size), axes again at lowering time
        self.I, self._size, _ = _broadcast(v.I, w.I, v._size, w._size, [[] for _ in X.type_leaves(v.I)],
                                           [[] for _ in X.type_leaves(w.I)], {}, {})
        if B is O.Pair:
            self.T = (v.T, w.T)
        else:
            if isinstance(v.T, tuple) or isinstance(w.T, tuple):
                raise TypeError(f"{B!r} is not implemented for tuple-typed elements")
            self.T = v.T

    def _lower(self):
        gv, value_v = self.v._lower()
        gw, value_w = self.w._lower()
        table_v, table_w = {}, {}
        _, _, groups = _broadcast(self.v.I, self.w.I, self.v._size, self.w._size, list(gv), list(gw), table_v, table_w)
        value_v = L.map_value(value_v, _substituter(table_v))
        value_w = L.map_value(value_w, _substituter(table_w))
        if self.B is O.Pair:
            return groups, (value_v, value_w)
        return groups, _binary_node(self.B, value_v, value_w)


def _substituter(table):
    memo = {}
    return lambda n: L.substitute(n, table, memo)


# ---- pure index remappings: no data movement, only axis bookkeeping ---------------------------------------------------------------
class CoatView(View):  # src/view.rs:549-556, 1206-1230
    def __init__(self, v, I):
        self.v, self.I, self._size, self.T = v, Coated(v.I), v._size, v.T
        if I != v.I and I != Coated(v.I):
            raise X.IndexError_("coat::<I>() names the coated form of the view's own index type")

    def _lower(self):
        groups, value = self.v._lower()
        return [_flat(groups)], value


class Iso(View):  # src/view.rs:559-564, 1238-1258
    def __init__(self, v, J):
        X.check_type(J)
        self.v, self.I, self.T = v, J, v.T
        self._size = X.to_iso_size(v._size, v.I, J)

    def _lower(self):
        return self.v._lower()


class Transpose(View):  # src/view.rs:586-592, 1266-1294
    def __init__(self, v, I, Xt, Y, J):
        inner = (I, (Y, Xt), J)
        if not X.isomorphic(inner, v.I):
            raise X.IndexError_(f"transpose: {inner!r} is not isomorphic to {v.I!r}")
        self.v, self._parts, self.T = v, (I, Xt, Y, J), v.T
        si, (sy, sx), sj = X.to_iso_size(v._size, v.I, inner)
        self.I, self._size = (I, (Xt, Y), J), (si, (sx, sy), sj)

    def _lower(self):
        I, Xt, Y, J = self._parts
        groups, value = self.v._lower()
        gi, gy, gx, gj = _split_groups(groups, I, Y, Xt, J)
        return gi + gx + gy + gj, value


def _pin(groups, I, index, size):
    """Substitution that fixes the axes of `groups` (indexed by I) at the positions of `index`.  A leaf whose group
    has been re-split (to_usize / from_usize) is pinned through its LINEAR position, digit by digit."""
    table = {}
    for g, t, x, s in zip(groups, X.type_leaves(I), X.index_leaves(I, index), X.size_leaves(I, size)):
        pos, lens = X.index_positions(t, x, s), X.leaf_lengths(t, s)
        if [a.length for a in g] == lens:
            digits = pos
        else:
            k = 0
            for p_, n in zip(pos, lens):
                k = k * n + p_
            digits = []
            for a in reversed(g):
                digits.append(k % a.length if a.length else 0)
                k = k // a.length if a.length else 0
            digits.reverse()
        for a, d in zip(g, digits):
            table[a] = L.Sub(d)
    return table


class Row(View):  # src/view.rs:609-614, 1302-1322
    def __init__(self, v, I, J, i):
        if not X.isomorphic(v.I, (I, J)):
            raise X.IndexError_(f"row: {v.I!r} is not isomorphic to {(I, J)!r}")
        self.v, self._I, self._i, self.T = v, I, i, v.T
        self._isize, sj = X.to_iso_size(v._size, v.I, (I, J))
        self.I, self._size = J, sj

    def _lower(self):
        groups, value = self.v._lower()
        gi, gj = _split_groups(groups, self._I, self.I)
        return gj, L.map_value(value, _substituter(_pin(gi, self._I, self._i, self._isize)))


class Column(View):  # src/view.rs:639-644, 1350-1370
    def __init__(self, v, I, J, j):
        if not X.isomorphic(v.I, (I, J)):
            raise X.IndexError_(f"column: {v.I!r} is not isomorphic to {(I, J)!r}")
        self.v, self._J, self._j, self.T = v, J, j, v.T
        si, self._jsize = X.to_iso_size(v._size, v.I, (I, J))
        self.I, self._size = I, si

    def _lower(self):
        groups, value = self.v._lower()
        gi, gj = _split_groups(groups, self.I, self._J)
        return gi, L.map_value(value, _substituter(_pin(gj, self._J, self._j, self._jsize)))


class Rows(View):  # src/view.rs:617-622, 1330-1342
    """View of Row views.  On the device its one use is `.map(ops.Fold(B, init))` — the
    reference's spelling of a reduction over the trailing axes J."""

    def __init__(self, v, I, J):
        if not X.isomorphic(v.I, (I, J)):
            raise X.IndexError_(f"rows: {v.I!r} is not isomorphic to {(I, J)!r}")
        self.v, self._J = v, J
        si, _ = X.to_iso_size(v._size, v.I, (I, J))
        self.I, self._size, self.T = I, si, ("Row", v.T)

    def at(self, i):  # src/view.rs:1341
        return Row(self.v, self.I, self._J, i)

    def _lower_rows(self):
        groups, value = self.v._lower()
        gi, gj = _split_groups(groups, self.I, self._J)
        return gi, gj, value

    def _lower(self):
        raise Unsupported("a view of views has no device representation; map it with ops.Fold")


class Columns(View):  # src/view.rs:647-652, 1376-1390
    def __init__(self, v, I, J):
        if not X.isomorphic(v.I, (I, J)):
            raise X.IndexError_(f"columns: {v.I!r} is not isomorphic to {(I, J)!r}")
        self.v, self._I = v, I
        _, sj = X.to_iso_size(v._size, v.I, (I, J))
        self.I, self._size, self.T = J, sj, ("Column", v.T)

    def at(self, j):  # src/view.rs:1389
        return Column(self.v, self._I, self.I, j)

    def _lower(self):
        raise Unsupported("a view of views has no device representation")


class Concat(View):  # src/view.rs:327-339, 920-946
    def __init__(self, v, w, I, J):
        for x in (v, w):
            if not X.isomorphic(x.I, (I, usize, J)):
                raise X.IndexError_(f"concat: {x.I!r} is not isomorphic to {(I, usize, J)!r}")
        if not _same_T(v.T, w.T):
            raise TypeError("concat: element types differ")
        vi, self._nv, vj = X.to_iso_size(v._size, v.I, (I, usize, J))
        wi, nw, wj = X.to_iso_size(w._size, w.I, (I, usize, J))
        if vi != wi:  # assert_eq!(self_i, other_i), :336
            raise Panic(F.ERR_SIZE, f"assertion `left == right` failed\n  left: {vi!r}\n right: {wi!r}")
        if vj != wj:  # assert_eq!(self_j, other_j), :337
            raise Panic(F.ERR_SIZE, f"assertion `left == right` failed\n  left: {vj!r}\n right: {wj!r}")
        self.v, self.w, self._parts, self.T = v, w, (I, J), v.T
        self.I, self._size = (I, usize, J), (vi, self._nv + nw, vj)

    def _lower(self):
        I, J = self._parts
        gv, value_v = self.v._lower()
        gw, value_w = self.w._lower()
        vi, vk, vj = _split_groups(gv, I, usize, J)
        wi, wk, wj = _split_groups(gw, I, usize, J)
        if len(vk[0]) != 1 or len(wk[0]) != 1:
            raise Unsupported("concat along an axis that is a merged group (to_usize) needs device div/mod")
        K = L.Axis(self._size[1])
        table_v, table_w = {}, {}
        gi = [_unify_group(a, b, table_v, table_w) for a, b in zip(vi, wi)]
        gj = [_unify_group(a, b, table_v, table_w) for a, b in zip(vj, wj)]
        table_v[vk[0][0]] = L.Sub(0, ((K, 1),))
        table_w[wk[0][0]] = L.Sub(-self._nv, ((K, 1),))  # W is addressed with k - len(V), :943
        sv, sw = _substituter(table_v), _substituter(table_w)
        lv, lw = L.flatten_value(value_v), L.flatten_value(value_w)
        out = [L.Node(F.CONCAT, a.dtype, children=(sv(a), sw(b)), pairs=((K, self._nv),)) for a, b in zip(lv, lw)]
        value = _build_like(self.T, list(out)) if isinstance(self.T, tuple) else out[0]
        return gi + [[K]] + gj, value


class FromUsize(View):  # src/view.rs:352-363, 993-1021
    def __init__(self, v, I, Xt, J, from_length):
        if not X.isomorphic(v.I, (I, usize, J)):
            raise X.IndexError_(f"from_usize: {v.I!r} is not isomorphic to {(I, usize, J)!r}")
        self.v, self._parts, self.T = v, (I, Xt, J), v.T
        si, old, sj = X.to_iso_size(v._size, v.I, (I, usize, J))
        xsize = from_length(old)
        if X.length(Xt, xsize) != old:  # assert_eq!(X::length(size), old_size), :361
            raise Panic(F.ERR_SIZE, f"assertion `left == right` failed\n  left: {X.length(Xt, xsize)}\n right: {old}")
        self.I, self._size, self._xsize = (I, Xt, J), (si, xsize, sj), xsize

    def _lower(self):
        I, Xt, J = self._parts
        groups, value = self.v._lower()
        gi, gk, gj = _split_groups(groups, I, usize, J)
        # x.to_usize(size) is row-major over X's position axes (:1019); the usize axis may itself be a merged group
        # (a to_usize further down), so both factorisations are rewritten over their common refinement
        old = gk[0]
        lens_x = [n for t, sz in zip(X.type_leaves(Xt), X.size_leaves(Xt, self._xsize)) for n in X.leaf_lengths(t, sz)]
        pieces, map_old, map_x = _refine([a.length for a in old], lens_x)
        axes = [L.Axis(n) for n in pieces]
        table = {a: _sub_of([axes[k] for k in idx]) for a, idx in zip(old, map_old)}
        gx, at = [], 0
        for t, sz in zip(X.type_leaves(Xt), X.size_leaves(Xt, self._xsize)):
            g = []
            for _ in X.leaf_lengths(t, sz):
                g.extend(axes[k] for k in map_x[at])
                at += 1
            gx.append(g)
        value = L.map_value(value, _substituter(table))
        return gi + gx + gj, value


class ToUsize(View):  # src/view.rs:373-378, 1029-1059
    """In position space an axis indexed by X and the usize axis of length X::length are the same
    run of positions; the merged axis is kept as a GROUP of position axes."""

    def __init__(self, v, I, Xt, J):
        if not X.isomorphic(v.I, (I, Xt, J)):
            raise X.IndexError_(f"to_usize: {v.I!r} is not isomorphic to {(I, Xt, J)!r}")
        self.v, self._parts, self.T = v, (I, Xt, J), v.T
        si, sx, sj = X.to_iso_size(v._size, v.I, (I, Xt, J))
        self.I, self._size = (I, usize, J), (si, X.length(Xt, sx), sj)

    def _lower(self):
        I, Xt, J = self._parts
        groups, value = self.v._lower()
        gi, gx, gj = _split_groups(groups, I, Xt, J)
        return gi + [_flat(gx)] + gj, value


class InsertOne(View):  # src/view.rs:391-397, 1067-1096
    def __init__(self, v, I, J, K, size):
        if not X.isomorphic(v.I, (I, K)):
            raise X.IndexError_(f"insert_one: {v.I!r} is not isomorphic to {(I, K)!r}")
        if X.length(J, size) != 1:  # :395
            raise Panic(F.ERR_SIZE, f"assertion `left == right` failed\n  left: {X.length(J, size)}\n right: 1")
        self.v, self._parts, self._jsize, self.T = v, (I, J, K), size, v.T
        si, sk = X.to_iso_size(v._size, v.I, (I, K))
        self.I, self._size = (I, J, K), (si, size, sk)

    def _lower(self):
        I, J, K = self._parts
        groups, value = self.v._lower()
        gi, gk = _split_groups(groups, I, K)
        return gi + _fresh_groups(J, self._jsize) + gk, value


class RemoveOne(View):  # src/view.rs:408-418, 1104-1132
    def __init__(self, v, I, J, K):
        if not X.isomorphic(v.I, (I, J, K)):
            raise X.IndexError_(f"remove_one: {v.I!r} is not isomorphic to {(I, J, K)!r}")
        si, sj, sk = X.to_iso_size(v._size, v.I, (I, J, K))
        if X.length(J, sj) != 1:  # :413
            raise Panic(F.ERR_SIZE, f"assertion `left == right` failed\n  left: {X.length(J, sj)}\n right: 1")
        self.v, self._parts, self.T = v, (I, J, K), v.T
        self.I, self._size = (I, K), (si, sk)

    def _lower(self):
        I, J, K = self._parts
        groups, value = self.v._lower()
        gi, gj, gk = _split_groups(groups, I, J, K)
        table = {a: L.Sub(0) for a in _flat(gj)}
        return gi + gk, L.map_value(value, _substituter(table))


def fold_rows(v, I, J, B, init):
    """`v.rows::<I,J>().map(|row| { let mut s = init; row.each(|x| s = B(s, x)); s })`
    (src/view.rs:617-622, 1341, 250-252): sequential, in index order."""
    return v.rows(I, J).map(O.Fold(B, init))
