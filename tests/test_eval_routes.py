"""Which instantiation of the rank-N evaluator serves which plan, and is it right there.

`k_eval` is not one kernel: it is every line of the four `variants_*.inc` lists (a pre-built signature or the interpreter,
times slot width, vector width V, stack depth, 32/64-bit coordinates and rank bound MAXR), plus the two run-time
specialisations `mdim_jit_kernel[ops]` and `mdim_jit_kernel[ops+shape]`.  Several choices are made at launch, after
`describe()`: the 256-bit stores (output 32-byte aligned), the V=1 re-plan of an output aligned to its element only, and the
JIT level, which depends on how often the process has collected the same shape.

So every case here names
  * the planned route, a prefix of `describe()` plus the instantiation it selects (checked on the CPU),
  * the exact `last_kernel()` under each setting that re-routes it: MDIM_JIT=0 (the pre-built signature or the interpreter),
    MDIM_JIT_SHAPES=0 (the signature or `[ops]`), MDIM_JIT_SHAPES=1 (`[ops+shape]` for every generic, non-wide plan), the
    COLLECT_NO_STATIC flag (the interpreter) and the default (the first collect as under MDIM_JIT_SHAPES=0, the second on
    `[ops+shape]`).  The environment settings are read once per process, so each one runs in a subprocess of its own;
  * a reference computed with numpy from the input arrays: element-type arithmetic (integers wrap through unsigned views,
    nothing is fused), fancy indexing for strides and gathers, and the sequential fold of test_kernel_routes.

The cases are hand-built descriptors (the C ABI the evaluator serves), so that every stride, offset, alignment and
predicate is explicit.  On the CPU the host form of the same instantiation (tests/emu: the library's planner, which selects and
names the instantiation, over a host build of every line of the `.inc` lists) must report the same kernel and, with the C
oracle, equal the reference bit for bit.
"""
import ctypes as C
import functools
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from helpers import oracle_lib, emu_lib, assert_same_bits
import multidimension_b200 as P
from multidimension_b200 import _ffi as F
from multidimension_b200 import lowering as L
from multidimension_b200.runtime import Storage, NP_OF, describe_nodevice
from test_kernel_routes import _apply, rand

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_MAX_ELEMS = 1 << 20
OPS = {F.ADD: P.Add, F.SUB: P.Sub, F.MUL: P.Mul, F.DIV: P.Div}
DT = {"u8": F.U8, "i32": F.I32, "u32": F.U32, "i64": F.I64, "u64": F.U64, "f32": F.F32, "f64": F.F64}
NPD = {F.U8: np.uint8, F.I32: np.int32, F.U32: np.uint32, F.I64: np.int64, F.U64: np.uint64, F.F32: np.float32, F.F64: np.float64}

# settings -> environment; each runs in its own process (the JIT switches and the shape counter are per process)
KNOBS = {"jit=0": {"MDIM_JIT": "0"}, "shapes=0": {"MDIM_JIT_SHAPES": "0"}, "shapes=1": {"MDIM_JIT_SHAPES": "1"}, "default": {}}


# ---- the instantiation registry, as the library builds it -------------------------------------------------------------------
def _emu():
    lib = emu_lib()
    lib.mdim_emu_last_kernel.argtypes = [C.c_char_p, C.c_size_t]
    lib.mdim_emu_variant_name.argtypes = [C.c_int, C.c_char_p, C.c_size_t]
    lib.mdim_emu_find_divisor.argtypes = [C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.mdim_emu_find_divisor.restype = None
    return lib


@functools.lru_cache(maxsize=None)
def registry():
    """Every line of the four variants_*.inc lists, named as last_kernel() names it."""
    lib, out, buf = _emu(), [], C.create_string_buffer(96)
    while lib.mdim_emu_variant_name(len(out), buf, 96) == F.OK:
        out.append(buf.value.decode())
    return tuple(out)


def _parse(name):
    f = name[len("k_eval<"):-1].split(",")
    return {"sig": f[0], "slot": int(f[1][1:]) // 8, "vec": int(f[2][1:]), "depth": int(f[3][1:]), "wide": "wide" in f, "maxr": int(f[-1][1:])}


def instantiation(sig, slot, vec, depth, wide, need):
    """The selection rule, restated independently of the library's select_variant (plan.cpp): the signature's smallest
    MAXR >= need, else the interpreter's smallest MAXR and depth that cover the plan."""
    cands = [(_parse(n), n) for n in registry()]
    if sig and not wide:
        ok = [(p["maxr"], n) for p, n in cands if p["sig"] == sig and p["slot"] == slot and p["vec"] == vec and p["maxr"] >= need]
        if ok:
            return min(ok)[1]
    ok = [(p["maxr"], p["depth"], n) for p, n in cands if p["sig"] == "interp" and p["slot"] == slot and p["vec"] == vec and
          p["wide"] == wide and p["maxr"] >= need and p["depth"] >= depth]
    assert ok, (sig, slot, vec, depth, wide, need)
    return min(ok)[2]


# ---- numpy reference of a descriptor tree -----------------------------------------------------------------------------------
class Ref:
    """Evaluates a node tree over the full grid of output (and reduction) axes with numpy.  Every value comes with a mask of
    the positions where evaluating it panics; Diagonal and Concat only evaluate (and panic in) the side they select."""

    def __init__(self, axes):
        self.axes = list(axes)

    def coords(self, all_axes):
        n = len(all_axes)
        return {a: np.arange(a.length, dtype=np.int64).reshape([-1 if i == k else 1 for i in range(n)]) for k, a in enumerate(all_axes)}

    def lin(self, node, co):
        idx = np.int64(node.offset)
        for a, s in node.stride.items():
            idx = idx + co[a] * np.int64(s)
        return idx

    def ev(self, n, co):
        K, dt = n.kind, NPD[n.dtype]
        if K == F.LEAF:
            i = self.lin(n, co)
            return n.buf.host[i].astype(dt), np.zeros(np.shape(i), bool)
        if K == F.IOTA:
            i = self.lin(n, co).astype(np.uint64)
            return (i & np.uint64(0xff)).astype(dt) if dt == np.uint8 else i.astype(dt), np.zeros(np.shape(i), bool)
        if K == F.CONST:
            return np.array(n.imm, dtype=dt), np.array(False)
        if K == F.UNARY:
            v, e = self.ev(n.children[0], co)
            if n.op == F.CAST:
                return v.astype(dt), e
            assert n.op == F.NEG
            return (-v if dt in (np.float32, np.float64) else (np.uint64(0) - v.astype(np.uint64)).astype(dt)), e
        if K == F.BINARY:
            (a, ea), (b, eb) = self.ev(n.children[0], co), self.ev(n.children[1], co)
            if n.op in (F.DIV, F.REM) and np.dtype(dt).kind == "u":
                zero = b == 0
                with np.errstate(all="ignore"):
                    r = np.where(zero, 0, (a // np.where(zero, 1, b)) if n.op == F.DIV else (a % np.where(zero, 1, b))).astype(dt)
                return r, ea | eb | zero
            return _apply(OPS[n.op], a, b).astype(dt), ea | eb
        if K == F.DIAG:
            v, e = self.ev(n.children[0], co)
            m = np.array(True)
            for pr in n.pairs:
                rhs = pr[1] if isinstance(pr[1], int) else co[pr[1]] + (pr[2] if len(pr) > 2 else 0)
                m = m & (co[pr[0]] == rhs)
            return np.where(m, v, np.array(n.imm, dtype=dt)), e & m
        if K == F.CONCAT:
            (v, ev_), (w, ew) = self.ev(n.children[0], co), self.ev(n.children[1], co)
            m = co[n.pairs[0][0]] < n.pairs[0][1]
            return np.where(m, v, w), np.where(m, ev_, ew)
        if K == F.GATHER:
            i, err = self.lin(n, co), np.array(False)
            for c, g, bd in zip(n.children, n.gstride, n.bound):
                k, e = self.ev(c, co)
                bad = k.astype(np.uint64) >= np.uint64(bd)
                err = err | e | (bad & ~err)
                i = i + np.where(bad, 0, k.astype(np.int64)) * np.int64(g)
            return np.where(err, 0, n.buf.host[np.where(err, 0, i)]).astype(dt), err
        if K == F.FOLD:
            body = n.children[-1]
            red = list(n.red_axes)
            v, e = self.ev(body, co)
            shape = np.broadcast_shapes(*[co[a].shape for a in self.all_axes])
            v, e = np.broadcast_to(v, shape), np.broadcast_to(e, shape)
            nout = len(self.all_axes) - len(red)
            flat_v = v.reshape(shape[:nout] + (-1,))
            if len(n.children) == 2:
                init, ei = self.ev(n.children[0], co)
                init = np.broadcast_to(init, shape[:nout] + (1,) * len(red)).reshape(shape[:nout])
                acc = init.astype(dt).copy()
                ei = np.broadcast_to(ei, shape[:nout] + (1,) * len(red)).reshape(shape[:nout])
            else:
                acc, ei = np.full(shape[:nout], np.array(n.imm, dtype=dt)), np.zeros(shape[:nout], bool)
            for k in range(flat_v.shape[-1]):
                acc = _apply(OPS[n.op], acc, flat_v[..., k]).astype(dt)
            err = ei | e.reshape(shape[:nout] + (-1,)).any(axis=-1)
            return acc.reshape(shape[:nout] + (1,) * len(red)), err.reshape(shape[:nout] + (1,) * len(red))
        raise AssertionError(K)

    def run(self, roots):
        """-> ([flat output per root], flat error mask)."""
        red = []

        def walk(n):
            for c in n.children:
                walk(c)
            if n.kind == F.FOLD:
                red.extend(n.red_axes)
        for r in roots:
            walk(r)
        self.all_axes = self.axes + red
        co = self.coords(self.all_axes)
        out_shape = tuple(a.length for a in self.axes)
        outs, err = [], np.zeros(out_shape, bool)
        for r in roots:
            v, e = self.ev(r, co)
            full = out_shape + (1,) * len(red)
            outs.append(np.broadcast_to(v, full).reshape(out_shape).reshape(-1).copy())
            err = err | np.broadcast_to(e, full).reshape(out_shape)
        return outs, err.reshape(-1)


# ---- one subject: a descriptor, its reference and three executors ----------------------------------------------------------
def _host_out(dtype, n, shift):
    """A zeroed host output of n elements whose first element sits `shift` bytes past a 32-byte boundary."""
    es = np.dtype(NPD[dtype]).itemsize
    raw = np.zeros(n * es + 64, np.uint8)
    k = (-raw.ctypes.data) % 32 + shift
    return raw, raw[k:k + n * es].view(NPD[dtype])


def _status(info):
    return (info.status, info.position, info.node, info.component, info.value, info.bound)


class Subject:
    def __init__(self, roots, axes, shift=0):
        self.roots = roots if isinstance(roots, list) else [roots]
        self.axes, self.shift = axes, shift

    def root(self):
        return self.roots if len(self.roots) > 1 else self.roots[0]

    def describe(self, flags=0):
        st, text = describe_nodevice(L.emit(self.root(), self.axes, "any").expr, flags)
        return text if st == F.OK else f"error {st}: {text}"

    def reference(self):
        return Ref(self.axes).run(self.roots)

    def _host(self, run):
        em = L.emit(self.root(), self.axes, "host")
        keep = [_host_out(dt, em.out_len, self.shift) for dt in em.out_dtypes]
        info = F.ErrorInfo()
        st = run(em, [o for _, o in keep], info)
        return [o.copy() for _, o in keep], (st, _status(info)) if st else None

    def oracle(self):
        lib = oracle_lib()
        lib.mdim_oracle_collect_tuple.restype = C.c_int

        def run(em, outs, info):
            if len(outs) == 1:
                return lib.mdim_oracle_collect(C.byref(em.expr), outs[0].ctypes.data, C.byref(info))
            ptrs = (C.c_void_p * len(outs))(*[o.ctypes.data for o in outs])
            return lib.mdim_oracle_collect_tuple(C.byref(em.expr), ptrs, len(outs), C.byref(info))
        return self._host(run)

    def emu(self, flags=0):
        """-> (outputs, error or None, the instantiation the emu ran)."""
        lib = _emu()
        lib.mdim_emu_collect_tuple.restype = C.c_int

        def run(em, outs, info):
            ptrs = (C.c_void_p * len(outs))(*[o.ctypes.data for o in outs])
            return lib.mdim_emu_collect_tuple(C.byref(em.expr), ptrs, len(outs), C.c_uint32(flags), C.byref(info), None, C.c_size_t(0))
        outs, err = self._host(run)
        buf = C.create_string_buffer(96)
        lib.mdim_emu_last_kernel(buf, 96)
        return outs, err, buf.value.decode()

    def gpu(self, ctx, flags=0):
        """-> (outputs, error or None, last_kernel())."""
        for n in self._leaves():
            n.buf.ensure_device(ctx)
        em = L.emit(self.root(), self.axes, "device")
        outs = []
        for dt in em.out_dtypes:
            es = F.DTYPE_SIZE[dt]
            base = ctx.alloc(em.out_len * es + 64)
            outs.append((base, base + (-base) % 32 + self.shift, dt))
        ptrs = [p for _, p, _ in outs]
        err = None
        try:
            if len(ptrs) == 1:
                ctx.collect(em.expr, ptrs[0], flags)
            else:
                ctx.collect_tuple(em.expr, ptrs, flags)
        except F.MdimError as e:
            err = (e.status, _status(e.info))
        ran = ctx.last_kernel()
        got = []
        for base, p, dt in outs:
            h = np.empty(em.out_len, NPD[dt])
            ctx.download(h, p)
            ctx.free(base)
            got.append(h)
        return got, err, ran

    def _leaves(self):
        seen, out = set(), []

        def walk(n):
            for c in n.children:
                walk(c)
            if n.kind in (F.LEAF, F.GATHER) and id(n.buf) not in seen:
                seen.add(id(n.buf))
                out.append(n)
        for r in self.roots:
            walk(r)
        return out


# ---- building blocks -------------------------------------------------------------------------------------------------------
_BIG = {}


def src(key, T, n, lo=-4.0, hi=4.0):
    """A seeded source Storage, one per key and process (shared by the cases that name it)."""
    if key not in _BIG:
        rng = np.random.default_rng(zlib.crc32(key.encode()))
        _BIG[key] = Storage.from_host(DT[T], rand(rng, T, n, lo, hi))
    return _BIG[key]


def sparse_src(key, T, n, fill):
    """A source of n elements, zero (lazily allocated) except where fill(array) writes."""
    if key not in _BIG:
        a = np.zeros(n, NP_OF[DT[T]] if T != "u8" else np.uint8)
        fill(a)
        _BIG[key] = Storage(DT[T], n, host=a)
    return _BIG[key]


def leaf(T, buf, offset, stride):
    return L.Node(F.LEAF, DT[T], buf=buf, offset=offset, stride={a: s for a, s in stride.items() if s})


def binary(op, a, b):
    return L.Node(F.BINARY, a.dtype, op=op, children=(a, b))


def const(T, v):
    return L.Node(F.CONST, DT[T], imm=v)


def dense(axes, pad=0):
    """Row-major strides over `axes`, each row `pad` elements longer than it needs (pad > 0: no two axes merge)."""
    st, acc = {}, 1
    for a in reversed(axes):
        st[a] = acc
        acc = acc * a.length + pad
    return st, acc


def operand(key, T, axes, pad=0, offset=0, lo=-4.0, hi=4.0):
    st, n = dense(axes, pad)
    return leaf(T, src(key, T, n + offset + 8, lo, hi), offset, st)


def bcast(key, T, axes, keep, pad=0):
    """An operand over `axes` that has only the axes in `keep` (stride 0 on the others)."""
    st, n = dense([a for a in axes if a in keep], pad)
    return leaf(T, src(key, T, n + 8), 0, st)


def deep(T, x, depth, op=F.ADD):
    """x (op) (c1 (op) (c2 ...)): right-nested so that the value stack reaches `depth`."""
    v = x
    for k in range(depth - 1):
        v = binary(op, const(T, 1 + k), v)
    return v


# ---- the case table --------------------------------------------------------------------------------------------------------
class Case:
    """build() -> Subject.  Planned route: kind (stream / generic), sig (the pre-built signature, or None), slot, V, rank+red,
    depth, wide.  launch_vec: the V the launch runs (1 when the output is only element-aligned)."""

    def __init__(self, id, build, sig, slot, vec, rank, red, depth, wide=False, stream=False, launch_vec=None, err=False):
        self.id, self.build, self.sig, self.slot, self.vec = id, build, sig, slot, vec
        self.rank, self.red, self.depth, self.wide, self.stream, self.err = rank, red, depth, wide, stream, err
        self.launch_vec = launch_vec or vec

    def __repr__(self):
        return self.id

    @property
    def route(self):
        return (f"{'stream' if self.stream else 'generic'}.{'static' if self.sig else 'interp'} s{self.slot * 8} v{self.vec}x1"
                f"{' wide' if self.wide else ''} rank={self.rank}+{self.red} depth={self.depth} ")

    @property
    def planned(self):
        """What describe() shows in brackets: the instantiation select_variant picks for the plan (before any launch re-plan)."""
        p = _parse(instantiation(self.sig, self.slot, self.vec, self.depth, self.wide, self.need))
        return f"[{'NoSig' if p['sig'] == 'interp' else p['sig']} r{p['maxr']}"

    @property
    def need(self):
        return 1 if self.stream else self.rank + self.red

    def kernel(self, knob):
        # the V=1 re-plan of an element-aligned output keeps the op sequence: a signature with a V=1 instantiation still serves it
        static = instantiation(self.sig, self.slot, self.launch_vec, self.depth, self.wide, self.need)
        interp = instantiation(None, self.slot, self.launch_vec, self.depth, self.wide, self.need)
        pre = static if "interp" not in static else None
        if knob in ("jit=0", "no_static"):
            return interp if knob == "no_static" else static
        first = pre or "mdim_jit_kernel[ops]"
        shaped = "mdim_jit_kernel[ops+shape]" if not self.stream and not self.wide else first
        return {"shapes=0": first, "shapes=1": shaped, "default": first, "default#2": shaped}[knob]


CASES = []


def case(id, sig, slot, vec, rank, red, depth, **kw):
    def deco(build):
        CASES.append(Case(id, build, sig, slot, vec, rank, red, depth, **kw))
        return build
    return deco


def axes(*lens):
    return [L.Axis(n) for n in lens]


def add_static_s32():
    two = {"SigAddF32": F.ADD, "SigSubF32": F.SUB, "SigMulF32": F.MUL, "SigDivF32": F.DIV}
    cst = {"SigAddCF32": F.ADD, "SigSubCF32": F.SUB, "SigMulCF32": F.MUL, "SigDivCF32": F.DIV}
    # MAXR 1 (a stream), 2, 3, 5 (rank 4: one padding axis; rank 5 on the MulAdd form)
    shapes = {1: (24,), 2: (5, 16), 3: (3, 7, 8), 5: (2, 3, 5, 8)}
    for sig in ["SigCopyF32"] + list(two) + list(cst) + ["SigMulAddCF32"]:
        for r, shp in shapes.items():
            if sig == "SigMulAddCF32" and r == 5:
                shp = (2, 2, 3, 5, 8)

            def build(sig=sig, shp=shp, r=r):
                ax = axes(*shp)
                pad = 8 if r > 1 else 0
                a = operand(f"a32-{len(shp)}", "f32", ax, pad)
                b = operand(f"b32-{len(shp)}", "f32", ax, pad, lo=0.5, hi=4.0)
                if sig == "SigCopyF32":
                    v = a
                elif sig in two:
                    v = binary(two[sig], a, b)
                elif sig in cst:
                    v = binary(cst[sig], a, const("f32", 1.5))
                else:
                    v = binary(F.ADD, binary(F.MUL, a, b), const("f32", 1.0))
                return Subject(v, ax)
            case(f"{sig}-r{r}-{'x'.join(map(str, shp))}", sig, 4, 8, len(shp), 0, 1 if sig == "SigCopyF32" else 2 if sig != "SigMulAddCF32" else 2,
                 stream=r == 1)(build)


def add_bcast_s32():
    ops = {"Add": F.ADD, "Sub": F.SUB, "Mul": F.MUL, "Div": F.DIV}
    shapes = {2: (5, 16), 3: (3, 7, 8), 5: (2, 3, 5, 8)}
    for r, shp in shapes.items():
        for name, op in ops.items():
            def build(op=op, shp=shp):  # x (op) b[row]: b has no vector axis (LEAF_BCAST)
                ax = axes(*shp)
                return Subject(binary(op, operand(f"a32-{len(shp)}", "f32", ax, 8), bcast(f"r32-{len(shp)}", "f32", ax, ax[:-1])), ax)
            case(f"Sig{name}BcastF32-r{r}", f"Sig{name}BcastF32", 4, 8, len(shp), 0, 2)(build)
            if name != "Div":
                def build(op=op, shp=shp):  # x (op) w[col]: a row vector re-read over the outer axes (LEAF_VEC aux 1)
                    ax = axes(*shp)
                    return Subject(binary(op, operand(f"a32-{len(shp)}", "f32", ax, 8), bcast(f"w32-{len(shp)}", "f32", ax, ax[-1:])), ax)
                case(f"Sig{name}VecBcastF32-r{r}", f"Sig{name}VecBcastF32", 4, 8, len(shp), 0, 2)(build)

        def build(shp=shp):  # x - b[row] / 256
            ax = axes(*shp)
            return Subject(binary(F.SUB, operand(f"a32-{len(shp)}", "f32", ax, 8),
                                  binary(F.DIV, bcast(f"r32-{len(shp)}", "f32", ax, ax[:-1]), const("f32", 256.0))), ax)
        case(f"SigSubBcastDivF32-r{r}", "SigSubBcastDivF32", 4, 8, len(shp), 0, 3)(build)

        def build(shp=shp, lane=False):  # diagonal(0) of b[row] along (row, col): the vector axis is in the predicate
            ax = axes(*shp)
            d = L.Node(F.DIAG, F.F32, children=(bcast(f"r32-{len(shp)}", "f32", ax, ax[:-1], 1),), pairs=((ax[-2], ax[-1], 1),), imm=0.0)
            return Subject(d, ax)
        case(f"SigDiagF32-r{r}-lane", "SigDiagF32", 4, 8, len(shp), 0, 1)(build)

        def build(shp=shp):  # config-5 form: diagonal(0) of b[row] (predicate without the vector axis) * w[col] + 1
            ax = axes(*shp)
            d = L.Node(F.DIAG, F.F32, children=(bcast(f"r32-{len(shp)}", "f32", ax, ax[:-1]),), pairs=((ax[0], ax[-2]),), imm=0.0)
            return Subject(binary(F.ADD, binary(F.MUL, d, bcast(f"w32-{len(shp)}", "f32", ax, ax[-1:])), const("f32", 1.0)), ax)
        case(f"SigDiagMulAddCF32-r{r}", "SigDiagMulAddCF32", 4, 8, len(shp), 0, 2)(build)


def fold(T, op, body, red, init=0.0, init_view=None):
    return L.Node(F.FOLD, DT[T], op=op, children=(body,) if init_view is None else (init_view, body), red_axes=tuple(red), imm=init)


def add_fold_s32():
    # V8 needs >= 320000 outputs (a fold prefers narrower vectors below 40000 threads), V4 >= 160000
    # MAXR 2: a reversed reduction axis (so k_fold_cols, which needs a forward pitch, does not take it)
    for sig, op, strided in (("SigFoldAddVecF32", F.ADD, False), ("SigFoldMulVecF32", F.MUL, False), ("SigFoldAddStridedF32", F.ADD, True)):
        lo, hi = (0.9, 1.1) if op == F.MUL else (-4.0, 4.0)
        es = 2 if strided else 1

        def b2(op=op, es=es, lo=lo, hi=hi, n=320000, R=3):
            o, r = axes(n, R)
            s = src(f"fold2-{es}", "f32", n * R * es + 8, lo, hi)
            return Subject(fold("f32", op, leaf("f32", s, (R - 1) * n * es, {o: es, r: -n * es}), [r], 0.5), [o])
        case(f"{sig}-r2-reversed", sig, 4, 8, 1, 1, 2)(b2)

        def b3(op=op, es=es, lo=lo, hi=hi, n=320000):  # two reduction axes: the carry moves the slower one
            o, r1, r2 = axes(n, 2, 3)
            s = src(f"fold3-{es}", "f32", n * 8 * es + 8, lo, hi)
            return Subject(fold("f32", op, leaf("f32", s, 0, {o: es, r1: 4 * n * es, r2: n * es}), [r1, r2], 0.5), [o])
        case(f"{sig}-r3-two-red", sig, 4, 8, 1, 2, 2)(b3)

        def b5(op=op, es=es, lo=lo, hi=hi):  # rank 3 + 2 reduction axes
            o0, o1, o2, r1, r2 = axes(5, 8, 8008, 2, 3)
            n = 5 * 8 * 8008
            s = src(f"fold5-{es}", "f32", n * 8 * es + 8 * 64, lo, hi)
            return Subject(fold("f32", op, leaf("f32", s, 0, {o0: (8 * 8016 + 8) * es, o1: 8016 * es, o2: es, r1: 4 * n * es, r2: n * es}), [r1, r2], 0.5), [o0, o1, o2])
        case(f"{sig}-r5", sig, 4, 8, 3, 2, 2)(b5)

        def b3v4(op=op, es=es, lo=lo, hi=hi, n=200004):  # 8k + 4 outputs, fewer than 320000: V4
            o, r1, r2 = axes(n, 2, 2)
            s = src(f"fold3v4-{es}", "f32", (n * 4 + 32) * es + 8, lo, hi)
            return Subject(fold("f32", op, leaf("f32", s, 0, {o: es, r1: (2 * n + 8) * es, r2: n * es}), [r1, r2], 0.5), [o])
        case(f"{sig}-r3-v4", sig, 4, 4, 1, 2, 2)(b3v4)

        def b3v1(op=op, es=es, lo=lo, hi=hi, n=37):  # few outputs: V1; k = 0 .. red_fast_len over a prime length
            o, r1, r2 = axes(n, 3, 11)
            s = src(f"fold3v1-{es}", "f32", (n * 33 + 32) * es + 8, lo, hi)
            return Subject(fold("f32", op, leaf("f32", s, 0, {o: es, r1: (11 * n + 8) * es, r2: n * es}), [r1, r2], 0.5), [o])
        case(f"{sig}-r3-v1", sig, 4, 1, 1, 2, 2)(b3v1)


def add_static_s64():
    shapes = {1: (12,), 2: (5, 12), 3: (3, 7, 4)}
    sigs = ["SigCopyU64", "SigIotaU64", "SigGatherF32", "SigGatherU64", "SigCopyF64", "SigAddF64", "SigMulF64", "SigAddU64"]
    for sig in sigs:
        for r, shp in shapes.items():
            def build(sig=sig, shp=shp, r=r):
                ax = axes(*shp)
                pad = 4 if r > 1 else 0
                if sig in ("SigCopyU64", "SigAddU64"):
                    a = operand(f"u64-{len(shp)}", "u64", ax, pad)
                    v = a if sig == "SigCopyU64" else binary(F.ADD, a, operand(f"u64b-{len(shp)}", "u64", ax, pad))
                elif sig in ("SigCopyF64", "SigAddF64", "SigMulF64"):
                    a = operand(f"f64-{len(shp)}", "f64", ax, pad)
                    v = a if sig == "SigCopyF64" else binary(F.ADD if sig == "SigAddF64" else F.MUL, a, operand(f"f64b-{len(shp)}", "f64", ax, pad))
                elif sig == "SigIotaU64":  # IOTA over axes that do not merge: only a hand-built descriptor has it
                    st, _ = dense(ax, 3 if r > 1 else 0)
                    v = L.Node(F.IOTA, F.U64, offset=5, stride=st)
                else:
                    T = "f32" if sig == "SigGatherF32" else "u64"
                    st, n = dense(ax, pad)
                    idx = sparse_src(f"idx-{len(shp)}", "u64", n + 8, lambda a: a.__setitem__(slice(None), np.random.default_rng(n).integers(0, 1000, a.size)))
                    v = L.Node(F.GATHER, DT[T], buf=src(f"g{T}", T, 1000), children=(leaf("u64", idx, 0, st),), gstride=(1,), bound=(1000,))
                return Subject(v, ax)
            depth = 2 if sig in ("SigAddF64", "SigMulF64", "SigAddU64") else 1
            case(f"{sig}-r{r}", sig, 8, 4, len(shp), 0, depth, stream=r == 1)(build)


def add_interp():
    """Op trees without a pre-built signature, at every V / depth / MAXR of the interpreter (32-bit coordinates)."""
    for slot, T, vecs in ((4, "f32", (8, 4, 1)), (8, "f64", (4, 2, 1))):
        for V in vecs:
            inner = {8: 16, 4: 12, 2: 6, 1: 7}[V] if slot == 4 else {4: 8, 2: 6, 1: 7}[V]
            for r, shp in ((3, (3, 5, inner)), (8, (2, 3, 2, 3, 2, 3, 2, inner))):
                for depth in ((2, 6) if V == 1 else (2,)):
                    def build(shp=shp, depth=depth, T=T):  # (a * b) - c, nested to `depth`
                        ax = axes(*shp)
                        v = binary(F.SUB, binary(F.MUL, operand(f"ia-{T}-{len(shp)}", T, ax, 8), operand(f"ib-{T}-{len(shp)}", T, ax, 8)),
                                   operand(f"ic-{T}-{len(shp)}", T, ax, 8))
                        return Subject(deep(T, v, depth - 1) if depth > 2 else v, ax)
                    case(f"interp-s{slot * 8}-v{V}-d{depth}-r{r}", None, slot, V, len(shp), 0, depth)(build)
    # 7 output axes + 1 reduction axis; a fold with an init view, Sub (order-sensitive), integers that wrap
    def build():
        ax, (r,) = axes(2, 3, 2, 3, 2, 3, 5), axes(4)
        st, n = dense(ax + [r], 1)
        body = leaf("i32", src("fold8", "i32", n + 8), 0, st)
        return Subject(fold("i32", F.SUB, body, [r], init_view=bcast("fold8i", "i32", ax, ax[-1:])), ax)
    case("interp-fold-7+1-init-view-i32-sub", None, 4, 1, 7, 1, 2)(build)

    def build():  # f32 Div fold over a strided axis, 2 reduction axes, 8k outputs -> V1 (few outputs)
        o, r1, r2 = axes(16, 3, 5)
        s = src("fdiv", "f32", 16 * 16 * 2 + 8, 0.5, 2.0)
        return Subject(fold("f32", F.DIV, leaf("f32", s, 0, {o: 2 * 16, r1: 2 * 5 + 1, r2: 2}), [r1, r2], 1e6), [o])
    case("interp-fold-div-strided-2red", None, 4, 1, 1, 2, 2)(build)

    def build():  # a fold over an empty axis gives init, on the signature and on the interpreter
        o, r = axes(16, 0)
        return Subject(fold("f32", F.ADD, leaf("f32", src("a32-1", "f32", 40), 0, {o: 1, r: 16}), [r], 2.5), [o])
    case("fold-empty-axis", "SigFoldAddVecF32", 4, 1, 1, 1, 2)(build)


def add_edges():
    # V per innermost length: s32 8k -> v8, 8k+4 -> v4, odd -> v1; s64 4k, 4k+2, odd; non-power-of-two decode lengths
    for slot, T, lens in ((4, "f32", ((8 * 7, 8), (8 * 7 + 4, 4), (65537, 1))), (8, "f64", ((4 * 9, 4), (4 * 9 + 2, 2), (13, 1)))):
        for inner, V in lens:
            for outer in ((3, 5) if inner != 65537 else (3,)):
                def build(inner=inner, outer=outer, T=T):
                    ax = axes(outer, 7, inner)
                    return Subject(binary(F.SUB, binary(F.MUL, operand(f"e-{T}-{outer}x{inner}", T, ax, 8), operand(f"e2-{T}-{outer}x{inner}", T, ax, 8)), const(T, 0.25)), ax)
                case(f"vec-s{slot * 8}-{outer}x7x{inner}", None, slot, V, 3, 0, 2)(build)
    # output at +16 bytes (no 256-bit store) and at +4 bytes (re-planned to V=1, shown in the kernel name)
    for shift in (16, 4):
        def build(shift=shift):
            ax = axes(5, 16)
            return Subject(binary(F.ADD, operand("a32-2", "f32", ax, 8), operand("b32-2", "f32", ax, 8)), ax, shift=shift)
        case(f"SigAddF32-out+{shift}", "SigAddF32", 4, 8, 2, 0, 2, launch_vec=1 if shift % 16 else 8)(build)

        def build(shift=shift):  # a fold re-planned to V1 keeps its signature (the V1 instantiation)
            o, r = axes(320000, 3)
            s = src("fold2-1", "f32", 320000 * 3 + 8)
            return Subject(fold("f32", F.ADD, leaf("f32", s, 2 * 320000, {o: 1, r: -320000}), [r], 0.5), [o], shift=shift)
        case(f"SigFoldAddVecF32-out+{shift}", "SigFoldAddVecF32", 4, 8, 1, 1, 2, launch_vec=1 if shift % 16 else 8)(build)
    # operands 16- but not 32-byte aligned (no 256-bit loads), element-aligned only (LEAF_STRIDED: no signature)
    def build():
        ax = axes(5, 16)
        return Subject(binary(F.MUL, operand("a32-2", "f32", ax, 8, offset=4), operand("b32-2", "f32", ax, 8, offset=12)), ax)
    case("SigMulF32-operands+16", "SigMulF32", 4, 8, 2, 0, 2)(build)

    def build():
        ax = axes(5, 16)
        return Subject(binary(F.MUL, operand("a32-2", "f32", ax, 8, offset=1), operand("b32-2", "f32", ax, 8)), ax)
    case("interp-operand-element-aligned", None, 4, 8, 2, 0, 2)(build)

    def build():  # a reversed output axis
        o, c = axes(5, 16)
        s = src("a32-2", "f32", 5 * 24 + 8)
        return Subject(binary(F.ADD, leaf("f32", s, 4 * 24, {o: -24, c: 1}), const("f32", 3.0)), [o, c])
    case("SigAddCF32-reversed-axis", "SigAddCF32", 4, 8, 2, 0, 2)(build)

    # a Concat boundary inside a vector (partial lane mask), with an out-of-range gather on the side not selected
    for thr in (5, 13):
        def build(thr=thr):
            o, c = axes(3, 24)
            idx = sparse_src("cidx", "u64", 3 * 24, lambda a: a.__setitem__(slice(None), np.where(np.arange(a.size) % 24 < 13, 10 ** 6, np.arange(a.size) % 97)))
            g = L.Node(F.GATHER, F.F32, buf=src("gf32", "f32", 1000), children=(leaf("u64", idx, 0, {o: 24, c: 1}),), gstride=(1,), bound=(1000,))
            v = L.Node(F.CONCAT, F.F32, children=(operand("a32-2c", "f32", [o, c]), g if thr == 13 else operand("b32-2c", "f32", [o, c])), pairs=((c, thr),))
            return Subject(v, [o, c])
        case(f"concat-in-vector-{thr}", None, 8 if thr == 13 else 4, 4 if thr == 13 else 8, 2, 0, 2)(build)
    # gather of 1..3 components
    for nc in (1, 2, 3):
        def build(nc=nc):
            o, c = axes(4, 12)
            kids = tuple(leaf("u64", src(f"gi{k}", "u64", 4 * 12 + 8, 0, 0), 0, {o: 12, c: 1}) for k in range(nc))
            for k, kid in enumerate(kids):
                kid.buf.host[:] = np.random.default_rng(k).integers(0, 6, kid.buf.n)
            bounds = (6,) * nc
            gs = tuple(6 ** (nc - 1 - k) for k in range(nc))
            return Subject(L.Node(F.GATHER, F.F32, buf=src("gf32", "f32", 1000), children=kids, gstride=gs, bound=bounds), [o, c])
        case(f"gather-{nc}", "SigGatherF32" if nc == 1 else None, 8, 4, 1, 0, nc, stream=True)(build)
    # a tuple root: runs of f32 and u64 (slot 8), 16- but not 32-byte aligned
    for k in (2, 3, 4):
        def build(k=k):
            o, c = axes(3, 8)
            kids = [operand("tf", "f32", [o, c]), operand("tu", "u64", [o, c]), binary(F.ADD, operand("tf", "f32", [o, c]), const("f32", 1.0)),
                    L.Node(F.IOTA, F.U64, offset=0, stride={o: 8, c: 1})][:k]
            return Subject(kids, [o, c], shift=16)
        case(f"tuple-{k}", None, 8, 4, 1, 0, min(2 * k - 2, 4), stream=True)(build)


BIG_GATHER = (1 << 28) + (1 << 12)  # f32 elements: just over 1 GiB (PF_GATHER_BIG)
WIDE_N = (1 << 31) + (1 << 20)      # u8 elements: past 2^31, so coordinates and offsets are 64-bit
WIDE_ROW = (1 << 31) + 4096         # where the wide cases read


def add_big():
    def build():
        n = 4096
        rng = np.random.default_rng(7)
        ix = rng.integers(0, BIG_GATHER, n).astype(np.uint64)
        ix[:3] = (0, BIG_GATHER - 1, BIG_GATHER - 2)

        def fill(a):
            i = ix.astype(np.int64)
            a[np.where(i == BIG_GATHER - 1, i - 1, i + 1)] = 7.0  # each element's neighbour differs from it ...
            a[i] = np.random.default_rng(8).uniform(-4, 4, n).astype(np.float32)
        s = sparse_src("biggather", "f32", BIG_GATHER, fill)
        o, = axes(n)
        return Subject(L.Node(F.GATHER, F.F32, buf=s, children=(leaf("u64", Storage.from_host(F.U64, ix), 0, {o: 1}),), gstride=(1,), bound=(BIG_GATHER,)), [o])
    case("gather-big", "SigGatherF32", 8, 4, 1, 0, 1, stream=True)(build)

    def wide_src():
        return sparse_src("wide", "u8", WIDE_N, lambda a: a.__setitem__(slice(WIDE_ROW, WIDE_ROW + 65536), np.random.default_rng(9).integers(0, 256, 65536, dtype=np.uint8)))

    for slot, vecs in ((4, (8, 4, 1)), (8, (4, 2, 1))):
        for V in vecs:
            inner = {8: 16, 4: 12 if slot == 4 else 8, 2: 6, 1: 7}[V]
            for r, shp in ((3, (3, inner)), (8, (2, 2, 2, 2, 2, inner))):
                for depth in ((2, 6) if V == 1 else (2,)):
                    def build(shp=shp, slot=slot, depth=depth):
                        ax = axes(*shp)
                        st, n = dense(ax, 2)
                        x = leaf("u8", wide_src(), WIDE_ROW, st)
                        y = leaf("u8", wide_src(), WIDE_ROW + 3 * n, st)
                        T = "u32" if slot == 4 else "u64"
                        x = L.Node(F.UNARY, DT[T], op=F.CAST, src_dtype=F.U8, children=(x,))
                        y = L.Node(F.UNARY, DT[T], op=F.CAST, src_dtype=F.U8, children=(y,))
                        v = binary(F.SUB, binary(F.MUL, x, y), const(T, 3))
                        return Subject(deep(T, v, depth - 1, F.MUL) if depth > 2 else v, ax)
                    case(f"wide-s{slot * 8}-v{V}-d{depth}-r{r}", None, slot, V, len(shp), 0, depth, wide=True)(build)


def add_errors():
    # integer /0 and an out-of-bounds gather: the lowest failing position and its details, on every route
    def build():
        o, c = axes(6, 16)
        d = src("den", "u32", 6 * 16 + 8, 0, 0)
        d.host[:] = 3
        d.host[[37, 38, 70]] = 0
        return Subject(binary(F.DIV, operand("num", "u32", [o, c]), leaf("u32", d, 0, {o: 16, c: 1})), [o, c])
    case("error-div0-u32", None, 4, 8, 1, 0, 2, stream=True, err=True)(build)

    def build():
        o, c = axes(6, 16)
        ix = src("oobix", "u64", 6 * 16 + 8, 0, 0)
        ix.host[:] = np.arange(ix.n) % 50
        ix.host[[45, 46, 90]] = (1000, 5000, 1001)
        return Subject(L.Node(F.GATHER, F.F32, buf=src("gf32", "f32", 1000), children=(leaf("u64", ix, 0, {o: 16, c: 1}),), gstride=(1,), bound=(1000,)), [o, c])
    case("error-gather-oob", "SigGatherF32", 8, 4, 1, 0, 1, stream=True, err=True)(build)

    # the same on rank-2 plans (rows padded so that the axes do not merge), which also run on [ops+shape]
    def build():
        o, c = axes(6, 16)
        d = src("den2", "u32", 6 * 24 + 8, 0, 0)
        d.host[:] = 3
        d.host[[2 * 24 + 5, 2 * 24 + 6, 4 * 24 + 6]] = 0  # outputs 37, 38 and 70
        return Subject(binary(F.DIV, operand("num2", "u32", [o, c], 8), leaf("u32", d, 0, {o: 24, c: 1})), [o, c])
    case("error-div0-u32-rank2", None, 4, 8, 2, 0, 2, err=True)(build)

    def oob_index():
        ix = src("oobix2", "u64", 6 * 20 + 8, 0, 0)
        ix.host[:] = np.arange(ix.n) % 50
        ix.host[[2 * 20 + 13, 2 * 20 + 14, 5 * 20 + 10]] = (1000, 5000, 1001)  # outputs 45, 46 and 90
        return ix

    def build(plus=False):
        o, c = axes(6, 16)
        g = L.Node(F.GATHER, F.F32, buf=src("gf32", "f32", 1000), children=(leaf("u64", oob_index(), 0, {o: 20, c: 1}),), gstride=(1,), bound=(1000,))
        return Subject(binary(F.ADD, g, const("f32", 1.5)) if plus else g, [o, c])
    case("error-gather-oob-rank2", "SigGatherF32", 8, 4, 2, 0, 1, err=True)(build)
    case("error-gather-oob-rank2-plus", None, 8, 4, 2, 0, 2, err=True)(lambda: build(True))


add_static_s32()
add_bcast_s32()
add_fold_s32()
add_static_s64()
add_interp()
add_edges()
add_big()
add_errors()
CASE_IDS = [c.id for c in CASES]
assert len(set(CASE_IDS)) == len(CASE_IDS), "case ids must be unique"
HEAVY = {c.id for c in CASES if c.id.startswith(("wide-", "gather-big"))}


# ---- CPU half ----------------------------------------------------------------------------------------------------------------
def check_outputs(case, got, err, want, werr, what):
    if werr.any():
        assert err is not None, f"{what}: expected an error at {int(np.flatnonzero(werr)[0])}"
        assert err[1][1] == int(np.flatnonzero(werr)[0]), f"{what}: error at {err[1][1]}, expected the lowest {int(np.flatnonzero(werr)[0])}"
        return
    assert err is None, f"{what}: {err}"
    for g, w in zip(got, want):
        assert_same_bits(g, w, what)


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_planned_route_and_reference(case):
    """describe() names the planned route and instantiation; the emu runs the same instantiation by the library's rules, and
    the reference equals the emu and the C oracle bit for bit."""
    s = case.build()
    d = s.describe()
    assert d.startswith(case.route), d
    assert case.planned + "]" in d or case.planned + "," in d, (case.planned, d)
    want, werr = s.reference()
    emu_status = []
    for flags, knob in ((0, "jit=0"), (F.COLLECT_NO_STATIC, "no_static")):
        got, err, ran = s.emu(flags)
        assert ran == case.kernel(knob), f"{case.id} [emu {knob}]: ran {ran}, expected {case.kernel(knob)}"
        check_outputs(case, got, err, want, werr, f"{case.id} [emu {knob}] on {ran}")
        emu_status.append(err)
    assert emu_status[0] == emu_status[1], emu_status
    n_in = sum(n.buf.n for n in s._leaves())
    if n_in <= ORACLE_MAX_ELEMS or case.id in HEAVY:
        got, err = s.oracle()
        check_outputs(case, got, err, want, werr, f"{case.id} (oracle)")
        if err:
            assert err == emu_status[0], (err, emu_status[0])


def test_every_instantiation_is_named():
    """Every line of the four variants_*.inc lists is the kernel of some case under MDIM_JIT=0 or COLLECT_NO_STATIC."""
    named = {c.kernel(k) for c in CASES for k in ("jit=0", "no_static")}
    missing = [n for n in registry() if n not in named]
    assert not missing, missing
    assert len(registry()) == 141


def test_find_divisor():
    """q = umulhi(n, mul) >> shr is n / d for every numerator the 32-bit decode can meet (n < 2^31)."""
    lib = _emu()
    def is_prime(x):
        return x > 1 and all(x % p for p in range(2, int(x ** 0.5) + 1))

    def prime_near(x, step):
        while not is_prime(x):
            x += step
        return x
    ds = list(range(1, 65537))
    for k in range(2, 32):  # 2^k and its neighbours, and the nearest prime below and above it (2^31 - 1: the largest divisor)
        ds += [(1 << k) - 1, prime_near((1 << k) - 1, -1)]
        if k < 31:
            ds += [1 << k, (1 << k) + 1, prime_near((1 << k) + 1, 1)]
    assert 2 ** 31 - 1 in ds and 65537 in ds
    rng = np.random.default_rng(3)
    mul, shr = C.c_uint32(), C.c_uint32()
    muls, shrs = np.empty(len(ds), np.uint64), np.empty(len(ds), np.uint64)
    for i, d in enumerate(ds):
        lib.mdim_emu_find_divisor(d, C.byref(mul), C.byref(shr))
        muls[i], shrs[i] = mul.value, shr.value
    d = np.array(ds, np.uint64)
    top = np.uint64(2 ** 31 - 1)
    cols = [np.zeros_like(d), d - 1, d, np.minimum(d * np.uint64(7) - 1, top), np.full_like(d, top)]
    cols += [rng.integers(0, 2 ** 31, d.size).astype(np.uint64) for _ in range(8)]
    for n in cols:
        n = np.minimum(n, top)
        q = np.where(muls == 0, n, ((n * muls) >> np.uint64(32)) >> shrs)
        bad = np.flatnonzero(q != n // d)
        assert bad.size == 0, f"d={d[bad[0]]} n={n[bad[0]]}: {q[bad[0]]} != {n[bad[0]] // d[bad[0]]}"


# ---- GPU half ----------------------------------------------------------------------------------------------------------------
def run_case(case, ctx, knob, flags=0, want=None, seen=None):
    """seen: the (route, lengths) of the cases collected before in this process.  Two cases may share an op sequence and a
    shape (offsets and pointers are not part of it), so a repeat may already have reached the shape-specialised kernel."""
    s = case.build()
    if want is None:
        want = s.reference()
    got, err, ran = s.gpu(ctx, flags)
    expect = {case.kernel(knob)}
    if seen is not None:
        key = (s.describe(), tuple(a.length for a in s.axes))
        if key in seen:
            expect.add(case.kernel("default#2"))
        seen.add(key)
    assert ran in expect, f"{case.id} [{knob}]: ran {ran}, expected {expect} ({s.describe()})"
    check_outputs(case, got, err, want[0], want[1], f"{case.id} [{knob}] on {ran}")
    return err


def run_knob(knob):
    """Every case under the setting already in this process's environment; the default setting collects each case twice."""
    ctx = P.Context(0)
    n, seen = 0, set()
    for case in CASES:
        want = case.build().reference()
        err = run_case(case, ctx, knob, want=want, seen=seen if knob == "default" else None)
        if knob == "default":
            assert run_case(case, ctx, "default#2", want=want) == err, case.id
        n += 1
    ctx.close()
    return n


ERROR_CASES = [c for c in CASES if c.err]
AFTER_ERROR = "SigCopyF32-r1-24"  # a stream: the same kernel on the first and every later collect


def run_errors(knob):
    """Each error case alone in this process (so the shape counter starts at zero), under `knob`; the default setting collects
    it twice.  -> {case id: [[kernel, status, position, node, component, value, bound], ...]}.  After every failed collect an
    ordinary case must still run and be right on the same context."""
    flags = F.COLLECT_NO_STATIC if knob == "no_static" else 0
    after = next(c for c in CASES if c.id == AFTER_ERROR)
    ctx = P.Context(0)
    out = {}
    for case in ERROR_CASES:
        want = case.build().reference()
        out[case.id] = []
        for k in [knob] + (["default#2"] if knob == "default" else []):
            got, err, ran = case.build().gpu(ctx, flags)
            assert ran == case.kernel(k), f"{case.id} [{k}]: ran {ran}, expected {case.kernel(k)}"
            check_outputs(case, got, err, want[0], want[1], f"{case.id} [{k}] on {ran}")
            out[case.id].append([ran, err[0]] + [int(x) for x in err[1][1:]])
            run_case(after, ctx, "no_static" if knob == "no_static" else "default", flags)
    ctx.close()
    return out


@pytest.mark.gpu
def test_no_static_flag():
    """COLLECT_NO_STATIC runs the interpreter (it never consults the run-time specialiser)."""
    ctx = P.Context(0)
    for case in CASES:
        run_case(case, ctx, "no_static", F.COLLECT_NO_STATIC)
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("knob", list(KNOBS))
def test_knob(knob):
    code = f"import sys; sys.path.insert(0, 'tests'); import test_eval_routes as K; print('ran', K.run_knob({knob!r}))"
    env = dict(os.environ, **KNOBS[knob])
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and f"ran {len(CASES)}" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
def test_errors_agree_across_routes():
    """Integer /0 and an out-of-bounds gather report the same lowest position, node, component, value and bound on every
    route: the pre-built signature (MDIM_JIT=0), the interpreter (COLLECT_NO_STATIC), [ops] and [ops+shape]."""
    runs = {}
    for knob in list(KNOBS) + ["no_static"]:
        code = f"import sys, json; sys.path.insert(0, 'tests'); import test_eval_routes as K; print('json', json.dumps(K.run_errors({knob!r})))"
        env = dict(os.environ, **KNOBS.get(knob, {}))
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
        assert r.returncode == 0 and "json " in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
        runs[knob] = json.loads(r.stdout.split("json ", 1)[1])
    for case in ERROR_CASES:
        recs = [rec for knob in runs for rec in runs[knob][case.id]]
        assert len({tuple(rec[1:]) for rec in recs}) == 1, (case.id, recs)
        ran = {rec[0] for rec in recs}
        want = {case.kernel("jit=0"), case.kernel("no_static")} | ({"mdim_jit_kernel[ops]"} if case.sig is None else set())
        if not case.stream:
            want.add("mdim_jit_kernel[ops+shape]")
            assert runs["default"][case.id][1][0] == "mdim_jit_kernel[ops+shape]", runs["default"][case.id]
        assert ran == want, (case.id, ran, want)
