"""The 1- and 2-byte integers i8, i16 and u16: every operator, unary op and cast at its value edges, the folds and views that
serve them, and the Python API, against a reference written here from Rust's release-build rules.

The reference (independent of exec.cuh and k_fold_split.cu; the C oracle under oracle/ covers the older types only):
  * integers are Python ints reduced mod 2^w (w = 8 or 16): Add, Sub, Mul, Neg and Not wrap, Abs(MIN) = MIN; Div and Rem
    truncate toward zero; x / 0, x % 0, MIN / -1 and MIN % -1 panic; a shift takes the rhs's own bits masked by w - 1, and Shr
    is arithmetic on i8 / i16 and logical on u16;
  * casts are Rust `as`: int->int wraps (sign-extending a signed source), float->int truncates toward zero, saturates and maps
    NaN to 0, and every i8 / i16 / u16 value is exact in f32 and f64.
Each elementwise case runs through the evaluator forms of test_value_edges.py (stream, a 64-bit slot, half vector, an output
that is only element-aligned, rank 2), naming the exact kernel on each.
"""
import ctypes as C
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from helpers import assert_same_bits, emu_collect, emu_collect_tuple
import multidimension_b200 as P
from multidimension_b200 import _ffi as F
from multidimension_b200 import lowering as L
from multidimension_b200 import usize, Array, Scalar
from multidimension_b200.runtime import Storage
import test_eval_routes as R
from test_eval_routes import Subject, axes, fold, instantiation, KNOBS
from test_value_edges import Elem, forms, RUNS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = (F.I8, F.I16, F.U16)
INTS = (F.U8, F.I32, F.U32, F.I64, F.U64) + NEW
FLOATS = (F.F32, F.F64)
SIGNED = (F.I8, F.I16, F.I32, F.I64)
WIDTH = {F.U8: 8, F.I8: 8, F.I16: 16, F.U16: 16, F.I32: 32, F.U32: 32, F.I64: 64, F.U64: 64}
NPN = {F.I8: np.int8, F.I16: np.int16, F.U16: np.uint16}
NPD = {**R.NPD, **NPN}


def _with_narrow_tables(setitem):
    """The shared executors and builders of test_eval_routes (Subject, Ref, fold) look element types up in its NPD / DT tables:
    give them the three new types, through `setitem` (pytest's monkeypatch.setitem, undone after each test, or plain assignment
    in a process of its own)."""
    for d, t in NPN.items():
        setitem(R.NPD, d, t)
        setitem(R.DT, F.DTYPE_NAME[d], d)


@pytest.fixture(autouse=True)
def _narrow_tables(monkeypatch):
    _with_narrow_tables(monkeypatch.setitem)
NAME = F.DTYPE_NAME
OPNAME = {F.ADD: "add", F.SUB: "sub", F.MUL: "mul", F.DIV: "div", F.REM: "rem", F.AND: "and", F.OR: "or", F.XOR: "xor",
          F.SHL: "shl", F.SHR: "shr"}
PANIC = object()


# ---- the reference ----------------------------------------------------------------------------------------------------------
def int_range(dt):
    w = WIDTH[dt]
    return (-(1 << (w - 1)), (1 << (w - 1)) - 1) if dt in SIGNED else (0, (1 << w) - 1)


def wrap(v, dt):
    w = WIDTH[dt]
    v &= (1 << w) - 1
    return v - (1 << w) if dt in SIGNED and v >> (w - 1) else v


def ref_int(op, dt, rdt, a, b):
    if op in (F.ADD, F.SUB, F.MUL, F.AND, F.OR, F.XOR):
        return wrap({F.ADD: a + b, F.SUB: a - b, F.MUL: a * b, F.AND: a & b, F.OR: a | b, F.XOR: a ^ b}[op], dt)
    if op in (F.DIV, F.REM):
        if b == 0 or (dt in SIGNED and a == int_range(dt)[0] and b == -1):
            return PANIC
        q = abs(a) // abs(b)
        q = -q if (a < 0) != (b < 0) else q
        return q if op == F.DIV else a - b * q
    n = (b % (1 << WIDTH[rdt])) & (WIDTH[dt] - 1)
    return wrap(a << n, dt) if op == F.SHL else a >> n


def ref_binary(op, dt, rdt, a, b):
    r = [ref_int(op, dt, rdt, int(x), int(y)) for x, y in zip(a, b)]
    err = np.array([v is PANIC for v in r], bool)
    return np.array([0 if v is PANIC else v for v in r], NPD[dt]), err


def ref_unary(op, dt, a):
    f = {F.NEG: lambda x: -x, F.NOT: lambda x: ~x, F.ABS: abs}[op]
    return np.array([wrap(f(int(x)), dt) for x in a], NPD[dt])


def ref_cast_one(x, src, dst):
    if src in FLOATS:
        x = float(x)
        lo, hi = int_range(dst)
        if x != x:
            return 0
        if x in (float("inf"), float("-inf")):
            return lo if x < 0 else hi
        return min(max(int(x), lo), hi)
    x = int(x)
    if dst in INTS:
        return wrap(x, dst)
    assert src in NEW  # exact in either float type
    return np.float32(x) if dst == F.F32 else float(x)


def ref_cast(src, dst, a):
    return np.array([ref_cast_one(x, src, dst) for x in a], NPD[dst])


# ---- edge tables ------------------------------------------------------------------------------------------------------------
def edges(dt):
    if dt in FLOATS:
        t = NPD[dt]
        v = [np.nan, np.inf, -np.inf, 0.0, -0.0, 0.5, -0.5, 0.99, -0.99, 127.0, 127.99, 128.0, -128.0, -128.99, -129.0, 255.99, 256.0,
             300.7, -300.7, 32767.0, 32767.5, 32768.0, -32768.0, -32768.5, -32769.0, 65535.0, 65535.5, 65536.0, 1e30, -1e30, 1e-40]
        return np.array(v, t)
    lo, hi = int_range(dt)
    w = WIDTH[dt]
    v = [0, 1, -1, 2, -2, lo, lo + 1, hi, hi - 1, int("55" * (w // 8), 16), w - 1, w, 31, 7, 100, -100, 127, 128, -129, 255, 256,
         32767, 32768, -32769, 65535, 65536]
    return np.array(sorted({wrap(x, dt) for x in v}), NPD[dt])


# ---- elementwise cases ------------------------------------------------------------------------------------------------------
ELEMS = []


def cross(x, y):
    return np.repeat(x, len(y)), np.tile(y, len(x))


def add_binary(op, dt, rdt, a, b, tag="", drop_panics=True):
    want, werr = ref_binary(op, dt, rdt, a, b)
    if drop_panics and werr.any():
        keep = ~werr
        a, b, want, werr = np.asarray(a)[keep], np.asarray(b)[keep], want[keep], werr[keep]
    ELEMS.append(Elem(f"{OPNAME[op]}-{NAME[dt]}{'-' + NAME[rdt] if rdt != dt else ''}{tag}", dt, [(dt, a), (rdt, b)],
                      lambda x, y: L.Node(F.BINARY, dt, op=op, children=(x, y)), want, werr))


def add_binary_const(op, dt, c):
    a = edges(dt)
    want, werr = ref_binary(op, dt, dt, a, np.full(len(a), c, NPD[dt]))
    a, want, werr = a[~werr], want[~werr], werr[~werr]
    ELEMS.append(Elem(f"{OPNAME[op]}-{NAME[dt]}-const{c}", dt, [(dt, a)],
                      lambda x: L.Node(F.BINARY, dt, op=op, children=(x, L.Node(F.CONST, dt, imm=c))), want, werr, const_rhs=True))


for dt in NEW:
    a, b = cross(edges(dt), edges(dt))
    for op in (F.ADD, F.SUB, F.MUL, F.DIV, F.REM, F.AND, F.OR, F.XOR, F.SHL, F.SHR):
        add_binary(op, dt, dt, a, b)
    for rdt in (F.U8, F.I32, F.U64):  # a shift amount of another width: its own bits, masked
        a2, b2 = cross(edges(dt), edges(rdt))
        for op in (F.SHL, F.SHR):
            add_binary(op, dt, rdt, a2, b2)
    lo, hi = int_range(dt)
    for op, c in ((F.ADD, hi), (F.MUL, lo if dt in SIGNED else hi), (F.DIV, -1 if dt in SIGNED else 3), (F.REM, 7), (F.SHR, 15),
                  (F.XOR, -1 if dt in SIGNED else hi)):
        add_binary_const(op, dt, c)
    for op in (F.NEG, F.NOT, F.ABS):
        x = edges(dt)
        ELEMS.append(Elem(f"{ {F.NEG: 'neg', F.NOT: 'not', F.ABS: 'abs'}[op]}-{NAME[dt]}", dt, [(dt, x)],
                          lambda v, op=op, dt=dt: L.Node(F.UNARY, dt, op=op, children=(v,)), ref_unary(op, dt, x), np.zeros(len(x), bool)))
    for op in (F.DIV, F.REM):  # one panicking element at a known position among ordinary ones
        for kind, (p, q) in (("zero", (hi, 0)), ("min-1", (lo, -1))):
            if kind == "min-1" and dt not in SIGNED:
                continue
            a3 = np.array([hi, 7, lo, 100] * 6, NPD[dt])
            b3 = np.array([3, 2, 5, 1] * 6, NPD[dt])
            a3[13], b3[13] = p, q
            add_binary(op, dt, dt, a3, b3, tag=f"-panic-{kind}", drop_panics=False)
for src in INTS + FLOATS:
    for dst in INTS + FLOATS:
        if src != dst and (src in NEW or dst in NEW):
            x = edges(src)
            ELEMS.append(Elem(f"cast-{NAME[src]}-{NAME[dst]}", dst, [(src, x)],
                              lambda v, s=src, d=dst: L.Node(F.UNARY, d, op=F.CAST, src_dtype=s, children=(v,)), ref_cast(src, dst, x),
                              np.zeros(len(x), bool)))
ELEM_IDS = [e.id for e in ELEMS]
assert len(set(ELEM_IDS)) == len(ELEM_IDS)
assert sum(e.id.startswith("cast-") for e in ELEMS) == 48


# ---- folds and views --------------------------------------------------------------------------------------------------------
SPLIT_MIN_RED = 1 << 12  # program.hpp: kSplitMinRed
SOPS = (F.ADD, F.MUL, F.AND, F.OR, F.XOR)


def split_kernel(dst, src, op, layout):
    return f"k_fold_split<u{64 if F.DTYPE_SIZE[dst] == 8 else 32},src=u{F.DTYPE_SIZE[src] * 8},{OPNAME[op]},{layout}>"


def ref_fold(op, dst, init, x):
    """`let mut s = init; for v in row { s = s (op) v as dst }` over the last axis, mod 2^w (the operators are exact in any order)."""
    w = WIDTH[dst]
    v = np.asarray(x, np.int64).astype(np.uint64) & np.uint64((1 << w) - 1 if w < 64 else 2 ** 64 - 1)  # each element mod 2^w
    u = {F.ADD: np.add, F.MUL: np.multiply, F.AND: np.bitwise_and, F.OR: np.bitwise_or, F.XOR: np.bitwise_xor}[op]
    with np.errstate(over="ignore"):
        acc = u(np.uint64(wrap(init, dst) & ((1 << w) - 1)), u.reduce(v, axis=-1, dtype=np.uint64))
    acc = acc & np.uint64((1 << w) - 1 if w < 64 else 2 ** 64 - 1)
    return np.array([wrap(int(a), dst) for a in acc], NPD[dst])


class FoldCase:
    def __init__(self, id, build, route, kernel, flags=0):
        self.id, self.build, self.route, self.kernel, self.flags = id, build, route, kernel, flags

    def __repr__(self):
        return self.id


FOLDS = []


def split_values(op, src, n_out, K, rng):
    """n_out reductions of K elements of src, drawn so that every output depends on the elements that matter to its operator:
    Add and Xor over the whole range; Mul over odd values (a product of them is never 0); And over all-ones and Or over zeros,
    except that the first, the last and a middle element of each reduction clear (And) or set (Or) a bit of their own, the sign
    bit among them, so that losing or mis-extending any of them changes the result."""
    lo, hi = int_range(src)
    w = WIDTH[src]
    if op in (F.ADD, F.XOR):
        return rng.integers(lo, hi + 1, (n_out, K))
    if op == F.MUL:
        return rng.integers(lo, hi + 1, (n_out, K)) | 1
    x = np.full((n_out, K), -1 if op == F.AND else 0, np.int64)
    for i in range(n_out):
        for j, k in enumerate((0, K // 2 + i, K - 1)):
            bit = 1 << ((w - 1 - j - 2 * i) % w)  # the sign bit (w - 1) in the first reduction's first element
            x[i, k] = ~bit if op == F.AND else bit
    half = 1 << (w - 1) if src in SIGNED else 0
    return (x + half) % (1 << w) - half  # wrapped into src's range


# (elements per reduction, outputs, element offset of the first, row pitch) of each layout
SPLIT_LAYOUTS = {"runs": (SPLIT_MIN_RED + 37, 3, 3, None),        # 3 runs, 3 elements past a 32-byte boundary, a partial last vector
                 "cols-odd": (SPLIT_MIN_RED + 5, 37, 1, 40),      # columns from an odd offset: the scalar column walk
                 "cols": (SPLIT_MIN_RED + 5, 40, 0, 48)}          # 16-byte-aligned base and pitch: 128-bit column groups, one partial


def add_split(op, src, dst, layout):
    init = {F.AND: -1, F.OR: 0, F.MUL: 3}.get(op, -1 if dst in SIGNED else 3)  # And: all ones, so that every cleared bit shows
    K, n_out, off, pitch = SPLIT_LAYOUTS[layout]

    def build():
        rng = np.random.default_rng(op * 100 + src * 10 + dst + len(layout))
        v = split_values(op, src, n_out, K, rng)
        o, r = ax = axes(n_out, K)
        if pitch is None:
            mem = np.concatenate([np.zeros(off, np.int64), v.reshape(-1)])
            stride = {o: K, r: 1}
        else:
            mem = np.zeros(off + K * pitch, np.int64)
            mem[off:].reshape(K, pitch)[:, :n_out] = v.T
            stride = {o: 1, r: pitch}
        lf = L.Node(F.LEAF, src, buf=Storage.from_host(src, mem.astype(NPD[src])), offset=off, stride=stride)
        body = L.Node(F.UNARY, dst, op=F.CAST, src_dtype=src, children=(lf,)) if dst != src else lf
        return Subject(fold(NAME[dst], op, body, [r], init), [o]), ref_fold(op, dst, init, v)
    kind = layout.split("-")[0]
    FOLDS.append(FoldCase(f"split-{NAME[src]}-{NAME[dst]}-{OPNAME[op]}-{layout}", build, f"fold_split.{kind} ",
                          split_kernel(dst, src, op, kind)))


for op in SOPS:
    for src in NEW:
        for dst in ((src, F.I64) if src in SIGNED else (src, F.U64)):
            for layout in SPLIT_LAYOUTS:
                add_split(op, src, dst, layout)
# the routes the issue names: i8 -> i32 sums, and a u16 fold into a 32-bit slot of another type
for layout in SPLIT_LAYOUTS:
    add_split(F.ADD, F.I8, F.I32, layout)
    add_split(F.XOR, F.U16, F.U32, layout)


def add_eval_fold(dt, op, outer):
    def build():  # the evaluator's own fold from init -1: over the last axis of a (37, 5), or over its outer axis
        x = np.random.default_rng(dt * 10 + op).choice(edges(dt), 37 * 5).reshape(37, 5)
        o, r = ax = axes(5, 37) if outer else axes(37, 5)
        st = {o: 1, r: 5} if outer else {o: 5, r: 1}
        lf = L.Node(F.LEAF, dt, buf=Storage.from_host(dt, x.reshape(-1)), offset=0, stride=st)
        return Subject(fold(NAME[dt], op, lf, [r], -1), [o]), ref_fold(op, dt, -1, x.T if outer else x)
    FOLDS.append(FoldCase(f"eval-{NAME[dt]}-{OPNAME[op]}-{'outer' if outer else 'last'}", build, "generic.interp s32 v1x1 rank=1+1 ",
                          instantiation(None, 4, 1, 2, False, 2), F.COLLECT_NO_FASTPATH | F.COLLECT_NO_STATIC))


for dt in NEW:
    for op in (F.ADD, F.MUL, F.XOR):
        for outer in (False, True):
            add_eval_fold(dt, op, outer)
FOLD_IDS = [c.id for c in FOLDS]


def view_cases():
    """Selections on the evaluator (no arithmetic): a u16 transpose, a gather from i16, a concat and a diagonal whose zero is a
    negative i8.  -> [(id, Subject, expected describe() prefix)]; the reference is test_eval_routes.Ref."""
    rng = np.random.default_rng(5)
    out = []
    r, c = ax = axes(33, 40)
    m = Storage.from_host(F.U16, rng.integers(0, 65536, 33 * 40))
    out.append(("transpose-u16", Subject(L.Node(F.LEAF, F.U16, buf=m, offset=0, stride={r: 1, c: 33}), ax), "generic."))
    o, = ax1 = axes(1000)
    srcv = Storage.from_host(F.I16, rng.integers(-32768, 32768, 777))
    idx = Storage.from_host(F.U64, rng.integers(0, 777, 1000))
    g = L.Node(F.GATHER, F.I16, buf=srcv, children=(L.Node(F.LEAF, F.U64, buf=idx, offset=0, stride={o: 1}),), gstride=(1,), bound=(777,))
    out.append(("gather-i16", Subject(g, ax1), "stream."))
    a = Storage.from_host(F.I16, rng.integers(-32768, 32768, 1000))
    b = Storage.from_host(F.I16, rng.integers(-32768, 32768, 1000))
    cc = L.Node(F.CONCAT, F.I16, children=(L.Node(F.LEAF, F.I16, buf=a, offset=0, stride={o: 1}),
                                           L.Node(F.LEAF, F.I16, buf=b, offset=-613, stride={o: 1})), pairs=((o, 613),))
    out.append(("concat-i16", Subject(cc, ax1), "stream."))
    r2, c2 = ax2 = axes(24, 24)
    d8 = Storage.from_host(F.I8, rng.integers(-128, 128, 24 * 24))
    dg = L.Node(F.DIAG, F.I8, children=(L.Node(F.LEAF, F.I8, buf=d8, offset=0, stride={r2: 24, c2: 1}),), pairs=((r2, c2),), imm=-5)
    out.append(("diag-i8-zero-5", Subject(dg, ax2), "generic."))
    return out


# ---- CPU half ----------------------------------------------------------------------------------------------------------------
def test_reference_rules():
    assert ref_int(F.SHR, F.I8, F.I8, -128, 9) == -64  # the amount masked to 1
    assert ref_unary(F.ABS, F.I16, [-32768]).tolist() == [-32768]
    assert ref_cast_one(np.float32(300.7), F.F32, F.I8) == 127
    assert ref_cast_one(-1, F.I16, F.U64) == 2 ** 64 - 1
    assert ref_cast_one(float("nan"), F.F32, F.U16) == 0
    assert ref_int(F.DIV, F.I8, F.I8, -128, -1) is PANIC and ref_int(F.REM, F.U16, F.U16, 5, 0) is PANIC
    assert ref_int(F.SHR, F.U16, F.U16, 0x8000, 15) == 1 and ref_int(F.SHL, F.I16, F.I32, 1, -1) == -32768
    assert ref_int(F.DIV, F.I16, F.I16, -7, 2) == -3 and ref_int(F.REM, F.I8, F.I8, -7, 2) == -1


@pytest.mark.parametrize("elem", ELEMS, ids=ELEM_IDS)
def test_host_forms(elem):
    """Each form: describe() names the planned route and instantiation; the host emulator (the library's planner over a host
    build of exec.cuh) under the default route and under COLLECT_NO_STATIC equals the reference."""
    for fm in forms(elem):
        s, case = fm.subject(), fm.case
        d = s.describe()
        assert d.startswith(case.route), (case.id, case.route, d)
        assert case.planned + "]" in d or case.planned + "," in d, (case.id, case.planned, d)
        for flags, knob in ((0, "jit=0"), (F.COLLECT_NO_STATIC, "no_static")):
            got, err, ran = s.emu(flags)
            assert ran == case.kernel(knob), f"{case.id} [emu {knob}]: ran {ran}, expected {case.kernel(knob)}"
            fm.check(got, err, f"{case.id} [emu {knob}] on {ran}")


@pytest.mark.parametrize("case", FOLDS, ids=FOLD_IDS)
def test_host_folds(case):
    s, want = case.build()
    d = s.describe(case.flags)
    assert d.startswith(case.route), d
    got, err, ran = s.emu(case.flags)
    assert err is None, err
    assert_same_bits(got[0], want, f"{case.id} (emu on {ran})")


def test_host_views():
    for id, s, route in view_cases():
        assert s.describe().startswith(route), (id, s.describe())
        (want,), _ = s.reference()
        got, err, _ = s.emu(0)
        assert err is None, (id, err)
        assert_same_bits(got[0], want, id)


def test_dedicated_routes_refuse_narrow_types():
    """The tiled transpose, the row fold and the column walk take 4- and 8-byte types only."""
    for dt in NEW:
        r, c = ax = axes(64, 64)
        leaf = L.Node(F.LEAF, dt, buf=Storage.from_host(dt, np.zeros(64 * 64, NPD[dt])), offset=0, stride={r: 1, c: 64})
        assert not Subject(leaf, ax).describe().startswith("transpose"), NAME[dt]
        o, k = ax = axes(64, 64)
        rows = L.Node(F.LEAF, dt, buf=Storage.from_host(dt, np.zeros(64 * 64, NPD[dt])), offset=0, stride={o: 64, k: 1})
        assert Subject(fold(NAME[dt], F.ADD, rows, [k], 0), [o]).describe().startswith("generic."), NAME[dt]
        cols = L.Node(F.LEAF, dt, buf=Storage.from_host(dt, np.zeros(64 * 64, NPD[dt])), offset=0, stride={o: 1, k: 64})
        assert Subject(fold(NAME[dt], F.ADD, cols, [k], 0), [o]).describe().startswith("generic."), NAME[dt]


def test_jit_sources_compile():
    """NVRTC compiles the [ops] and [ops+shape] source of every form the GPU half runs through the run-time specialiser."""
    exprs = []
    for e in ELEMS:
        for fm in forms(e):
            if fm.name in ("stream", "s64", "rank2"):
                s = fm.subject()
                exprs.append((fm.case.id, s, L.emit(s.root(), s.axes, "host")))

    def check(item):
        log = C.create_string_buffer(2048)
        return item[0], F.lib().mdim_jit_check_nodevice(C.byref(item[2].expr), 0, log, 2048), log.value.decode()
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as pool:
        res = list(pool.map(check, exprs))
    if res and res[0][1] == F.ERR_UNSUPPORTED and "NVRTC" in res[0][2]:
        pytest.skip("NVRTC is not installed")
    bad = [(i, st, log[:300]) for i, st, log in res if st != F.OK]
    assert not bad, bad[:3]


def test_python_api():
    """Type inference from numpy, Scalar, a traced closure, to_raw, and tuples (i16, u64) from zip and enumerate."""
    x = np.array([-32768, -2, -1, 0, 1, 2, 12345, 32767], np.int16)
    for arr, T in ((x, "i16"), (x.astype(np.int8), "i8"), (x.view(np.uint16), "u16")):
        a = Array.new(usize, len(arr), arr)
        assert a.T == T and F.DTYPE_NAME[P.view.dtype_of(a.T)] == T
        assert_same_bits(np.asarray(a.to_raw()), arr, T)
    a = Array.new(usize, 8, x)
    want = np.array([wrap(int(v) * 3 - 1, F.I16) for v in x], np.int16)
    assert_same_bits(emu_collect(a.map(lambda v: v * 3 - 1)), want, "x * 3 - 1")
    assert_same_bits(emu_collect(a * Scalar(3, "i16") - Scalar(1, "i16")), want, "x * Scalar(3) - Scalar(1)")
    idx = Array.new(usize, 8, np.arange(8, dtype=np.uint64) * 3)
    got = emu_collect_tuple(a.zip(idx))
    assert got == [(int(v), 3 * k) for k, v in enumerate(x)], got
    got = emu_collect_tuple(a.enumerate())
    assert got == [(k, int(v)) for k, v in enumerate(x)], got


# ---- GPU half ----------------------------------------------------------------------------------------------------------------
NS = F.COLLECT_NO_STATIC


def run_setting(knob):
    """Every form of every case that `knob` runs (and, in the default setting, every fold and view).  -> collects checked."""
    _with_narrow_tables(lambda table, key, value: table.__setitem__(key, value))  # (a process of its own)
    ctx = P.Context(0)
    n = 0
    for e in ELEMS:
        for fm in forms(e):
            for flags in RUNS[knob].get(fm.name, ()):
                k = "no_static" if flags & NS else knob
                got, err, ran = fm.subject().gpu(ctx, flags)
                assert ran == fm.case.kernel(k), f"{fm.case.id} [{k}]: ran {ran}, expected {fm.case.kernel(k)}"
                fm.check(got, err, f"{fm.case.id} [{k}] on {ran}")
                n += 1
    if knob == "default":
        for case in FOLDS:
            s, want = case.build()
            got, err, ran = s.gpu(ctx, case.flags)
            assert err is None, (case.id, err)
            assert ran == case.kernel, f"{case.id}: ran {ran}, expected {case.kernel}"
            assert_same_bits(got[0], want, f"{case.id} on {ran}")
            n += 1
        for id, s, _ in view_cases():
            (want,), _ = s.reference()
            got, err, ran = s.gpu(ctx, NS)
            assert err is None, (id, err)
            assert "interp" in ran, (id, ran)
            assert_same_bits(got[0], want, f"{id} on {ran}")
            n += 1
    ctx.close()
    return n


def expected_runs(knob):
    n = sum(len(RUNS[knob].get(fm.name, ())) for e in ELEMS for fm in forms(e))
    return n + (len(FOLDS) + len(view_cases()) if knob == "default" else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("knob", list(RUNS))
def test_device_forms(knob):
    """The JIT settings are read once per process, so each runs in a subprocess of its own."""
    code = f"import sys; sys.path.insert(0, 'tests'); import test_narrow_ints as K; print('ran', K.run_setting({knob!r}))"
    env = dict(os.environ, **KNOBS[knob])
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and f"ran {expected_runs(knob)}" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.gpu
def test_i16_sum_past_32bit_offsets():
    """A whole-array i16 -> i64 sum over 2^31 + 37 elements (4 GiB + 74 bytes) on the split fold."""
    n = (1 << 31) + 37
    rng = np.random.default_rng(11)
    p = rng.integers(-32768, 32768, 1 << 20).astype(np.int16)
    x = np.concatenate([np.tile(p, n >> 20), p[:n & ((1 << 20) - 1)]])
    want = int(p.astype(np.int64).sum()) * (n >> 20) + int(p[:n & ((1 << 20) - 1)].astype(np.int64).sum())
    ctx = P.Context(0)
    st = Storage.from_host(F.I16, x)
    del x
    r, = ax = axes(n)
    lf = L.Node(F.LEAF, F.I16, buf=st, offset=0, stride={r: 1})
    s = Subject(fold("i64", F.ADD, L.Node(F.UNARY, F.I64, op=F.CAST, src_dtype=F.I16, children=(lf,)), [r], 0), [])
    got, err, ran = s.gpu(ctx, 0)
    assert err is None, err
    assert ran == "k_fold_split<u64,src=u16,add,runs>", ran
    assert int(got[0][0]) == want, (int(got[0][0]), want)
    del st, s, lf
    ctx.close()


@pytest.mark.gpu
def test_allreduce_refuses_16_bit():
    """NCCL has no 16-bit integer: mdim_allreduce refuses I16 / U16; I8 is NCCL's int8."""
    from multidimension_b200.sharding import Comm
    ctx = P.Context(0)
    try:
        uid = Comm.unique_id()
    except F.MdimError as e:
        ctx.close()
        pytest.skip(f"no NCCL: {e}")
    comm = Comm(ctx, 0, 1, uid)
    for dt in (F.I16, F.U16):
        st = Storage.device(ctx, dt, 16)
        with pytest.raises(F.MdimError) as ei:
            comm.all_reduce(st)
        assert ei.value.status == F.ERR_UNSUPPORTED, ei.value.status
    st = Storage.from_host(F.I8, np.array([-128, -1, 5, 127], np.int8))
    st.ensure_device(ctx)
    comm.all_reduce(st)
    ctx.sync()
    out = np.empty(4, np.int8)
    ctx.download(out, st.dptr)
    assert out.tolist() == [-128, -1, 5, 127]
    comm.close()
    ctx.close()
