"""Every operator, unary op and cast at its value edges, on every form of the evaluator, against an exact reference.

The route tests pin each kernel to its plan and check it at its shape edges with ordinary values.  This file checks the values:
INT_MIN against -1, shifts by the width and by a negative amount, NaN, signed zeros, subnormals, infinities, and each
float->int saturation and int->float rounding boundary.  An operator can be wrong at such a value on one route only (the device
`cvt`, `fmodf` and `sqrtf`, the NVRTC-built kernels, a narrow type carried in a 64-bit slot, u8 lanes packed into a word), so
every case runs through each form of the evaluator that serves it, and names the kernel it expects on each.

The reference is written here from Rust's release-build rules, independently of exec.cuh and of the C oracle:
  * integers are Python ints reduced mod 2^w: Add, Sub, Mul and Neg wrap, Abs(MIN) = MIN; Div and Rem truncate toward zero;
    x / 0, x % 0, MIN / -1 and MIN % -1 panic; a shift takes its amount from the rhs in the rhs's own type (two's complement),
    masked by width - 1, and Shr is arithmetic on i32 / i64 and logical otherwise;
  * floats are numpy in the element type, one correctly rounded operation at a time (Rem is np.fmod, which is exact; Sqrt is
    np.sqrt); Neg and Abs act on the sign bit only;
  * casts are Rust `as`: float->int truncates the exact value toward zero, saturates, and maps NaN to 0; int->int wraps;
    int->float rounds the exact integer to nearest even in integer arithmetic (never through f64, which rounds twice);
    f64->f32 is numpy's correctly rounded conversion.
Comparison is bit for bit, except that any NaN equals any NaN (Rust leaves the payload unspecified).

The forms, each asserting the exact `last_kernel()`:
  * stream:  rank 1, output 32-byte aligned (256-bit stores; u8 lanes packed 8 to a word): the interpreter under
             COLLECT_NO_STATIC, the pre-built signature or `mdim_jit_kernel[ops]` by default, the signature or the
             interpreter under MDIM_JIT=0;
  * s64:     a 32-bit dtype computed in a 64-bit slot, as one run of a tuple whose other run is a u64 IOTA;
  * half:    8k + 4 (s32) or 4k + 2 (s64) elements, half the vector width, on the interpreter;
  * v1:      the output one element past its alignment, re-planned to scalar stores, on the interpreter;
  * rank2:   a transposed operand over two axes that do not merge: `[ops+shape]` under MDIM_JIT_SHAPES=1 and the
             interpreter under MDIM_JIT=0.
The JIT settings are read once per process, so each runs in a subprocess of its own.  Folds run on the row fold (plain and
with the fused epilogue, whose f32 operators k_fold.cu restates), the column fold, the few-output split fold and the
evaluator's own fold, each against a sequential fold of the same reference.
"""
import ctypes as C
import math
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from helpers import assert_same_bits, oracle_collect, emu_collect
import multidimension_b200 as P
from multidimension_b200 import _ffi as F
from multidimension_b200 import lowering as L
from multidimension_b200 import usize, Array, Scalar, fold_rows
from multidimension_b200.runtime import Storage
from test_eval_routes import Subject, Case, axes, fold, instantiation, registry, _parse, check_outputs, KNOBS, DT, NPD
from test_kernel_routes import fold_rows_kernel
from test_fold_split_routes import split_kernel, SPLIT_MIN_RED

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FLOATS = (F.F32, F.F64)
INTS = (F.U8, F.I32, F.U32, F.I64, F.U64)
SIGNED = (F.I32, F.I64)
WIDTH = {F.U8: 8, F.I32: 32, F.U32: 32, F.I64: 64, F.U64: 64}
UINT = {F.F32: np.uint32, F.F64: np.uint64}
NAME = F.DTYPE_NAME
OPNAME = {F.ADD: "add", F.SUB: "sub", F.MUL: "mul", F.DIV: "div", F.REM: "rem", F.AND: "and", F.OR: "or", F.XOR: "xor",
          F.SHL: "shl", F.SHR: "shr"}
UNNAME = {F.NEG: "neg", F.NOT: "not", F.ABS: "abs", F.SQRT: "sqrt"}
PANIC = object()


# ---- the exact reference ----------------------------------------------------------------------------------------------------
def int_range(dt):
    w = WIDTH[dt]
    return (-(1 << (w - 1)), (1 << (w - 1)) - 1) if dt in SIGNED else (0, (1 << w) - 1)


def wrap(v, dt):
    w = WIDTH[dt]
    v &= (1 << w) - 1
    return v - (1 << w) if dt in SIGNED and v >> (w - 1) else v


def ref_int_binary(op, dt, rdt, a, b):
    """One element of `a (op) b` for an integer dtype: the value, or PANIC."""
    if op == F.ADD:
        return wrap(a + b, dt)
    if op == F.SUB:
        return wrap(a - b, dt)
    if op == F.MUL:
        return wrap(a * b, dt)
    if op in (F.DIV, F.REM):
        if b == 0 or (dt in SIGNED and a == int_range(dt)[0] and b == -1):
            return PANIC
        q = abs(a) // abs(b)  # truncation toward zero (Python's // floors)
        if (a < 0) != (b < 0):
            q = -q
        return q if op == F.DIV else a - b * q
    if op == F.AND:
        return wrap(a & b, dt)
    if op == F.OR:
        return wrap(a | b, dt)
    if op == F.XOR:
        return wrap(a ^ b, dt)
    n = (b % (1 << WIDTH[rdt])) & (WIDTH[dt] - 1)  # the rhs's own bits, masked by the lhs width - 1
    return wrap(a << n, dt) if op == F.SHL else a >> n  # >> on a Python int: arithmetic when signed, logical when not


def ref_binary(op, dt, rdt, a, b):
    """Elementwise `a (op) b` over two sequences -> (array of dt, panic mask)."""
    if dt in FLOATS:
        x, y = np.asarray(a, NPD[dt]), np.asarray(b, NPD[dt])
        with np.errstate(all="ignore"):
            r = {F.ADD: np.add, F.SUB: np.subtract, F.MUL: np.multiply, F.DIV: np.divide, F.REM: np.fmod}[op](x, y)
        return r.astype(NPD[dt]), np.zeros(r.shape, bool)
    r = [ref_int_binary(op, dt, rdt, int(x), int(y)) for x, y in zip(a, b)]
    err = np.array([v is PANIC for v in r], bool)
    return np.array([0 if v is PANIC else v for v in r], NPD[dt]), err


def ref_unary(op, dt, a):
    if dt in FLOATS:
        u = np.asarray(a, NPD[dt]).view(UINT[dt])
        sign = UINT[dt](1 << (8 * np.dtype(UINT[dt]).itemsize - 1))
        if op == F.NEG:
            return (u ^ sign).view(NPD[dt])
        if op == F.ABS:
            return (u & ~sign).view(NPD[dt])
        assert op == F.SQRT
        with np.errstate(all="ignore"):
            return np.sqrt(np.asarray(a, NPD[dt]))
    f = {F.NEG: lambda x: wrap(-x, dt), F.NOT: lambda x: wrap(~x, dt), F.ABS: lambda x: wrap(abs(x), dt)}[op]
    return np.array([f(int(x)) for x in a], NPD[dt])


def round_int(v, mant):
    """The integer v rounded to `mant` significant bits, to nearest, ties to even: exact, in integer arithmetic."""
    m = abs(v)
    sh = m.bit_length() - mant
    if sh > 0:
        q, r, half = m >> sh, m & ((1 << sh) - 1), 1 << (sh - 1)
        if r > half or (r == half and q & 1):
            q += 1
        m = q << sh
    return -m if v < 0 else m


def ref_cast_one(x, src, dst):
    if src in FLOATS:
        x = float(x)  # exact: every f32 is an f64
        if dst in FLOATS:
            with np.errstate(over="ignore"):
                return np.float32(x) if dst == F.F32 else x  # numpy's f64 -> f32 is correctly rounded, subnormals and overflow too
        lo, hi = int_range(dst)
        if math.isnan(x):
            return 0
        if math.isinf(x):
            return lo if x < 0 else hi
        return min(max(int(x), lo), hi)  # int() of a finite float truncates its exact value
    x = int(x)
    if dst in INTS:
        return wrap(x, dst)
    r = round_int(x, 24 if dst == F.F32 else 53)  # at most 24 / 53 significant bits: float() and np.float32() are exact
    return np.float32(float(r)) if dst == F.F32 else float(r)


def ref_cast(src, dst, a):
    return np.array([ref_cast_one(x, src, dst) for x in a], NPD[dst])


# ---- edge tables ------------------------------------------------------------------------------------------------------------
def _int_edges(dt):
    lo, hi = int_range(dt)
    if dt == F.U8:
        return [0, 1, 7, 8, 127, 128, 254, 255]
    v = [0, 1, 2, lo, lo + 1, hi, hi - 1, 2 ** 24 - 1, 2 ** 24 + 1, 31, 32, 33, 63, 64, 65]
    if dt in SIGNED:
        v += [-1, -2, -(2 ** 24 + 1), -31, -33]
    if WIDTH[dt] == 64:
        v += [2 ** 53 - 1, 2 ** 53 + 1, 2 ** 60 + 2 ** 36, 2 ** 60 + 2 ** 36 + 1, 2 ** 32 + 3, 2 ** 31]
        if dt in SIGNED:
            v += [-(2 ** 53 + 1), -(2 ** 60 + 2 ** 36 + 1)]
    if dt == F.U32:
        v += [2 ** 31, 2 ** 31 - 1, 2 ** 31 + 1, 2 ** 32 - 129, 2 ** 32 - 128]
    if dt == F.U64:
        v += [2 ** 63, 2 ** 63 - 1, 2 ** 63 + 1, 2 ** 64 - 2 ** 39, 2 ** 64 - 2 ** 39 - 1, 2 ** 64 - 2 ** 40, 2 ** 63 + 2 ** 39 + 1]
    return sorted(set(v))


def _float_edges(dt):
    t = NPD[dt]
    fi = np.finfo(t)
    up, down = t(np.inf), t(-np.inf)
    v = [0.0, -0.0, 1.0, -1.0, 0.5, -0.5, 1.5, -2.5, np.nextafter(t(1), t(0)), np.nextafter(t(-1), t(0)),
         fi.smallest_subnormal, -fi.smallest_subnormal, fi.smallest_normal - fi.smallest_subnormal, fi.smallest_normal,
         -fi.smallest_normal, fi.max, -fi.max, np.inf, -np.inf, np.nan]
    for b in (255, 256, 2 ** 31, -2 ** 31, 2 ** 32, 2 ** 63, -2 ** 63, 2 ** 64):  # each float->int saturation boundary
        x = t(b)
        v += [np.nextafter(x, down), x, np.nextafter(x, up)]
    if dt == F.F64:
        over = 3.4028235677973366e38  # f32 MAX + half an ulp: the tie that rounds to inf
        tiny = 2.0 ** -150            # half the smallest f32 subnormal: the tie that rounds to 0
        for x in (over, tiny, -tiny, 1.5 * 2.0 ** -149):
            v += [np.nextafter(x, -np.inf), x, np.nextafter(x, np.inf)]
        v += [1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24, 16777217.0, -16777219.0, float(np.finfo(np.float32).max), 2.0 ** 128, 1e-320]
    return np.array(v, t)


def edges(dt):
    return _float_edges(dt) if dt in FLOATS else np.array(_int_edges(dt), NPD[dt])


# ---- one elementwise case ---------------------------------------------------------------------------------------------------
class Elem:
    """An op over one or two operand sequences.  make(leaves) -> the op node over the given operand nodes; want, werr: the
    reference and its panic mask, one per element."""

    def __init__(self, id, out_dt, operands, make, want, werr, sig=None, const_rhs=False):
        self.id, self.out_dt, self.operands, self.make = id, out_dt, operands, make
        self.want, self.werr, self.sig, self.const_rhs = want, werr, sig, const_rhs
        dts = [out_dt] + [dt for dt, _ in operands]
        self.slot = 8 if any(F.DTYPE_SIZE[d] == 8 for d in dts) else 4
        self.depth = 1 + (len(operands) == 2 or const_rhs)

    def __repr__(self):
        return self.id


ELEMS = []


def _sig_two(op, dt, const_rhs):
    if dt == F.F32 and op in (F.ADD, F.SUB, F.MUL, F.DIV):
        return f"Sig{OPNAME[op].capitalize()}{'C' if const_rhs else ''}F32"
    if not const_rhs and (dt, op) in ((F.F64, F.ADD), (F.F64, F.MUL), (F.U64, F.ADD)):
        return f"Sig{OPNAME[op].capitalize()}{NAME[dt].upper()}"
    return None


def add_binary(op, dt, rdt, a, b, tag="", drop_panics=True):
    want, werr = ref_binary(op, dt, rdt, a, b)
    if drop_panics and werr.any():
        keep = ~werr
        a, b, want, werr = np.asarray(a)[keep], np.asarray(b)[keep], want[keep], werr[keep]
    ELEMS.append(Elem(f"{OPNAME[op]}-{NAME[dt]}{'-' + NAME[rdt] if rdt != dt else ''}{tag}", dt, [(dt, a), (rdt, b)],
                      lambda x, y: L.Node(F.BINARY, dt, op=op, children=(x, y)), want, werr, sig=_sig_two(op, dt, False)))


def add_binary_const(op, dt, a, c):
    want, werr = ref_binary(op, dt, dt, a, np.full(len(a), c, NPD[dt]))
    a, want, werr = a[~werr], want[~werr], werr[~werr]  # MIN / -1 and MIN % -1 are the panic cases' business
    imm = float(c) if dt in FLOATS else int(c)
    ELEMS.append(Elem(f"{OPNAME[op]}-{NAME[dt]}-const{imm!r}", dt, [(dt, a)],
                      lambda x: L.Node(F.BINARY, dt, op=op, children=(x, L.Node(F.CONST, dt, imm=imm))), want, werr,
                      sig=_sig_two(op, dt, True), const_rhs=True))


def cross(x, y):
    return np.repeat(x, len(y)), np.tile(y, len(x))


def build_elems():
    for dt in INTS + FLOATS:
        e = edges(dt)
        a, b = cross(e, e)
        for op in (F.ADD, F.SUB, F.MUL, F.DIV, F.REM) + ((F.AND, F.OR, F.XOR) if dt in INTS else ()):
            add_binary(op, dt, dt, a, b)
    for dt in INTS:  # shifts: every (lhs, rhs) pair of integer dtypes
        for rdt in INTS:
            a, b = cross(edges(dt), edges(rdt))
            for op in (F.SHL, F.SHR):
                add_binary(op, dt, rdt, a, b)
    for dt, op, cs in ((F.F32, F.ADD, (np.float32(-0.0), np.float32(np.inf))), (F.F32, F.SUB, (np.float32(np.inf),)),
                       (F.F32, F.MUL, (np.float32(-0.0), np.float32(2.0 ** -126))), (F.F32, F.DIV, (np.float32(-0.0), np.float32(3.0))),
                       (F.F32, F.REM, (np.float32(-1.5),)), (F.F64, F.DIV, (-0.0,)), (F.F64, F.REM, (2.0 ** -1074,)),
                       (F.I32, F.DIV, (-1,)), (F.I64, F.REM, (-1,)), (F.U8, F.MUL, (255,)), (F.U64, F.SHR, (65,))):
        for c in cs:
            add_binary_const(op, dt, edges(dt), c)
    for dt in INTS + FLOATS:
        for op in (F.NEG, F.ABS) + ((F.NOT,) if dt in INTS else (F.SQRT,)):
            x = edges(dt)
            ELEMS.append(Elem(f"{UNNAME[op]}-{NAME[dt]}", dt, [(dt, x)], lambda v, op=op, dt=dt: L.Node(F.UNARY, dt, op=op, children=(v,)),
                              ref_unary(op, dt, x), np.zeros(len(x), bool)))
    for src in INTS + FLOATS:
        for dst in INTS + FLOATS:
            if src != dst:
                x = edges(src)
                ELEMS.append(Elem(f"cast-{NAME[src]}-{NAME[dst]}", dst, [(src, x)],
                                  lambda v, s=src, d=dst: L.Node(F.UNARY, d, op=F.CAST, src_dtype=s, children=(v,)),
                                  ref_cast(src, dst, x), np.zeros(len(x), bool)))
    # x / 0, x % 0, MIN / -1, MIN % -1: one panicking element at a known position among ordinary ones
    for dt in INTS:
        lo, hi = int_range(dt)
        for op in (F.DIV, F.REM):
            for kind, (p, q) in (("zero", (hi, 0)), ("min-1", (lo, -1))):
                if kind == "min-1" and dt not in SIGNED:
                    continue
                a = np.array([hi, 7, lo, 200 % (hi + 1)] * 6, NPD[dt])
                b = np.array([3, 2, 5, 1] * 6, NPD[dt])
                a[13], b[13] = p, q
                add_binary(op, dt, dt, a, b, tag=f"-panic-{kind}", drop_panics=False)


build_elems()
ELEM_IDS = [e.id for e in ELEMS]
assert len(set(ELEM_IDS)) == len(ELEM_IDS), "case ids must be unique"
assert sum(e.id.startswith("cast-") for e in ELEMS) == 42


# ---- the forms of the evaluator each case runs through -----------------------------------------------------------------------
def _take(x, n):
    return np.resize(np.asarray(x), n)  # the sequence repeated cyclically to n elements


def _vec(slot, n):
    for v in ((8, 4, 1) if slot == 4 else (4, 2, 1)):
        if n % v == 0:
            return v


class Form:
    """One way to collect an Elem: a Subject, the Case that names its route and kernels, and its reference."""

    def __init__(self, elem, name):
        self.elem, self.name = elem, name
        e = elem
        n0 = len(e.want)
        n = -(-n0 // 8) * 8
        if name == "half":
            n += 4 if e.slot == 4 else 2  # 8k + 4 (s32) or 4k + 2 (s64): half the vector width
        if name == "rank2":
            n = max(n, 16)  # at least two rows: the planner drops a length-1 axis
        self.n = n
        idx = np.arange(n) % n0
        self.want, self.werr = e.want[idx], e.werr[idx]
        slot = 8 if name == "s64" else e.slot
        V = _vec(slot, 8 if name == "rank2" else n)
        out_es = F.DTYPE_SIZE[e.out_dt]
        shift = out_es if name == "v1" else 0
        self.shift = shift
        if name == "rank2":
            self.case = Case(f"{e.id}[{name}]", None, None, slot, V, 2, 0, e.depth)
        elif name == "s64":
            self.case = Case(f"{e.id}[{name}]", None, None, 8, V, 1, 0, max(e.depth, 2), stream=True)
        else:  # a signature is built at some vector widths only
            sig = e.sig if any(p["sig"] == e.sig and p["slot"] == slot and p["vec"] == V for p in map(_parse, registry())) else None
            self.case = Case(f"{e.id}[{name}]", None, sig, slot, V, 1, 0, e.depth, stream=True, launch_vec=1 if shift else None)

    def subject(self):
        e, n = self.elem, self.n
        if self.name == "rank2":
            R, Cn = n // 8, 8
            r, c = ax = axes(R, Cn)
            # a transposed operand: output (r, c) reads element c * R + r, so no two axes merge
            leaves = [L.Node(F.LEAF, dt, buf=Storage.from_host(dt, _take(v, n).reshape(R, Cn).T.copy().reshape(-1)), offset=0, stride={r: 1, c: R})
                      for dt, v in e.operands]
            return Subject(e.make(*leaves), ax)
        o, = ax = axes(n)
        leaves = [L.Node(F.LEAF, dt, buf=Storage.from_host(dt, _take(v, n)), offset=0, stride={o: 1}) for dt, v in e.operands]
        root = e.make(*leaves)
        if self.name == "s64":  # the narrow value computed in a 64-bit slot: one run of a tuple whose other run is a u64 IOTA
            return Subject([root, L.Node(F.IOTA, F.U64, offset=0, stride={o: 1})], ax)
        return Subject(root, ax, shift=self.shift)

    def check(self, got, err, what):
        want = [self.want] + ([np.arange(self.n, dtype=np.uint64)] if self.name == "s64" else [])
        check_outputs(self.case, got, err, want, self.werr, what)
        if self.werr.any():
            assert err[0] == F.ERR_ARITH, f"{what}: status {err[0]}"


FORM_NAMES = ("stream", "s64", "half", "v1", "rank2")


def forms(elem):
    return [Form(elem, f) for f in FORM_NAMES if f != "s64" or elem.slot == 4]


# ---- CPU half ----------------------------------------------------------------------------------------------------------------
def test_reference_rules():
    """The reference at hand-checked points, so that a wrong rule cannot hide behind agreeing executors."""
    assert ref_int_binary(F.DIV, F.I32, F.I32, -7, 2) == -3 and ref_int_binary(F.REM, F.I32, F.I32, -7, 2) == -1
    assert ref_int_binary(F.REM, F.I64, F.I64, 7, -2) == 1 and ref_int_binary(F.DIV, F.I64, F.I64, -2 ** 63, 1) == -2 ** 63
    assert ref_int_binary(F.DIV, F.I32, F.I32, -2 ** 31, -1) is PANIC and ref_int_binary(F.REM, F.U8, F.U8, 5, 0) is PANIC
    assert ref_int_binary(F.SHL, F.U8, F.U8, 1, 9) == 2 and ref_int_binary(F.SHL, F.U32, F.I32, 1, -1) == 2 ** 31
    assert ref_int_binary(F.SHR, F.I32, F.U64, -8, 2 ** 32 + 3) == -1 and ref_int_binary(F.SHR, F.U32, F.U8, 2 ** 31, 31) == 1
    assert ref_int_binary(F.SHL, F.U64, F.I32, 3, -1) == 2 ** 63 and ref_int_binary(F.SHR, F.I64, F.I64, -2 ** 63, 64) == -2 ** 63
    assert ref_unary(F.ABS, F.I64, [-2 ** 63]).tolist() == [-2 ** 63] and ref_unary(F.NOT, F.U8, [0]).tolist() == [255]
    assert ref_cast_one(2 ** 60 + 2 ** 36 + 1, F.I64, F.F32) == np.float32(2.0 ** 60 + 2.0 ** 37)
    assert float(np.float32(float(2 ** 60 + 2 ** 36 + 1))) == 2.0 ** 60  # what rounding through f64 first gives
    assert ref_cast_one(2 ** 64 - 2 ** 39 - 1, F.U64, F.F32) == np.float32(2.0 ** 64 - 2.0 ** 40)
    assert ref_cast_one(float("nan"), F.F64, F.I32) == 0 and ref_cast_one(-1e300, F.F64, F.U64) == 0
    assert ref_cast_one(np.float32(2.0 ** 31), F.F32, F.I32) == 2 ** 31 - 1 and ref_cast_one(-0.99, F.F64, F.U8) == 0
    assert ref_cast_one(255.99999999999997, F.F64, F.U8) == 255 and ref_cast_one(2.0 ** 64, F.F64, F.U64) == 2 ** 64 - 1
    assert np.isinf(ref_cast_one(3.4028235677973366e38, F.F64, F.F32))
    assert ref_cast_one(np.nextafter(3.4028235677973366e38, 0), F.F64, F.F32) == np.finfo(np.float32).max
    assert ref_cast_one(2.0 ** -150, F.F64, F.F32) == 0 and ref_cast_one(np.nextafter(2.0 ** -150, 1), F.F64, F.F32) == 2.0 ** -149


@pytest.mark.parametrize("elem", ELEMS, ids=ELEM_IDS)
def test_host_forms(elem):
    """Each form: describe() names the planned route and instantiation, and the host emulator (the library's planner over a
    host build of exec.cuh) under the pre-built route and under COLLECT_NO_STATIC, and the C oracle, equal the reference."""
    for fm in forms(elem):
        s, case = fm.subject(), fm.case
        d = s.describe()
        assert d.startswith(case.route), (case.id, case.route, d)
        assert case.planned + "]" in d or case.planned + "," in d, (case.id, case.planned, d)
        for flags, knob in ((0, "jit=0"), (F.COLLECT_NO_STATIC, "no_static")):
            got, err, ran = s.emu(flags)
            assert ran == case.kernel(knob), f"{case.id} [emu {knob}]: ran {ran}, expected {case.kernel(knob)}"
            fm.check(got, err, f"{case.id} [emu {knob}] on {ran}")
        got, err = s.oracle()
        fm.check(got, err, f"{case.id} (oracle)")


def test_jit_sources_compile():
    """NVRTC compiles the [ops] and [ops+shape] source of every form the GPU half runs through the run-time specialiser."""
    exprs = []
    for e in ELEMS:
        for fm in forms(e):
            if fm.name in ("stream", "s64", "rank2") and (fm.name != "stream" or e.sig is None):
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


# ---- folds at edge values ---------------------------------------------------------------------------------------------------
def seq_fold(op, dt, init, x):
    """`let mut s = init; for v in row { s = s (op) v }` over the last axis of x, one reference step at a time."""
    acc = np.full(x.shape[:-1], init, NPD[dt])
    for k in range(x.shape[-1]):
        acc, err = ref_binary(op, dt, dt, acc.reshape(-1), x[..., k].reshape(-1))
        assert not err.any()
        acc = acc.reshape(x.shape[:-1])
    return acc


def edge_rows(dt, rows, row_len, seed):
    """rows x row_len values drawn from the edge table (each row a different draw)."""
    e = edges(dt)
    return np.random.default_rng(seed).choice(e, rows * row_len).astype(NPD[dt]).reshape(rows, row_len)


class FoldCase:
    """build() -> (subject, want).  A View subject runs through the View API; a Subject (hand-built descriptor) through the C
    ABI with `flags`.  route: what describe() starts with; kernel: the exact last_kernel()."""

    def __init__(self, id, build, route, kernel, flags=0):
        self.id, self.build, self.route, self.kernel, self.flags = id, build, route, kernel, flags

    def __repr__(self):
        return self.id


FOLDS = []
OPS = {F.ADD: P.Add, F.SUB: P.Sub, F.MUL: P.Mul, F.DIV: P.Div, F.REM: P.Rem, F.AND: P.BitAnd, F.OR: P.BitOr, F.XOR: P.BitXor}


def add_fold_rows(op, init, row_len):
    def build():  # k_fold_rows: the row fold's own restatement of the f32 operators (apply_f32)
        x = edge_rows(F.F32, 40, row_len, op * 100 + row_len)
        a = Array.new((usize, usize), x.shape, x.reshape(-1), "f32")
        return fold_rows(a, usize, usize, OPS[op], np.float32(init)), seq_fold(op, F.F32, init, x)
    FOLDS.append(FoldCase(f"rows-f32-{OPNAME[op]}-init{init!r}-{row_len}", build, "fold_rows ", fold_rows_kernel(row_len, False, 0)))


def add_fused(eop, post, c, row_len, init=-0.0):
    def build():  # x (eop) (fold_add(row) (post) c): the fused epilogue
        x = edge_rows(F.F32, 40, row_len, eop * 1000 + post * 10 + row_len)
        a = Array.new((usize, usize), x.shape, x.reshape(-1), "f32")
        f = fold_rows(a, usize, usize, P.Add, np.float32(init)).binary(Scalar(np.float32(c), "f32"), OPS[post])
        g, _ = ref_binary(post, F.F32, F.F32, seq_fold(F.ADD, F.F32, init, x), np.full(40, c, np.float32))
        want, _ = ref_binary(eop, F.F32, F.F32, x.reshape(-1), np.repeat(g, row_len))
        return a.binary(f.iso((usize, ())), OPS[eop]), want
    FOLDS.append(FoldCase(f"fused-f32-{OPNAME[eop]}-post{OPNAME[post]}{c!r}-{row_len}", build, "fold_rows.fused",
                          fold_rows_kernel(row_len, True, 0)))


def add_fold_cols(T, op, init):
    dt = DT[T]

    def build():  # k_fold_cols: a fold over the outer axis of a (13, 6) array
        x = edge_rows(dt, 13, 6, op * 7 + dt)
        a = Array.new((usize, usize), x.shape, x.reshape(-1), T)
        v = fold_rows(a.transpose((), usize, usize, ()).iso((usize, usize)), usize, usize, OPS[op], NPD[dt](init))
        return v, seq_fold(op, dt, init, x.T.copy())
    FOLDS.append(FoldCase(f"cols-{T}-{OPNAME[op]}-init{init!r}", build, "fold_cols", "k_fold_cols"))


SPLIT_EDGES = {F.U8: [0x80, 0xff, 0x7f, 1], F.I32: [-2 ** 31, -1, 0x80, 0xff, 2 ** 31 - 1], F.U32: [2 ** 32 - 1, 2 ** 31, 0x80, 0xff]}


def add_split(src, dst, op, init, n_out):
    def build():  # k_fold_split: a narrow source widened by the cast, folded in the wide slot
        K = SPLIT_MIN_RED + 64
        x = np.resize(np.array(SPLIT_EDGES[src], NPD[src]), n_out * K)
        o, r = ax = axes(n_out, K)
        lf = L.Node(F.LEAF, src, buf=Storage.from_host(src, x), offset=0, stride={o: K, r: 1})
        body = L.Node(F.UNARY, dst, op=F.CAST, src_dtype=src, children=(lf,))
        want = seq_fold(op, dst, init, ref_cast(src, dst, x).reshape(n_out, K))
        return Subject(fold(NAME[dst], op, body, [r], init), [o]), want
    FOLDS.append(FoldCase(f"split-{NAME[src]}-{NAME[dst]}-{OPNAME[op]}-{n_out}", build, "fold_split.runs ",
                          split_kernel(NAME[dst], NAME[src], op, "runs")))


EVAL_SPECIALS = {F.F32: np.array([np.inf, -np.inf, 0.0, -0.0, 1.0, -2.0, 2.0 ** -149, 3.4028235e38], np.float32),
                 F.F64: np.array([np.inf, -np.inf, 0.0, -0.0, 1.0, -2.0, 5e-324, 1.7976931348623157e308], np.float64)}


def add_eval_fold(dt, op):
    slot = F.DTYPE_SIZE[dt]
    flags = F.COLLECT_NO_FASTPATH | F.COLLECT_NO_STATIC

    def build():  # the evaluator's own fold: chains through inf - inf, 0 * inf and x / 0 from a -0.0 init
        x = np.random.default_rng(op * 10 + dt).choice(EVAL_SPECIALS[dt], 37 * 5).astype(NPD[dt]).reshape(37, 5)
        x[0] = (np.inf, -np.inf, 1, 1, 1)
        x[1] = (0.0, np.inf, -0.0, 1, 1)
        x[2] = (-0.0, -0.0, -0.0, -0.0, -0.0)
        o, r = ax = axes(37, 5)
        lf = L.Node(F.LEAF, dt, buf=Storage.from_host(dt, x.reshape(-1)), offset=0, stride={o: 5, r: 1})
        return Subject(fold(NAME[dt], op, lf, [r], -0.0), [o]), seq_fold(op, dt, -0.0, x)
    FOLDS.append(FoldCase(f"eval-{NAME[dt]}-{OPNAME[op]}", build, f"generic.interp s{slot * 8} v1x1 rank=1+1 ",
                          instantiation(None, slot, 1, 2, False, 2), flags))


for row_len in (36, 64):
    for op in (F.ADD, F.SUB, F.MUL, F.DIV, F.REM):
        for init in (-0.0, 1.0):
            add_fold_rows(op, init, row_len)
    for eop in (F.DIV, F.REM, F.SUB):
        for post, c in ((F.DIV, -0.0), (F.DIV, 3.0), (F.REM, 0.75), (F.REM, -0.0)):
            add_fused(eop, post, c, row_len)
for T in ("f64", "i64", "u64"):
    for op, init in ((F.ADD, 1), (F.SUB, -1), (F.MUL, 3)) + (((F.AND, -1), (F.OR, 0), (F.XOR, 2 ** 62)) if T != "f64" else ()):
        add_fold_cols(T, op, init if T != "u64" else init % 2 ** 64)
for src, dst, op, init in ((F.U8, F.U32, F.ADD, 5), (F.U8, F.U64, F.ADD, 0), (F.U8, F.I64, F.XOR, -1), (F.U8, F.I32, F.SUB, 3),
                           (F.I32, F.I64, F.ADD, 0), (F.I32, F.U64, F.OR, 0), (F.I32, F.I64, F.XOR, 0), (F.I32, F.U32, F.MUL, 1),
                           (F.U32, F.U64, F.ADD, 0), (F.U32, F.I64, F.XOR, -1), (F.U32, F.I64, F.AND, -1)):
    for n_out in (1, 3):
        add_split(src, dst, op, init, n_out)
for dt in FLOATS:
    for op in (F.ADD, F.SUB, F.MUL, F.DIV, F.REM):
        add_eval_fold(dt, op)
FOLD_IDS = [c.id for c in FOLDS]
assert len(set(FOLD_IDS)) == len(FOLD_IDS), "case ids must be unique"


@pytest.mark.parametrize("case", FOLDS, ids=FOLD_IDS)
def test_host_folds(case):
    """describe() names the dedicated route; the C oracle (and, for descriptors, the host emulator) equals the reference."""
    s, want = case.build()
    if isinstance(s, Subject):
        d = s.describe(case.flags)
        assert d.startswith(case.route), d
        got, err, ran = s.emu(case.flags)
        assert err is None, err
        assert_same_bits(got[0], want, f"{case.id} (emu on {ran})")
        got, err = s.oracle()
        assert err is None, err
        assert_same_bits(got[0], want, f"{case.id} (oracle)")
    else:
        assert s.describe().startswith(case.route), s.describe()
        assert_same_bits(np.asarray(oracle_collect(s)), want, f"{case.id} (oracle)")
        assert_same_bits(np.asarray(emu_collect(s)), want, f"{case.id} (emu)")


# ---- GPU half ----------------------------------------------------------------------------------------------------------------
NS = F.COLLECT_NO_STATIC
# setting -> {form: the collect flags it runs under}.  In the default setting a rank-1 stream never reaches [ops+shape].
RUNS = {"default": {"stream": (0, NS), "s64": (0, NS), "half": (NS,), "v1": (NS,)},
        "shapes=1": {"rank2": (0,)},
        "jit=0": {"stream": (0,), "rank2": (0,)}}


def run_setting(knob):
    """Every form of every case that `knob` runs, under the setting already in this process's environment (and, in the
    default setting, every fold).  -> the number of collects checked."""
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
            if isinstance(s, Subject):
                got, err, ran = s.gpu(ctx, case.flags)
                assert err is None, (case.id, err)
                got = got[0]
            else:
                got = s.collect(location="device", ctx=ctx).as_ref()
                ran = ctx.last_kernel()
            assert ran == case.kernel, f"{case.id}: ran {ran}, expected {case.kernel}"
            assert_same_bits(np.asarray(got), want, f"{case.id} on {ran}")
            n += 1
    ctx.close()
    return n


def expected_runs(knob):
    n = sum(len(RUNS[knob].get(fm.name, ())) for e in ELEMS for fm in forms(e))
    return n + (len(FOLDS) if knob == "default" else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("knob", list(RUNS))
def test_device_forms(knob):
    """The JIT settings are read once per process, so each runs in a subprocess of its own."""
    code = f"import sys; sys.path.insert(0, 'tests'); import test_value_edges as K; print('ran', K.run_setting({knob!r}))"
    env = dict(os.environ, **KNOBS[knob])
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and f"ran {expected_runs(knob)}" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
