"""Which dedicated kernel serves which shape, and is it right there.

The parity tests compare the GPU with the C oracle over the descriptor the product emits; they check values, not which kernel
produced them, and the `[emu]` twin has no tile transpose, row fold or column walk at all.  Several of those choices are made
at launch time, after `describe()` has spoken (`launch_transpose`: TMA, else the register-staged kernel in vec or scalar form;
`launch_fold_rows`: register or shared-memory form).  A planner or launcher change that moved a shape to another kernel would
keep those tests green and leave the old kernel untested.

So every case here names
  * the planner route `describe()` must report (checked on the CPU),
  * the kernel `Context.last_kernel()` must report after the GPU collect, under the default launch settings and under each
    launch knob that changes it (MDIM_TR_*, MDIM_FOLD_MODE; those are read once per process, so knobs run in a subprocess),
  * a reference computed with numpy from the input arrays alone — no lowering, descriptor or C oracle: `np.transpose(...)`
    for transposes, an explicit left-to-right loop in the element type for folds (wrapping integers in unsigned numpy
    arithmetic), and for f32 sums also an f64 error bound, so that a wrong reference cannot hide behind bit-equality.
On the CPU the references themselves are checked bit for bit against the C oracle at small sizes.
"""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

from helpers import oracle_lib, oracle_collect, assert_same_bits
import multidimension_b200 as P
from multidimension_b200 import usize, Array, Scalar, fold_rows, Add, Sub, Mul, Div, Rem, BitAnd, BitOr, BitXor
from multidimension_b200 import _ffi as F
from multidimension_b200 import lowering as L
from multidimension_b200.runtime import Storage, NP_OF, describe_nodevice

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NP = {"f32": np.float32, "f64": np.float64, "i32": np.int32, "u32": np.uint32, "i64": np.int64, "u64": np.uint64}
UNSIGNED = {np.dtype(np.int32): np.uint32, np.dtype(np.uint32): np.uint32, np.dtype(np.int64): np.uint64, np.dtype(np.uint64): np.uint64}
ORACLE_MAX_ELEMS = 1 << 20  # the CPU half checks the reference against the oracle up to this many input elements

# launch knobs -> environment.  "default" runs in the test process; the others in a subprocess each.
KNOBS = {
    "default": {},
    "tr_tma=0": {"MDIM_TR_TMA": "0"},
    "tr_pipe": {"MDIM_TR_TMA": "0", "MDIM_TR_PIPE": "1"},
    "tr_tile=32x128": {"MDIM_TR_TILE": "32x128"},
    "tr_tile=32x128,tma=0": {"MDIM_TR_TILE": "32x128", "MDIM_TR_TMA": "0"},
    "tr_order=0": {"MDIM_TR_ORDER": "0"},
    "tr_order=1": {"MDIM_TR_ORDER": "1"},
    "tr_order=1,tma=0": {"MDIM_TR_ORDER": "1", "MDIM_TR_TMA": "0"},
    "fold_mode=1": {"MDIM_FOLD_MODE": "1"},
    "fold_mode=2": {"MDIM_FOLD_MODE": "2"},
}
TRANSPOSE_KNOBS = [k for k in KNOBS if k.startswith("tr_")]
FOLD_KNOBS = ["fold_mode=1", "fold_mode=2"]


# ---- references: numpy, from the input arrays -------------------------------------------------------------------------------
def _apply(op, a, b):
    """One step of `s = s (op) x` elementwise in the arrays' own type; integers wrap (computed unsigned)."""
    dt = np.result_type(a, b)
    if dt.kind in "iu":
        u = UNSIGNED[dt]
        a, b = np.asarray(a).astype(dt).view(u), np.asarray(b).astype(dt).view(u)
    f = {Add: np.add, Sub: np.subtract, Mul: np.multiply, Div: np.divide, Rem: np.fmod,
         BitAnd: np.bitwise_and, BitOr: np.bitwise_or, BitXor: np.bitwise_xor}[op]
    with np.errstate(all="ignore"):
        r = f(a, b)
    return r.view(dt) if dt.kind in "iu" else r


def seq_fold(x, op, init, axis):
    """The reference's fold: `let mut s = init; for x in row { s = s (op) x }`, strictly in index order along `axis`."""
    x = np.moveaxis(x, axis, -1)
    acc = np.full(x.shape[:-1], np.array(init).astype(x.dtype))  # integer inits wrap into the type, as the descriptor does
    for k in range(x.shape[-1]):
        acc = _apply(op, acc, x[..., k])
    return acc


def f32_sum_bound(got, x, init, axis):
    """|got - S| <= (n + 1) 2^-24 sum|.|, S the exact (f64) sum of init and the row: a left-to-right f32 sum stays that close."""
    x64 = np.moveaxis(x.astype(np.float64), axis, -1)
    with np.errstate(invalid="ignore"):
        exact = x64.sum(axis=-1) + float(init)
        mag = np.abs(x64).sum(axis=-1) + abs(float(init))
    got = np.asarray(got, dtype=np.float64).reshape(exact.shape)
    fin = np.isfinite(exact) & np.isfinite(mag)
    n = x64.shape[-1]
    err = np.abs(got[fin] - exact[fin])
    assert np.all(err <= (n + 1) * 2.0 ** -24 * mag[fin]), f"f32 sum off its f64 bound by up to {np.max(err - (n + 1) * 2.0 ** -24 * mag[fin])}"


def rand(rng, T, n, lo=-4.0, hi=4.0):
    if T in ("f32", "f64"):
        return rng.uniform(lo, hi, n).astype(NP[T])
    info = np.iinfo(NP[T])
    return rng.integers(info.min, info.max, n, dtype=NP[T], endpoint=True)


def with_special_rows(x2d, axis):
    """Lines (along `axis`) of all -0.0, and with NaN, +Inf, -Inf and +Inf beside -Inf, at the front of a float array."""
    x = np.moveaxis(x2d.copy(), axis, -1)
    x[0] = -0.0
    x[1, x.shape[-1] // 2] = np.nan
    x[2, -1] = np.inf
    x[3, 0] = -np.inf
    x[4, 0], x[4, -1] = np.inf, -np.inf
    return np.moveaxis(x, -1, axis)


# ---- a raw descriptor the View API cannot spell: a LEAF with a negative row stride --------------------------------------------
class RawLeafTranspose:
    """out[a, b] = src[offset + b * stride_b + a]: one LEAF over axes (A, B), A unit-stride, emitted by hand.  `Reversed`
    lowers to IOTA, not to a strided leaf, so a negative source row stride exists only at the C ABI."""

    def __init__(self, src, len_a, len_b, offset, stride_b):
        self.offset, self.stride_b = offset, stride_b
        self.axes = [L.Axis(len_a), L.Axis(len_b)]
        self.storage = Storage.from_host({np.float32: F.F32, np.float64: F.F64, np.uint64: F.U64}[src.dtype.type], src)

    def node(self):
        return L.Node(F.LEAF, self.storage.dtype, buf=self.storage, offset=self.offset, stride={self.axes[0]: 1, self.axes[1]: self.stride_b})

    def describe(self):
        st, text = describe_nodevice(L.emit(self.node(), self.axes, "any").expr)
        return text if st == F.OK else f"error {st}: {text}"

    def oracle(self):
        em = L.emit(self.node(), self.axes, "host")
        out = np.zeros(em.out_len, dtype=NP_OF[em.out_dtype])
        info = F.ErrorInfo()
        assert oracle_lib().mdim_oracle_collect(C.byref(em.expr), out.ctypes.data, C.byref(info)) == F.OK, info.message
        return out

    def gpu(self, ctx):
        self.storage.ensure_device(ctx)
        em = L.emit(self.node(), self.axes, "device")
        out = Storage.device(ctx, em.out_dtype, em.out_len)
        ctx.collect(em.expr, out.dptr)
        return out.to_numpy()


def oracle(subject):
    return subject.oracle() if isinstance(subject, RawLeafTranspose) else oracle_collect(subject)


def gpu_collect(subject, ctx):
    if isinstance(subject, RawLeafTranspose):
        return subject.gpu(ctx)
    return subject.collect(location="device", ctx=ctx).as_ref()


# ---- the case table ---------------------------------------------------------------------------------------------------------------
class Case:
    """`build(sm_count)` -> (subject, want, extra check or None); `route`: what describe() starts with; `kernels`: knob -> the
    exact last_kernel() string (knobs that do not apply to the case are absent)."""

    def __init__(self, group, id, build, route, kernels, n_in):
        self.group, self.id, self.build, self.route, self.kernels, self.n_in = group, id, build, route, kernels, n_in

    def __repr__(self):
        return self.id


CASES = []


def _ix(k):
    """An index type of k usize axes (tuples have arity <= 3, so longer ones nest)."""
    return () if k == 0 else usize if k == 1 else (usize,) * k if k <= 3 else (usize, _ix(k - 1))


def permuted(a, n, perm):
    """np.transpose(x, perm) of the rank-n Array `a`, spelled as Transposes of neighbouring axes."""
    v, cur = a, list(range(n))
    for i, ax in enumerate(perm):
        j = cur.index(ax)
        while j > i:  # Transpose<I, X, Y, J> swaps Y (position j - 1) and X (position j)
            v = v.transpose(_ix(j - 1), usize, usize, _ix(n - j - 1)).iso(_ix(n))
            cur[j - 1], cur[j] = cur[j], cur[j - 1]
            j -= 1
    return v


def transpose_kernels(base):
    """The kernel under every transpose knob, from the one that runs by default.  TMA takes every case whose strides and base
    are 16-byte aligned with <= 3 batch axes; without it the register-staged kernel loads 16 bytes at a time where the case
    is aligned (vec), else element by element (scalar); MDIM_TR_PIPE=1 swaps the aligned register-staged kernel for the
    cp.async ring (default tile only)."""
    out = {}
    for knob in ["default"] + TRANSPOSE_KNOBS:
        env = KNOBS[knob]
        k = base
        if base != "k_transpose<regs,scalar>":
            if base == "k_transpose_tma" and env.get("MDIM_TR_TMA") == "0":
                k = "k_transpose<regs,vec>"
            if k == "k_transpose<regs,vec>" and env.get("MDIM_TR_PIPE") == "1" and "MDIM_TR_TILE" not in env:
                k = "k_transpose_pipe"
        out[knob] = k
    return out


def add_transpose(id, T, shape, perm, kernel, pin=None):
    """np.transpose of a seeded Array of `shape` by `perm`; pin = i: the Array has one more (outer) axis, pinned at i by `row`."""
    n = len(shape)
    full = ((pin + 2,) if pin is not None else ()) + tuple(shape)

    def build(sm_count):
        rng = np.random.default_rng(zlib.crc32(f"{id}-{T}".encode()))
        x = rand(rng, T, int(np.prod(full))).reshape(full)
        a = Array.new(_ix(len(full)), full, x.reshape(-1), T)
        if pin is not None:
            a, x = a.row(usize, _ix(n), pin), x[pin]
        return permuted(a, n, perm), np.transpose(x, perm).copy().reshape(-1), None
    CASES.append(Case("transpose", f"transpose-{id}-{T}", build, "transpose.tile", transpose_kernels(kernel), int(np.prod(full))))


def add_raw_transpose(id, T, len_a, len_b, pitch, pad):
    """Source rows `pitch` elements apart, walked from the last row backwards (row stride -pitch), starting `pad` elements in."""
    def build(sm_count):
        rng = np.random.default_rng(len_a * 1000 + len_b)
        src = rand(rng, T, pitch * len_b + pad)
        offset = (len_b - 1) * pitch + pad
        want = np.array([[src[offset + b * -pitch + a] for b in range(len_b)] for a in range(len_a)], dtype=src.dtype).reshape(-1)
        return RawLeafTranspose(src, len_a, len_b, offset, -pitch), want, None
    CASES.append(Case("transpose", f"transpose-{id}-{T}", build, "transpose.tile", transpose_kernels("k_transpose<regs,vec>"), pitch * len_b + pad))


def _tr_base(shape, es):
    """2-D: TMA when both row pitches are whole 16-byte chunks, else the scalar register-staged kernel."""
    R, Cc = shape
    return "k_transpose_tma" if (R * es) % 16 == 0 and (Cc * es) % 16 == 0 else "k_transpose<regs,scalar>"


for T in ("f32", "f64", "u64"):
    es = np.dtype(NP[T]).itemsize
    for shape in [(16, 16), (64, 64), (63, 64), (65, 64), (64, 63), (64, 65), (63, 65), (100, 36), (130, 68)]:
        add_transpose(f"{shape[0]}x{shape[1]}", T, shape, (1, 0), _tr_base(shape, es))
    add_transpose("pinned-row-64x36", T, (64, 36), (1, 0), "k_transpose_tma", pin=1)              # non-zero, 16-byte-aligned offset
    add_transpose("batch1-3x40x68", T, (3, 40, 68), (0, 2, 1), "k_transpose_tma")
    add_transpose("batch2-3x2x20x36", T, (3, 2, 20, 36), (1, 0, 3, 2), "k_transpose_tma")         # batch axes swapped: no merge
    add_transpose("batch3-2x3x2x20x36", T, (2, 3, 2, 20, 36), (2, 1, 0, 4, 3), "k_transpose_tma")
    # four batch axes: beyond a rank-5 tensor map -> the register-staged kernel, 16 bytes at a time
    add_transpose("batch4-2x3x2x3x20x36", T, (2, 3, 2, 3, 20, 36), (1, 0, 3, 2, 5, 4), "k_transpose<regs,vec>")
    add_raw_transpose("negative-row-stride", T, 36, 20, 40, 16 // es)
add_transpose("pitch-not-16B-64x66", "f32", (64, 66), (1, 0), "k_transpose<regs,scalar>")        # 264-byte rows, 4-byte-aligned output
add_transpose("pitch-not-16B-30x64", "f32", (30, 64), (1, 0), "k_transpose<regs,scalar>")        # 120-byte output rows


# ---- fold over the last axis: k_fold_rows / k_fold_regs --------------------------------------------------------------------------
K_FOLD_THREADS = 256        # k_fold.cu / kernels.cuh: kFoldThreads
K_FOLD_GRID_MULT = 16       # k_fold.cu: CTAs queued per SM (MDIM_FOLD_GRID_MULT unset)
K_FOLD_SMEM = 227 * 1024 - 512   # k_fold.cu: the opt-in shared memory of an SM less the mbarriers (kBarBytes)


def fold_rows_kernel(row_len, fused, mode):
    """launch_fold_rows: the register form for row_len = 32 L (L a power of two <= 32) when asked for (MDIM_FOLD_MODE=2) or by
    default for the fused form; the shared-memory / TMA form otherwise."""
    L_ = row_len // 32
    regs_ok = row_len % 32 == 0 and 1 <= L_ <= 32 and (L_ & (L_ - 1)) == 0
    want_regs = mode == 2 or (mode == 0 and fused)
    return "k_fold_regs" if want_regs and regs_ok else "k_fold_rows"


def rows_past_ring_wrap(row_len, sm_count):
    """Rows enough that every warp of k_fold_rows walks more than 2 x stages items, so each mbarrier's parity wraps: the
    launcher's sizing (fold only, dense rows <= 512) restated."""
    tile = 32 * row_len * 4
    max_tiles = max(1, K_FOLD_SMEM // tile)
    n_warps = min(K_FOLD_THREADS // 32, max_tiles)
    stages = max(1, min(4, max_tiles // n_warps))
    total_warps = sm_count * K_FOLD_GRID_MULT * n_warps
    return 32 * total_warps * (2 * stages + 1)


def fold_kernels(row_len, fused):
    return {"default": fold_rows_kernel(row_len, fused, 0), "fold_mode=1": fold_rows_kernel(row_len, fused, 1),
            "fold_mode=2": fold_rows_kernel(row_len, fused, 2)}


def add_fold_rows(T, rows, row_len, op, init, lo=-4.0, hi=4.0, special=False, big=False):
    name = op.name

    def build(sm_count):
        n_rows = rows_past_ring_wrap(row_len, sm_count) if big else rows
        rng = np.random.default_rng(n_rows * 7 + row_len)
        x = rand(rng, T, n_rows * row_len, lo, hi).reshape(n_rows, row_len)
        if special:
            x = with_special_rows(x, 1)
        a = Array.new((usize, usize), (n_rows, row_len), x.reshape(-1), T)
        want = seq_fold(x, op, init, 1)
        extra = (lambda got: f32_sum_bound(got, x, init, 1)) if (T == "f32" and op is Add) else None
        return fold_rows(a, usize, usize, op, init), want, extra
    rid = "wrap" if big else rows
    CASES.append(Case("fold_rows", f"fold-{T}-{name}-{rid}x{row_len}{'-special' if special else ''}", build, "fold_rows ",
                      fold_kernels(row_len, False), (rows_past_ring_wrap(row_len, 1) if big else rows) * row_len))


def add_fused(T, rows, row_len, eop, post, c=None, lo=-4.0, hi=4.0, special=False, init=0):
    """x (eop) g[row] with g = fold(row) [post c]: the fused epilogue (BASELINE config 4 is f32, Add fold, Sub, post Div)."""
    en, pn = eop.name, (post.name if post else "none")

    def build(sm_count):
        rng = np.random.default_rng(rows * 31 + row_len)
        x = rand(rng, T, rows * row_len, lo, hi).reshape(rows, row_len)
        if special:
            x = with_special_rows(x, 1)
        a = Array.new((usize, usize), (rows, row_len), x.reshape(-1), T)
        f = fold_rows(a, usize, usize, Add, init)
        g = seq_fold(x, Add, init, 1)
        if post is not None:
            f = f.binary(Scalar(c, T), post)
            g = _apply(post, g, np.array(c, dtype=NP[T]))
        return a.binary(f.iso((usize, ())), eop), _apply(eop, x, g[:, None]).reshape(-1), None
    CASES.append(Case("fold_rows", f"fused-{T}-{en}-post{pn}-{rows}x{row_len}{'-special' if special else ''}", build, "fold_rows.fused",
                      fold_kernels(row_len, True), rows * row_len))


# fold only: the f32 sum at every row length (minimum, skew 0 / 1, the largest dense tile, the first chunked length, a short last
# chunk) and row count (the fewest, around a 32-row tile, 2^k + 1).  The fewest is 2: the planner drops a length-1 axis, so a
# single row is a full reduction, which the evaluator serves.
ROW_LENS = [8, 12, 28, 32, 36, 128, 508, 512, 516, 1028]
for row_len in ROW_LENS:
    for rows in (2, 31, 32, 33, 257):
        add_fold_rows("f32", rows, row_len, Add, np.float32(0.25), 0.0, 1.0)
for row_len in (8, 36, 128, 516):
    for T in ("i32", "u32"):
        for op, init in ((Add, 7), (Sub, -3), (Mul, 3), (BitAnd, -1), (BitOr, 0), (BitXor, 0x5a5a5a5a)):
            add_fold_rows(T, 33, row_len, op, init)
    add_fold_rows("f32", 33, row_len, Sub, np.float32(3))
    add_fold_rows("f32", 33, row_len, Mul, np.float32(1), 0.9, 1.1)
    add_fold_rows("f32", 33, row_len, Div, np.float32(1e10), 0.9, 1.1)
    add_fold_rows("f32", 33, row_len, Rem, np.float32(1e6), 1.0, 100.0)
add_fold_rows("f32", None, 8, Add, np.float32(0), 0.0, 1.0, big=True)   # each warp's mbarrier ring wraps more than twice
add_fold_rows("u32", None, 8, Add, 0, big=True)
for row_len in (32, 36, 516):
    add_fold_rows("f32", 40, row_len, Add, np.float32(-0.0), special=True)
    add_fold_rows("f32", 40, row_len, Mul, np.float32(-0.0), 0.9, 1.1, special=True)

# fused: every epilogue operator and post operator, on both kernels; the register form at every width it has
for row_len in (128, 36):
    for eop in (Sub, Add, Mul, Div):
        for post, c in ((None, None), (Div, 128.0), (Mul, 0.5)):
            add_fused("f32", 37, row_len, eop, post, c)
for L_ in range(1, 17):
    if L_ == 4:
        continue  # row_len 128: the grid above
    add_fused("f32", 37, 32 * L_, Sub, None)
    add_fused("f32", 37, 32 * L_, Mul, Div, 3.0, 0.5, 2.0)
for rows in (2, 37):
    add_fused("f32", rows, 96, Sub, Div, 96.0)
    add_fused("f32", rows, 96, Add, None)
for T, row_len in (("i32", 64), ("u32", 36)):
    for eop in (Add, Sub, Mul, BitXor):
        for post, c in ((None, None), (Mul, 3)):
            add_fused(T, 37, row_len, eop, post, c)
for row_len in (64, 36):
    add_fused("f32", 40, row_len, Sub, None, special=True, init=np.float32(-0.0))
    add_fused("f32", 40, row_len, Mul, Div, 7.0, special=True, init=np.float32(-0.0))


# ---- fold over an outer axis: k_fold_cols -----------------------------------------------------------------------------------------
def add_fold_cols(id, T, n_rows, cols, op, init, lo=-4.0, hi=4.0, window=None, batch=None, special=False):
    """A fold over the OUTER axis of an (n_rows, cols) Array — or of a column window: the middle index of an (n_rows, window, cols)
    Array pinned at 1, so rows are window * cols apart — or over the middle axis of a (batch, n_rows, cols) Array."""
    name = op.name

    def build(sm_count):
        rng = np.random.default_rng(n_rows * 13 + cols)
        if batch is not None:
            x = rand(rng, T, batch * n_rows * cols, lo, hi).reshape(batch, n_rows, cols)
            a = Array.new((usize, usize, usize), x.shape, x.reshape(-1), T)
            v = fold_rows(a.transpose(usize, usize, usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, op, init)
            return v, seq_fold(x, op, init, 1).reshape(-1), None
        if window is not None:
            xw = rand(rng, T, n_rows * window * cols, lo, hi).reshape(n_rows, window, cols)
            a = Array.new((usize, usize, usize), xw.shape, xw.reshape(-1), T)
            src, x = a.transpose((), usize, usize, usize).iso((usize, usize, usize)).row(usize, (usize, usize), 1), xw[:, 1, :]
        else:
            x = rand(rng, T, n_rows * cols, lo, hi).reshape(n_rows, cols)
            if special:
                x = with_special_rows(x, 0)
            src = Array.new((usize, usize), x.shape, x.reshape(-1), T)
        v = fold_rows(src.transpose((), usize, usize, ()).iso((usize, usize)), usize, usize, op, init)
        extra = (lambda got: f32_sum_bound(got, x, init, 0)) if (T == "f32" and op is Add) else None
        return v, seq_fold(x, op, init, 0), extra
    n_in = (batch or 1) * n_rows * (window or 1) * cols
    CASES.append(Case("fold_cols", f"cols-{id}-{T}-{name}-{n_rows}x{cols}", build, "fold_cols", {"default": "k_fold_cols"}, n_in))


# around the walk's 12-row window; the fewest rows is 2 (a length-1 folded axis is dropped: a plain copy on the evaluator)
for n_rows in (2, 11, 12, 13, 23, 24, 25, 1000):
    add_fold_cols("half-group", "f32", n_rows, 36, Add, np.float32(0.5), 0.0, 1.0)   # 144-byte rows: 4.5 32-byte groups, 16-byte pitch
    add_fold_cols("aligned", "f32", n_rows, 64, Add, np.float32(0.5), 0.0, 1.0)      # 256-byte rows and pitch: 256-bit loads
for n_rows in (13, 25):
    add_fold_cols("window32", "f32", n_rows, 64, Sub, np.float32(1), window=3)       # pitch 768 bytes (32-byte aligned)
    add_fold_cols("window16", "f32", n_rows, 36, Add, np.float32(1), window=3)       # pitch 432 bytes (16-byte aligned only)
    for T in ("f64", "i64", "u64"):
        for op, init in ((Sub, 5), (Mul, 3)):
            lo, hi = (0.9, 1.1) if op is Mul else (-4.0, 4.0)
            add_fold_cols("es8", T, n_rows, 6, op, NP[T](init), lo, hi)               # 48-byte rows: 1.5 groups
    for T in ("i32", "u32"):
        add_fold_cols("es4", T, n_rows, 12, BitXor, NP[T](0))
        add_fold_cols("es4", T, n_rows, 12, Mul, NP[T](3))
    add_fold_cols("special", "f32", n_rows, 36, Add, np.float32(-0.0), special=True)
add_fold_cols("batch-half", "f32", 13, 4, Add, np.float32(0.5), batch=3)             # one half group per batch, 16-byte batch pitch
add_fold_cols("batch-1.5", "f32", 25, 12, Add, np.float32(0.5), batch=5)
add_fold_cols("batch-4.5", "f32", 24, 36, Sub, np.float32(0.5), batch=2)

CASE_IDS = [c.id for c in CASES]
assert len(set(CASE_IDS)) == len(CASE_IDS), "case ids must be unique"


# ---- CPU half: the planner's route and the references ------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_planned_route_and_reference(case):
    """describe() names the route the GPU case expects, and the numpy reference equals the C oracle bit for bit (small cases:
    the wrapped-ring fold is built for one SM here, which keeps its reference code and shrinks it)."""
    subject, want, extra = case.build(1)
    assert subject.describe().startswith(case.route), subject.describe()
    if case.n_in <= ORACLE_MAX_ELEMS:
        assert_same_bits(want, oracle(subject), case.id + " (reference vs oracle)")
        if extra is not None:
            extra(want)


def test_four_batch_axes_stay_four():
    """The rank-6 permutation keeps 4 batch axes after the planner merges neighbours (the evaluator's describe shows the
    canonical rank): more than a rank-5 tensor map holds, which is what sends it to the register-staged kernel."""
    for case in CASES:
        if "batch4" in case.id:
            subject, _, _ = case.build(1)
            assert " rank=6+0 " in subject.describe(F.COLLECT_NO_FASTPATH), subject.describe(F.COLLECT_NO_FASTPATH)


def test_case_table_names_every_dedicated_kernel():
    named = {k for c in CASES for k in c.kernels.values()}
    for k in ("k_transpose_tma", "k_transpose<regs,vec>", "k_transpose<regs,scalar>", "k_transpose_pipe", "k_fold_rows", "k_fold_regs", "k_fold_cols"):
        assert k in named, k


# ---- GPU half ------------------------------------------------------------------------------------------------------------------------
def run_case(case, ctx, knob):
    subject, want, extra = case.build(ctx.device_info()["sm_count"])  # the SM count launch_fold_rows sizes its grid with
    got = gpu_collect(subject, ctx)
    ran = ctx.last_kernel()
    assert ran == case.kernels[knob], f"{case.id} [{knob}]: ran {ran}, expected {case.kernels[knob]} ({subject.describe()})"
    assert_same_bits(got, want, f"{case.id} [{knob}] on {ran}")
    if extra is not None:
        extra(got)


def run_group(group, knob):
    """Every case of `group` under the launch knob already set in this process's environment (see test_launch_knobs)."""
    ctx = P.Context(0)
    n = 0
    for case in CASES:
        if case.group == group and knob in case.kernels:
            run_case(case, ctx, knob)
            n += 1
    ctx.close()
    return n


_ctx = []


@pytest.fixture
def gpu_ctx():
    if not _ctx:
        _ctx.append(P.Context(0))
    return _ctx[0]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_kernel_route(case, gpu_ctx):
    run_case(case, gpu_ctx, "default")


@pytest.mark.gpu
@pytest.mark.parametrize("knob", TRANSPOSE_KNOBS + FOLD_KNOBS)
def test_launch_knobs(knob):
    """The launch knobs are read once per process: each runs in a subprocess over the cases it re-routes (every transpose for
    MDIM_TR_*, every last-axis fold for MDIM_FOLD_MODE), asserting the kernel each case must then run on."""
    group = "transpose" if knob.startswith("tr_") else "fold_rows"
    code = (f"import sys; sys.path.insert(0, 'tests'); import test_kernel_routes as K; "
            f"print('ran', K.run_group({group!r}, {knob!r}))")
    env = dict(os.environ, **KNOBS[knob])
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=ROOT)
    want = sum(1 for c in CASES if c.group == group and knob in c.kernels)
    assert r.returncode == 0 and f"ran {want}" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
