"""The few-output integer fold (`k_fold_split`): which folds take it, which keep their route, and is it right there.

An integer fold whose operator is wrapping Add, Sub, Mul, BitAnd, BitOr or BitXor gives the same bits in any order of
combination, so a fold with at most SPLIT_MAX_OUTS outputs and at least SPLIT_MIN_RED reduced elements per output is cut into
chunks spread over the whole GPU (at most SPLIT_MAX_COLS outputs when they are columns).  Every case here names
  * the planner route `describe()` must report (checked on the CPU),
  * the exact `last_kernel()` after the GPU collect (`None`: a case that must keep a route other than the split fold),
  * a reference computed with numpy from the input array: the leaf's elements gathered by index arithmetic, cast with
    `astype` (Rust `as` for integers) and reduced in the element type through unsigned views (numpy would otherwise promote
    small integer types).  On the CPU the reference equals the C oracle's sequential fold bit for bit.
The cases are hand-built descriptors (the C ABI), so that every stride, offset and alignment is explicit.
"""
import zlib

import numpy as np
import pytest

from helpers import assert_same_bits
import multidimension_b200 as P
from multidimension_b200 import _ffi as F
from multidimension_b200 import lowering as L
from multidimension_b200.runtime import Storage
from test_eval_routes import Subject, fold, axes, DT, NPD

SPLIT_MAX_OUTS = 4096       # program.hpp: kSplitMaxOuts
SPLIT_MAX_COLS = 1024       # program.hpp: kSplitMaxCols
SPLIT_MIN_RED = 1 << 12     # program.hpp: kSplitMinRed
ORACLE_MAX_ELEMS = 1 << 22  # the CPU half checks the reference against the oracle up to this many gathered elements
NPT = {"u8": np.uint8, "i32": np.int32, "u32": np.uint32, "i64": np.int64, "u64": np.uint64, "f32": np.float32, "f64": np.float64}
UNS = {1: np.uint8, 4: np.uint32, 8: np.uint64}
OPNAME = {F.ADD: "add", F.SUB: "add", F.MUL: "mul", F.AND: "and", F.OR: "or", F.XOR: "xor"}
UFUNC = {F.ADD: np.add, F.SUB: np.add, F.MUL: np.multiply, F.AND: np.bitwise_and, F.OR: np.bitwise_or, F.XOR: np.bitwise_xor}


def values(key, T, n, kind="rand"):
    rng = np.random.default_rng(zlib.crc32(key.encode()))
    if kind == "bool":
        return (rng.random(n) < 0.5).astype(np.uint8)
    if kind == "ones":
        return np.ones(n, NPT[T])
    if kind == "threes":  # a few 3s among 1s: the product is 3^k, wrapping once k is large
        x = np.ones(n, NPT[T])
        x[rng.integers(0, n, 45)] = 3
        return x
    if T in ("f32", "f64"):
        return rng.uniform(-4, 4, n).astype(NPT[T])
    if kind == "small":
        return rng.integers(-3, 4, n).astype(NPT[T])
    info = np.iinfo(NPT[T])
    return rng.integers(info.min, info.max, n, dtype=NPT[T], endpoint=True)


def reference(x, T_src, T, op, init, offset, out, red):
    """out / red: lists of (length, stride).  -> the folded outputs in row-major output order, dtype T."""
    es = x.itemsize
    v = np.lib.stride_tricks.as_strided(x[offset:], shape=[n for n, _ in out + red], strides=[s * es for _, s in out + red], writeable=False)
    u = UNS[np.dtype(NPT[T]).itemsize]
    i = np.array(int(init) & ((1 << (8 * np.dtype(u).itemsize)) - 1), dtype=u)
    res = []
    for o in np.ndindex(*[n for n, _ in out]):
        g = np.ascontiguousarray(v[o]).reshape(-1).astype(NPT[T]).view(u)
        p = UFUNC[op].reduce(g, dtype=u)
        with np.errstate(over="ignore"):
            res.append((i - p) if op == F.SUB else UFUNC[op](i, p))
    return np.array(res, dtype=u).view(NPT[T])


class Case:
    def __init__(self, id, build, route, kernel, n_elems, host=False):
        self.id, self.build, self.route, self.kernel, self.n_elems, self.host = id, build, route, kernel, n_elems, host

    def __repr__(self):
        return self.id


CASES = []


def split_kernel(T, T_src, op, layout):
    slot = 64 if np.dtype(NPT[T]).itemsize == 8 else 32
    return f"k_fold_split<u{slot},src=u{np.dtype(NPT[T_src]).itemsize * 8},{OPNAME[op]},{layout}>"


def add(id, T, op, init, out, red, *, T_src=None, pad=0, offset=0, kind="rand", route=None, kernel="auto", shift=0, init_view=False,
        body="leaf", host=False):
    """A fold over one leaf of T_src (cast to T when they differ).  out / red: lists of (length, stride) in elements of T_src; the
    buffer holds every element the view reaches from `offset`, plus `pad`.  route: the describe() prefix (default: the split fold,
    runs when the reduction is unit-stride after reordering, else cols)."""
    T_src = T_src or T
    n_elems = int(np.prod([n for n, _ in out + red], dtype=np.int64))
    if route is None:
        strides = sorted(abs(s) for _, s in red)
        route = "fold_split.runs " if strides[0] == 1 else "fold_split.cols "
    if kernel == "auto":
        kernel = split_kernel(T, T_src, op, route.split(".")[1].strip()) if route.startswith("fold_split") else None

    def build():
        reach_lo = offset + sum(min(0, (n - 1) * s) for n, s in out + red)
        reach_hi = offset + sum(max(0, (n - 1) * s) for n, s in out + red)
        assert reach_lo >= 0, id
        x = values(id, T_src, reach_hi + 1 + pad, kind)
        buf = Storage.from_host(DT[T_src], x)
        ax = axes(*[n for n, _ in out + red])
        lf = L.Node(F.LEAF, DT[T_src], buf=buf, offset=offset, stride={a: s for a, (_, s) in zip(ax, out + red) if s})
        b = lf if T_src == T else L.Node(F.UNARY, DT[T], op=F.CAST, src_dtype=DT[T_src], children=(lf,))
        if body == "gather":  # g[k % 4] over the reduction index k: a gathered body stays on the evaluator
            b = L.Node(F.GATHER, DT[T], buf=Storage.from_host(DT[T], values(id + "g", T, 4)),
                       children=(L.Node(F.BINARY, F.U64, op=F.REM, children=(L.Node(F.IOTA, F.U64, offset=0, stride={ax[-1]: 1}), L.Node(F.CONST, F.U64, imm=4))),),
                       gstride=(1,), bound=(4,))
        red_ax = ax[len(out):]
        if init_view:
            iv = L.Node(F.CONST, DT[T], imm=init)
            f = L.Node(F.FOLD, DT[T], op=op, children=(iv, b), red_axes=tuple(red_ax), imm=0)
        else:
            f = fold(T, op, b, red_ax, init)
        want = None
        if body == "leaf" and op in UFUNC and T not in ("f32", "f64"):  # the others: the C oracle's fold is the reference
            want = reference(x, T_src, T, op, init, offset, out, red)
        return Subject(f, ax[:len(out)], shift=shift), want
    CASES.append(Case(id, build, route, kernel, n_elems, host))


K, Cmax, Ccols = SPLIT_MIN_RED, SPLIT_MAX_OUTS, SPLIT_MAX_COLS

# ---- route edges: outputs 1, 2, 3, C, C + 1; reduction K - 1, K; each other condition failing once ------------------------------
for n_out in (1, 2, 3):
    add(f"edge-runs-outs{n_out}", "u32", F.ADD, 5, [(n_out, K + 3)], [(K, 1)])
add(f"edge-runs-outsC", "u8", F.XOR, 5, [(Cmax, 1)], [(K, 1)])                 # overlapping runs: output o reads [o, o + K)
add(f"edge-runs-outsC+1", "u8", F.XOR, 5, [(Cmax + 1, 1)], [(K, 1)], route="generic.")     # too many outputs
add(f"edge-cols-outsC", "u8", F.ADD, 5, [(Ccols, 1)], [(K, Ccols)])
add(f"edge-cols-outsC+1", "u32", F.ADD, 5, [(Ccols + 4, 1)], [(K, Ccols + 4)], route="fold_cols ")
add(f"edge-cols-batch-outsC+1", "u8", F.ADD, 5, [(3, K * 400), (342, 1)], [(K, 400)], route="generic.")  # 1026 outputs in 3 batches
add(f"edge-red-K-1", "u64", F.ADD, 1, [], [(K - 1, 1)], route="generic.interp")
add(f"edge-red-K", "u64", F.ADD, 1, [], [(K, 1)])
add(f"edge-rows-K-1", "u32", F.ADD, 1, [(4, K - 1)], [(K - 1, 1)], route="generic.interp")           # row_len % 4 != 0: not fold_rows
add(f"edge-rows-K-4", "u32", F.ADD, 1, [(4, K - 4)], [(K - 4, 1)], route="fold_rows ")
add(f"edge-cols-K-1", "u32", F.ADD, 1, [(4, 1)], [(K - 1, 4)], route="fold_cols ")
add(f"keeps-f32", "f32", F.ADD, 0.5, [], [(K, 1)], route="generic.")
add(f"keeps-f64-cols", "f64", F.ADD, 0.5, [(4, 1)], [(K, 4)], route="fold_cols ")
add(f"keeps-div", "u32", F.DIV, 7, [], [(K, 1)], kind="ones", route="generic.")
add(f"keeps-shl", "u32", F.SHL, 1, [], [(K, 1)], kind="ones", route="generic.")
add(f"keeps-init-view", "u32", F.ADD, 5, [], [(K, 1)], init_view=True, route="generic.")
add(f"keeps-gather", "u64", F.ADD, 5, [], [(K, 1)], body="gather", route="generic.")
add(f"keeps-stride0-red", "u32", F.ADD, 5, [], [(K, 0)], route="generic.")

# ---- sizes and layouts ------------------------------------------------------------------------------------------------------------
# One output of n elements is cut into min(3 x SMs, n x es / 32 KiB) chunks of a multiple of 32 elements (k_fold_split.cu): e
# elements of a type are one such chunk.  One chunk, two exactly, two with a short tail, a chunk less one, several with an odd tail.
CHUNK = 32 * 1024
for T in ("u8", "u32", "u64"):
    e = CHUNK // np.dtype(NPT[T]).itemsize
    for n in (max(K, e // 2), 2 * e - 1, 2 * e, 2 * e + 1, 7 * e + 37):
        add(f"len-{T}-{n}", T, F.ADD, 3, [], [(n, 1)])
add("len-u32-many-chunks", "u32", F.ADD, 3, [], [((1 << 24) + 37, 1)])
add("len-u8-one-chunk-512-outs", "u8", F.ADD, 3, [(512, K + 1)], [(K, 1)])
add("len-u8-one-chunk-512-outs+1", "u8", F.ADD, 3, [(512, K + 1)], [(K, 1)], offset=1)
for off in (0, 1, 15):
    add(f"u8-start+{off}", "u8", F.ADD, 0, [], [(K + 77, 1)], offset=off)
    add(f"u8-rows-start+{off}", "u8", F.XOR, 0, [(3, K + 5)], [(K + 3, 1)], offset=off)          # row pitch K + 5: not 16-byte aligned
add("u32-rows-pitch-not-16B", "u32", F.ADD, 9, [(2, K + 3)], [(K, 1)])  # pitch 4 (K + 3) bytes
add("u32-rows-2d-out", "u32", F.MUL, 1, [(2, 3 * (K + 8)), (3, K + 8)], [(K, 1)], kind="threes")
add("u64-reversed", "u64", F.ADD, 11, [], [(3 * K + 1, -1)], offset=3 * K)
add("u32-reversed-rows", "u32", F.XOR, 11, [(3, -(K + 4))], [(K + 4, -1)], offset=3 * (K + 4) - 1)
add("i32-transposed-full", "i32", F.ADD, -5, [], [(512, 1), (256, 512)])      # the reduction walks columns outermost: reordered
add("u64-transposed-full", "u64", F.ADD, 0, [], [(130, 1), (1000, 130)])
add("u32-three-red-axes", "u32", F.OR, 0, [], [(8, 1), (16, 8), (1024, 128)])
add("u32-transposed-reversed", "u32", F.XOR, 0, [], [(300, -1), (400, 300)], offset=299)
# columns: half 32-byte groups, pitch > row length, a batch axis, an unaligned pitch, a reversed row axis
add("cols-u32-36", "u32", F.ADD, 1, [(36, 1)], [(K, 36)])
add("cols-u32-4", "u32", F.ADD, 1, [(4, 1)], [(K, 4)])
add("cols-u8-20-pitch-24", "u8", F.ADD, 1, [(20, 1)], [(K, 24)])
add("cols-u64-6-pitch-9", "u64", F.XOR, 1, [(6, 1)], [(K, 9)])
add("cols-u32-batch3", "u32", F.ADD, 2, [(3, 12 * (K + 1)), (12, 1)], [(K + 1, 12)])
add("cols-i64-batch-reversed", "i64", F.SUB, 2, [(2, -(5 * K)), (5, 1)], [(K, 5)], offset=5 * K)
add("cols-u32-reversed-rows", "u32", F.AND, -1, [(8, 1)], [(K, -8)], offset=8 * (K - 1), kind="bool")
add("cols-u32-many", "u32", F.ADD, 1, [(1000, 1)], [(K, 1000)])

# ---- values: each operator x dtype with a non-identity init ------------------------------------------------------------------------
for T in ("u8", "i32", "u32", "i64", "u64"):
    for op, init in ((F.ADD, 7), (F.SUB, -3), (F.MUL, 3), (F.AND, 0x5a), (F.OR, 0x11), (F.XOR, 0x5a5a)):
        kind = "threes" if op == F.MUL else "rand"
        add(f"val-{T}-{OPNAME[op] if op != F.SUB else 'sub'}", T, op, init, [], [(K + 19, 1)], kind=kind)
        add(f"val-cols-{T}-{OPNAME[op] if op != F.SUB else 'sub'}", T, op, init, [(3, 1)], [(K, 3)], kind=kind)
add("u8-add-wraps", "u8", F.ADD, 200, [], [(K, 1)], kind="ones")
add("i32-add-overflow", "i32", F.ADD, 2 ** 31 - 10, [], [(K, 1)], kind="ones")
add("i32-sub-from-min", "i32", F.SUB, -2 ** 31, [], [(K, 1)], kind="ones")
add("u64-mul-wraps", "u64", F.MUL, 3, [], [(K, 1)], kind="threes")
add("u64-mul-3s", "u64", F.MUL, 1, [], [(K, 1)], kind="ones")
for kind in ("bool", "ones"):
    for op in (F.AND, F.OR, F.XOR):
        add(f"bool-{OPNAME[op]}-{kind}", "u8", op, 1 if op == F.AND else 0, [], [(K + 1, 1)], kind=kind)


def one_false(id, op):
    def build():
        x = np.ones(K + 9, np.uint8)
        x[K // 2 + 1] = 0
        ax = axes(K + 9)
        lf = L.Node(F.LEAF, F.U8, buf=Storage.from_host(F.U8, x), offset=0, stride={ax[0]: 1})
        return Subject(fold("u8", op, lf, ax, 1 if op == F.AND else 0), []), reference(x, "u8", "u8", op, 1 if op == F.AND else 0, 0, [], [(K + 9, 1)])
    CASES.append(Case(id, build, "fold_split.runs ", split_kernel("u8", "u8", op, "runs"), K + 9))


for op in (F.AND, F.OR, F.XOR):
    one_false(f"bool-{OPNAME[op]}-single-false", op)

# ---- casts ------------------------------------------------------------------------------------------------------------------------
add("cast-bool-u64-count", "u64", F.ADD, 0, [], [(K + 5, 1)], T_src="u8", kind="bool")
add("cast-u32-u64-sum", "u64", F.ADD, 0, [], [(K + 5, 1)], T_src="u32")
add("cast-i32-i64-sum", "i64", F.ADD, 0, [], [(K + 5, 1)], T_src="i32")
add("cast-i32-u64-neg", "u64", F.ADD, 0, [], [(K + 5, 1)], T_src="i32", kind="small")
add("cast-i32-u64-xor", "u64", F.XOR, 0, [], [(K + 5, 1)], T_src="i32", kind="small")
add("cast-u64-u32", "u32", F.ADD, 0, [], [(K + 5, 1)], T_src="u64")
add("cast-u64-u8", "u8", F.ADD, 0, [], [(K + 5, 1)], T_src="u64")
add("cast-u64-u8-mul", "u8", F.MUL, 1, [], [(K + 5, 1)], T_src="u64", kind="threes")
add("cast-u8-i32-cols", "i32", F.SUB, 0, [(5, 1)], [(K, 5)], T_src="u8")
add("cast-i32-i64-cols", "i64", F.ADD, 0, [(5, 1)], [(K, 7)], T_src="i32", kind="small")

# ---- launcher -----------------------------------------------------------------------------------------------------------------------
add("out+4", "u32", F.ADD, 1, [(3, K)], [(K, 1)], shift=4)
add("cols-out+4", "u32", F.ADD, 1, [(3, 1)], [(K, 3)], shift=4)
add("host-collect", "u64", F.ADD, 1, [(2, K + 1)], [(K + 1, 1)], T_src="u32", host=True)

CASE_IDS = [c.id for c in CASES]
assert len(set(CASE_IDS)) == len(CASE_IDS), "case ids must be unique"


# ---- CPU half -----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_planned_route_and_reference(case):
    """describe() names the route; the numpy reference equals the C oracle bit for bit; NO_FASTPATH sends the split fold to the
    evaluator."""
    subject, want = case.build()
    d = subject.describe()
    assert d.startswith(case.route), d
    if case.route.startswith("fold_split"):
        assert subject.describe(F.COLLECT_NO_FASTPATH).startswith("generic."), subject.describe(F.COLLECT_NO_FASTPATH)
    else:
        assert "fold_split" not in d
    if want is not None and case.n_elems <= ORACLE_MAX_ELEMS:
        (got,), err = subject.oracle()
        assert err is None, err
        assert_same_bits(want, got, case.id + " (reference vs oracle)")


def test_describe_fields():
    subject, _ = next(c for c in CASES if c.id == "cast-u32-u64-sum").build()
    assert subject.describe() == f"fold_split.runs outs=1 red={K + 5} slot=s64 src=u32 op=0"
    subject, _ = next(c for c in CASES if c.id == "cols-u32-batch3").build()
    assert subject.describe() == f"fold_split.cols outs=36 red={K + 1} slot=s32 src=u32 op=0"


# ---- GPU half -----------------------------------------------------------------------------------------------------------------------
_ctx = []


@pytest.fixture
def gpu_ctx():
    if not _ctx:
        _ctx.append(P.Context(0))
    return _ctx[0]


def host_collect(subject, ctx):
    em = L.emit(subject.root(), subject.axes, "host")
    out = np.zeros(em.out_len, NPD[em.out_dtypes[0]])
    ctx.collect_host(em.expr, out.ctypes.data)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_kernel_route(case, gpu_ctx):
    subject, want = case.build()
    before = gpu_ctx.launch_count()
    (got,), err, ran = subject.gpu(gpu_ctx)
    assert err is None, err
    if case.kernel is not None:
        assert ran == case.kernel, f"{case.id}: ran {ran}, expected {case.kernel} ({subject.describe()})"
        assert gpu_ctx.launch_count() - before == 1
    else:
        assert not ran.startswith("k_fold_split"), ran
    if want is None:
        (want,), _ = subject.oracle()
    assert_same_bits(got, want, f"{case.id} on {ran}")
    if case.host:
        assert_same_bits(host_collect(subject, gpu_ctx), want, f"{case.id} (collect_host)")


@pytest.mark.gpu
def test_async_back_to_back(gpu_ctx):
    """Two split folds on independent operands, launched ASYNC back to back: the second waits for the first's scratch."""
    subs = [c.build() for c in CASES if c.id in ("edge-runs-outs3", "cols-u32-batch3")]
    outs = []
    for subject, _ in subs:
        for n in subject._leaves():
            n.buf.ensure_device(gpu_ctx)
        em = L.emit(subject.root(), subject.axes, "device")
        p = gpu_ctx.alloc(em.out_len * F.DTYPE_SIZE[em.out_dtypes[0]])
        outs.append((p, em))
    for rep in range(3):
        for (p, em), (subject, _) in zip(outs, subs):
            gpu_ctx.collect(em.expr, p, F.COLLECT_ASYNC)
            assert gpu_ctx.last_kernel().startswith("k_fold_split")
        gpu_ctx.sync()
        for (p, em), (subject, want) in zip(outs, subs):
            h = np.empty(em.out_len, NPD[em.out_dtypes[0]])
            gpu_ctx.download(h, p)
            assert_same_bits(h, want, f"async rep {rep}")
    for p, _ in outs:
        gpu_ctx.free(p)


@pytest.mark.gpu
def test_wide_bool_count(gpu_ctx):
    """A bool -> u64 count over 2^32 + 37 bytes: the count passes 2^32, which a 32-bit accumulator would wrap."""
    n = (1 << 32) + 37
    x = np.ones(n, np.uint8)
    zeros = np.random.default_rng(5).integers(0, n, 20)
    x[zeros] = 0
    want = np.array([n - np.unique(zeros).size + 9], np.uint64)
    assert want[0] > 1 << 32
    ax = axes(n)
    lf = L.Node(F.LEAF, F.U8, buf=Storage.from_host(F.U8, x), offset=0, stride={ax[0]: 1})
    del x
    b = L.Node(F.UNARY, F.U64, op=F.CAST, src_dtype=F.U8, children=(lf,))
    subject = Subject(fold("u64", F.ADD, b, ax, 9), [])
    assert subject.describe().startswith("fold_split.runs ")
    (got,), err, ran = subject.gpu(gpu_ctx)
    assert err is None and ran == "k_fold_split<u64,src=u8,add,runs>", (err, ran)
    assert_same_bits(got, want, "wide bool count")
