"""Parity tests proper: every kernel family of the product against the C oracle on the same seeded
inputs (bit-exact for everything, including f32 — the kernels keep the reference's operation
order and never fuse multiply-add).

Each test runs twice: `[gpu]` (marked gpu; the sm_100a kernels through the C ABI on a B200) and
`[emu]` (CPU suite; the product's planner and per-thread evaluator compiled for the host, which
covers lowering, decode, load modes, predicates, gather/fold control flow and error reporting —
but not the dedicated transpose / row-fold kernels, which only exist as CUDA)."""
import os

import numpy as np
import pytest

from helpers import oracle_collect, assert_same_bits, CheckerPanic
import multidimension_b200 as P
from multidimension_b200 import usize, Array, Scalar, All, all_, fold_rows, Add, Sub, Mul, Div, Rem, BitAnd, BitOr, BitXor, Shl, Shr
from multidimension_b200 import _ffi as F

NP = {"f32": np.float32, "f64": np.float64, "i32": np.int32, "u32": np.uint32, "i64": np.int64, "u64": np.uint64, "u8": np.uint8}


from helpers import emu_collect

_gpu_ctx = []


@pytest.fixture(params=[pytest.param("emu", id="emu"), pytest.param("gpu", id="gpu", marks=pytest.mark.gpu)])
def ctx(request):
    if request.param == "emu":
        return "emu"
    if not _gpu_ctx:
        _gpu_ctx.append(P.Context(0))
        P.set_default_context(_gpu_ctx[0])
    return _gpu_ctx[0]


def collect(view, ctx, flags=0):
    """-> flat numpy array (or list of tuples) of the collected view on the chosen backend."""
    if ctx == "emu":
        return emu_collect(view, flags)
    return view.collect(location="device", flags=flags, ctx=ctx).as_ref()


def panic_info(excinfo):
    return excinfo.value.info


def rand(rng, T, n, lo=-4, hi=4):
    if T in ("f32", "f64"):
        return rng.uniform(lo, hi, n).astype(NP[T])
    if T is usize:
        return rng.integers(0, 1 << 40, n).astype(np.uint64)
    info = np.iinfo(NP[T])
    return rng.integers(info.min, info.max, n, dtype=NP[T], endpoint=True)


def check(view, ctx, flags=0, what=""):
    want = oracle_collect(view)
    got = collect(view, ctx, flags)
    if isinstance(want, list):
        assert got == want, what
    else:
        assert_same_bits(got, want, what or str(view.describe()))


# ---- K1: contiguous fused elementwise (config 2) ------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 7, 8, 1000, 4096, (1 << 20) + 24, (1 << 22) + 3])
def test_zip_map_mul_add(ctx, n):
    rng = np.random.default_rng(n)
    a = Array.new(usize, n, rand(rng, "f32", n))
    b = Array.new(usize, n, rand(rng, "f32", n))
    v = a.zip(b).map(lambda p: p[0] * p[1] + np.float32(1))
    check(v, ctx)
    check(a * b + Scalar(1.0, "f32"), ctx)
    check(v, ctx, F.COLLECT_NO_STATIC)


@pytest.mark.parametrize("T", ["f32", "f64", "i32", "u32", "i64", "u64", "u8"])
def test_every_binary_op(ctx, T):
    rng = np.random.default_rng(11)
    n = 4096 + 8
    a = Array.new(usize, n, rand(rng, T, n), T)
    bv = rand(rng, T, n)
    if T not in ("f32", "f64"):
        bv[bv == 0] = 1
        if T in ("i32", "i64"):
            bv[bv == -1] = 2
    b = Array.new(usize, n, bv, T)
    ops = [Add, Sub, Mul, Div, Rem] + ([] if T in ("f32", "f64") else [BitAnd, BitOr, BitXor, Shl, Shr])
    for B in ops:
        check(a.binary(b, B), ctx, what=f"{T} {B}")
        check(a.binary(Scalar(bv[3].item(), T), B), ctx, what=f"{T} {B} scalar")


def test_unary_and_casts(ctx):
    rng = np.random.default_rng(5)
    n = 2048
    f = Array.new(usize, n, np.concatenate([rand(rng, "f32", n - 6, -1e10, 1e10), np.float32([np.nan, np.inf, -np.inf, -0.0, 3e9, -3e9])]))
    for U in (P.Neg, P.Abs):
        check(f.map(U), ctx)
    check(f.map(P.Abs).map(P.Sqrt), ctx)
    for T in ("i32", "u32", "i64", "u64", "u8", "f64"):
        check(f.map(P.Cast(T)), ctx, what=f"f32 as {T}")
    i = Array.new(usize, n, rand(rng, "i64", n), "i64")
    for T in ("f32", "f64", "i32", "u8", "u64"):
        check(i.map(P.Cast(T)), ctx, what=f"i64 as {T}")
    for U in (P.Neg, P.Not, P.Abs):
        check(i.map(U), ctx)


def test_integer_division_by_zero(ctx):  # Rust panics in every build mode
    a = Array.new(usize, 100, np.arange(100, dtype=np.uint64))
    b = Array.new(usize, 100, np.where(np.arange(100) == 37, 0, 3).astype(np.uint64))
    with pytest.raises((P.Panic, CheckerPanic)) as e:
        collect(a / b, ctx)
    assert e.value.status == F.ERR_ARITH and panic_info(e).position == 37
    with pytest.raises(CheckerPanic):
        oracle_collect(a / b)
    check(a / Scalar(7), ctx)  # the context keeps working after a failure


# ---- K2: tiled transpose (config 1) ------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(64, 64), (128, 256), (100, 36), (17, 300), (1, 70), (70, 1), (5, 5), (1024, 1024), (250, 1030)])
@pytest.mark.parametrize("T", ["f32", "f64"])
def test_transpose_2d(ctx, shape, T):
    rng = np.random.default_rng(shape[0] * 7919 + shape[1])
    a = Array.new((usize, usize), shape, rand(rng, T, shape[0] * shape[1]), T)
    check(a.transpose((), usize, usize, ()), ctx)
    check(a.transpose((), usize, usize, ()), ctx, F.COLLECT_NO_FASTPATH)


def test_transpose_batched_and_grouped(ctx):
    rng = np.random.default_rng(3)
    a = Array.new(((usize, usize), (usize, usize)), ((3, 40), (70, 8)), rand(rng, "f32", 3 * 40 * 70 * 8))
    check(a.transpose(usize, usize, usize, usize), ctx)                 # I and J both present
    check(a.transpose((), usize, (usize, usize), usize), ctx)          # compound Y
    check(a.transpose((), (usize, usize), (usize, usize), ()), ctx)    # swap halves
    check(a.transpose((usize, usize), usize, usize, ()), ctx)          # innermost swap, batch of 120
    u = Array.new((usize, usize), (96, 200), rand(rng, usize, 96 * 200))
    check(u.transpose((), usize, usize, ()), ctx)                        # 8-byte integers


def test_transpose_iota_exact(ctx):  # SURVEY.md §8d C1 input: a[k] = k as f32, exact below 2^24
    n = 512
    a = Array.new((usize, usize), (n, n), np.arange(n * n, dtype=np.float32))
    got = collect(a.transpose((), usize, usize, ()), ctx)
    assert_same_bits(got, np.arange(n * n, dtype=np.float32).reshape(n, n).T.copy().reshape(-1))


# ---- K3: gather (config 3) ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_idx,n_src", [(0, 10), (1, 1), (1000, 17), (1 << 18, 1 << 20), ((1 << 16) + 5, 999)])
def test_compose_gather(ctx, n_idx, n_src):
    rng = np.random.default_rng(n_idx + n_src)
    src = Array.new(usize, n_src, rand(rng, "f32", n_src))
    idx = Array.new(usize, n_idx, rng.integers(0, n_src, n_idx).astype(np.uint64))
    check(idx.compose(src), ctx)
    check(idx.compose(src), ctx, F.COLLECT_NO_STATIC)
    src64 = Array.new(usize, n_src, rand(rng, usize, n_src))
    check(idx.compose(src64), ctx)


def test_compose_out_of_bounds(ctx):  # src/int.rs:17
    n = 1 << 16
    src = Array.new(usize, 1000, np.arange(1000, dtype=np.float32))
    iv = (np.arange(n) % 1000).astype(np.uint64)
    iv[40000] = 1000
    iv[50000] = 123456
    idx = Array.new(usize, n, iv)
    with pytest.raises((P.Panic, CheckerPanic), match="Index 1000 is out of bounds for size 1000") as e:
        collect(idx.compose(src), ctx)
    info = panic_info(e)
    assert (info.status, info.position, info.value, info.bound, info.component) == (F.ERR_OOB, 40000, 1000, 1000, 0)
    with pytest.raises(CheckerPanic, match="Index 1000 is out of bounds for size 1000"):
        oracle_collect(idx.compose(src))


def test_compose_two_components_and_map_axis(ctx):
    rng = np.random.default_rng(9)
    src = Array.new((usize, usize), (37, 53), rand(rng, "f32", 37 * 53))
    n = 5000
    i = Array.new(usize, n, rng.integers(0, 37, n).astype(np.uint64))
    j = Array.new(usize, n, rng.integers(0, 53, n).astype(np.uint64))
    check(i.zip(j).compose(src), ctx)                       # Array<usize,(usize,usize)> selecting from a matrix
    check(j.zip(i).compose(src.transpose((), usize, usize, ()).iso((usize, usize))), ctx)  # source is itself a view
    take = Array.new(usize, 400, rng.integers(0, 53, 400).astype(np.uint64))
    check(src.map_axis(take, usize, ()), ctx)               # take along the last axis
    take0 = Array.new(usize, 90, rng.integers(0, 37, 90).astype(np.uint64))
    check(src.map_axis(take0, (), usize), ctx)              # take along the first axis: rows stay contiguous
    check(take.compose(src.row(usize, usize, 5) * Scalar(2.0, "f32")), ctx)  # gather pushed through an operator


# ---- K4: sequential-order fold (+ broadcast epilogue) (config 4) ----------------------------------------------------
@pytest.mark.parametrize("rows,n", [(1, 8), (33, 64), (1000, 256), (257, 1024), (4096, 12), (70, 1028), (5, 7), (300, 2048)])
def test_fold_last_axis_sum(ctx, rows, n):
    rng = np.random.default_rng(rows * 31 + n)
    a = Array.new((usize, usize), (rows, n), rng.uniform(0, 1, rows * n).astype(np.float32))
    s = fold_rows(a, usize, usize, Add, np.float32(0))
    check(s, ctx)
    check(s, ctx, F.COLLECT_NO_FASTPATH)
    seq = np.add.accumulate(a.as_ref().reshape(rows, n), axis=1, dtype=np.float32)[:, -1]  # sequential, not pairwise
    assert_same_bits(collect(s, ctx), seq)


def test_fold_fused_broadcast_subtract(ctx):  # config 4 in miniature, all three spellings
    rng = np.random.default_rng(4)
    shape = (24, 40, 256)
    a = Array.new((usize, usize, usize), shape, rng.uniform(0, 1, int(np.prod(shape))).astype(np.float32))
    sums = fold_rows(a, (usize, usize), usize, Add, np.float32(0))
    mean = sums / Scalar(256.0, "f32")
    fused = a - mean.iso((usize, usize, ()))
    assert "fold_rows.fused" in fused.describe()
    check(fused, ctx)
    check(fused, ctx, F.COLLECT_NO_FASTPATH)
    means = Array.new((usize, usize), shape[:2], collect(mean, ctx))  # two-pass spelling: 4a then 4b
    check(a - means.iso((usize, usize, ())), ctx)
    check(a - sums.iso((usize, usize, ())), ctx)


def test_fold_other_ops_and_types(ctx):
    rng = np.random.default_rng(6)
    a = Array.new((usize, usize), (100, 48), rng.integers(0, 1 << 31, 4800).astype(np.uint32), "u32")
    check(fold_rows(a, usize, usize, Add, 0), ctx)
    check(fold_rows(a, usize, usize, BitXor, 0), ctx)
    check(fold_rows(a, usize, usize, Mul, 1), ctx)
    f = Array.new((usize, usize), (100, 48), rng.uniform(0.9, 1.1, 4800).astype(np.float32))
    check(fold_rows(f, usize, usize, Mul, np.float32(1)), ctx)
    d = Array.new((usize, usize), (50, 30), rng.uniform(0, 1, 1500))
    check(fold_rows(d, usize, usize, Add, 0.0), ctx)
    check(fold_rows(f.transpose((), usize, usize, ()).iso((usize, usize)), usize, usize, Add, np.float32(0)), ctx)  # strided rows
    check(fold_rows(f, (), (usize, usize), Add, np.float32(0)), ctx)                                               # full reduction


@pytest.mark.parametrize("shape", [(64, 40, 64), (7, 3, 8), (300, 5, 12), (33, 17, 1)])
def test_fold_over_outermost_axis(ctx, shape):  # the per-rank partial of a sharded-axis reduction
    rng = np.random.default_rng(sum(shape))
    I, J, K = shape
    a = Array.new((usize, usize, usize), shape, rng.uniform(0, 1, I * J * K).astype(np.float32))
    v = fold_rows(a.transpose((), (usize, usize), usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, Add, np.float32(0))
    check(v, ctx)
    check(v, ctx, F.COLLECT_NO_STATIC)
    seq = np.add.accumulate(a.as_ref().reshape(I, J * K), axis=0, dtype=np.float32)[-1]
    assert_same_bits(collect(v, ctx), seq)
    check(fold_rows(a.transpose((), (usize, usize), usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, Mul, np.float32(1)), ctx)


def test_fold_over_outer_axis_column_walk(ctx):
    """KK_FOLD_COLS (k_fold_cols): a sequential fold over an OUTER axis whose result is contiguous is a column walk with 256-bit
    loads — the one-GPU form of the fold over the sharded axis.  Every dtype / operator it takes, rows 32- and only 16-byte
    aligned, a column window of a wider Array (row pitch > row length), a tail of rows below the unroll, and the evaluator
    (NO_FASTPATH) as the second opinion."""
    rng = np.random.default_rng(77)

    def outer_fold(a, rows, cols, op, init):
        return fold_rows(a.transpose((), usize, usize, ()).iso((usize, usize)), usize, usize, op, init)
    for rows, cols in ((100, 64), (37, 1028), (16, 8), (5, 4), (129, 520)):
        f = Array.new((usize, usize), (rows, cols), rng.uniform(0.9, 1.1, rows * cols).astype(np.float32))
        for op, init in ((Add, np.float32(0.25)), (Mul, np.float32(1)), (P.Sub, np.float32(3))):
            v = outer_fold(f, rows, cols, op, init)
            assert "fold_cols" in v.describe(), v.describe()
            check(v, ctx)
            check(v, ctx, F.COLLECT_NO_FASTPATH)
        seq = np.full(cols, np.float32(0.25))
        for i in range(rows):
            seq = seq + f.as_ref().reshape(rows, cols)[i]
        assert_same_bits(collect(outer_fold(f, rows, cols, Add, np.float32(0.25)), ctx), seq)
    u = Array.new((usize, usize), (50, 36), rng.integers(0, 1 << 63, 1800).astype(np.uint64), usize)
    for op, init in ((Add, 7), (Mul, 3), (BitXor, 0), (P.BitAnd, (1 << 64) - 1), (P.BitOr, 0)):
        check(outer_fold(u, 50, 36, op, init), ctx)
    i32 = Array.new((usize, usize), (40, 12), rng.integers(-2**31, 2**31, 480).astype(np.int32), "i32")
    check(outer_fold(i32, 40, 12, Add, np.int32(-5)), ctx)     # wrapping
    d = Array.new((usize, usize), (33, 10), rng.uniform(0, 1, 330))
    check(outer_fold(d, 33, 10, Add, 0.5), ctx)
    # a fold over a MIDDLE axis: one column walk per outer coordinate (batch), results back to back
    for I, J, K in ((6, 10, 16), (3, 37, 8), (5, 2, 260), (2, 129, 4)):
        t = Array.new((usize, usize, usize), (I, J, K), rng.uniform(0, 1, I * J * K).astype(np.float32))
        v = fold_rows(t.transpose(usize, usize, usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, Add, np.float32(0.5))
        assert f"fold_cols batch={I} rows={J} cols={K}" in v.describe(), v.describe()
        check(v, ctx)
        check(v, ctx, F.COLLECT_NO_FASTPATH)
        seq = np.full((I, K), np.float32(0.5))
        for j in range(J):
            seq = seq + t.as_ref().reshape(I, J, K)[:, j, :]
        assert_same_bits(collect(v, ctx), seq.reshape(-1))
    t64 = Array.new((usize, usize, usize), (4, 9, 6), rng.integers(0, 1 << 62, 216).astype(np.uint64), usize)
    check(fold_rows(t64.transpose(usize, usize, usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, BitXor, 0), ctx)
    # 17 columns: rows not a multiple of 16 bytes -> the evaluator keeps it
    odd = Array.new((usize, usize), (9, 17), rng.uniform(0, 1, 153).astype(np.float32))
    v = outer_fold(odd, 9, 17, Add, np.float32(0))
    assert "fold_cols" not in v.describe()
    check(v, ctx)


# ---- K5: general rank-N evaluator (config 5) ----------------------------------------------------------------------------
def config5(P_, Q, R, rng):
    a = Array.new((usize, usize), (P_, Q), rand(rng, "f32", P_ * Q))
    w = Array.new(usize, R, rand(rng, "f32", R))
    t = a.transpose((), usize, usize, ())
    d = t.diagonal(np.float32(0))
    d5 = d.iso((((usize, usize), (usize, usize)), ()))
    z = d5.zip(w.iso(((), usize)))
    return z.map(lambda p: p[0] * p[1] + np.float32(1))


@pytest.mark.parametrize("dims", [(4, 4, 8), (6, 5, 16), (3, 7, 5), (8, 8, 64), (16, 16, 64)])
def test_rank5_chain(ctx, dims):
    v = config5(*dims, np.random.default_rng(sum(dims)))
    assert v.I == (((usize, usize), (usize, usize)), usize)
    check(v, ctx)
    check(v, ctx, F.COLLECT_NO_STATIC)


def test_diagonal_guards_gather(ctx):  # Diagonal::at never evaluates its inner view off the diagonal (src/view.rs:854-856)
    src = Array.new(usize, 4, np.float32([10, 11, 12, 13]))
    idx = Array.new(usize, 4, np.uint64([3, 2, 1, 0]))
    check(idx.compose(src).diagonal(np.float32(-1)), ctx)


def test_mixed_strides_broadcast(ctx):
    rng = np.random.default_rng(8)
    a = Array.new((usize, usize, usize), (12, 20, 32), rand(rng, "f32", 12 * 20 * 32))
    r = Array.new(usize, 20, rand(rng, "f32", 20))
    c = Array.new(usize, 12, rand(rng, "f32", 12))
    v = (a * r.iso(((), usize, ()))) - c.iso((usize, (), ()))
    check(v, ctx)
    check(v.transpose((), usize, (usize, usize), ()), ctx)
    check(a.row(usize, (usize, usize), 7) + a.row(usize, (usize, usize), 2), ctx)
    check(a.column((usize, usize), usize, 5), ctx)


def test_concat_along_every_axis(ctx):  # src/view.rs:920-946
    rng = np.random.default_rng(13)
    x = Array.new((usize, usize), (50, 16), rand(rng, "f32", 800))
    y = Array.new((usize, usize), (50, 24), rand(rng, "f32", 1200))
    c = x.concat(y, usize, ())                      # along the innermost (vector) axis
    check(c, ctx)
    check(c.transpose((), usize, usize, ()), ctx)
    ci = c.iso((usize, usize))                      # ((),()) does not broadcast in the reference, so regroup first
    check(ci * ci + Scalar(1.0, "f32"), ctx)
    check(c.column(usize, usize, 20), ctx)          # pinned inside W: only W survives the lowering
    check(c.row(usize, usize, 7), ctx)
    x2 = Array.new((usize, usize), (30, 40), rand(rng, "f32", 1200))
    y2 = Array.new((usize, usize), (70, 40), rand(rng, "f32", 2800))
    c2 = x2.concat(y2, (), usize)                   # along the outermost axis
    check(c2, ctx)
    check(c2.concat(c2, (), usize), ctx)            # nested concats
    odd = Array.new(usize, 13, rand(rng, "f32", 13)).concat(Array.new(usize, 30, rand(rng, "f32", 30)), (), ())
    check(odd, ctx)                                 # boundary inside a vector: per-lane masked loads
    # laziness: the side that is not selected is never evaluated (an out-of-range index there is harmless)
    src = Array.new(usize, 4, np.float32([10, 11, 12, 13]))
    good = Array.new(usize, 3, np.uint64([3, 2, 1])).compose(src)
    check(good.concat(Array.new(usize, 5, rand(rng, "f32", 5)), (), ()), ctx)


# ---- host-buffer entry point (mdim_collect_host) ------------------------------------------------------------------------
@pytest.mark.gpu
def test_collect_host_chunked():
    old = os.environ.get("MDIM_HOST_CHUNK_MB")
    os.environ["MDIM_HOST_CHUNK_MB"] = "1"
    try:
        c2 = P.Context(0)
    finally:
        if old is None:
            del os.environ["MDIM_HOST_CHUNK_MB"]
        else:
            os.environ["MDIM_HOST_CHUNK_MB"] = old
    rng = np.random.default_rng(12)
    n = (1 << 21) + 40
    a = Array.new(usize, n, rand(rng, "f32", n))
    b = Array.new(usize, n, rand(rng, "f32", n))
    v = a * b + Scalar(1.0, "f32")
    got = v.collect(ctx=c2)  # all operands in host memory -> mdim_collect_host, ~25 chunks
    assert got.storage.home == "host"
    assert_same_bits(got.as_ref(), oracle_collect(v))
    m = Array.new((usize, usize), (3000, 700), rand(rng, "f32", 3000 * 700))
    r = Array.new(usize, 700, rand(rng, "f32", 700))
    for view in (m.transpose((), usize, usize, ()), m - r.iso(((), usize)),
                 fold_rows(m, usize, usize, Add, np.float32(0)),
                 m - (fold_rows(m, usize, usize, Add, np.float32(0)) / Scalar(700.0, "f32")).iso((usize, ()))):
        assert_same_bits(view.collect(ctx=c2).as_ref(), oracle_collect(view), str(view.describe()))
    m2 = Array.new((usize, usize), (3000, 300), rand(rng, "f32", 3000 * 300))
    for view in (m.concat(m2, usize, ()), m.concat(m, (), usize), m.concat(m2, usize, ()).transpose((), usize, usize, ())):
        assert_same_bits(view.collect(ctx=c2).as_ref(), oracle_collect(view), "host concat " + str(view.describe()))
    src = Array.new(usize, 5000, rand(rng, "f32", 5000))
    iv = rng.integers(0, 5000, 1 << 19).astype(np.uint64)
    idx = Array.new(usize, iv.size, iv)
    assert_same_bits(idx.compose(src).collect(ctx=c2).as_ref(), oracle_collect(idx.compose(src)))
    iv[300000] = 5001
    with pytest.raises(P.Panic, match="Index 5001 is out of bounds for size 5000") as e:
        Array.new(usize, iv.size, iv).compose(src).collect(ctx=c2)
    assert e.value.info.position == 300000
    c2.close()


# ---- 64-bit coordinates (arrays past 2^31 elements): checked on the device against torch --------------------
@pytest.mark.gpu
def test_wide_coordinates_past_2_31_elements():
    import torch
    from multidimension_b200.runtime import Storage
    c = P.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    c.set_stream(stream.cuda_stream)
    n = (1 << 31) + 1024                                   # u8 stream: offsets need 64 bits
    ta = torch.randint(0, 255, (n,), device="cuda", dtype=torch.uint8)
    to = torch.empty(n, device="cuda", dtype=torch.uint8)
    a = Array.from_device(usize, n, ta.data_ptr(), "u8", ctx=c, keep=ta)
    v = a + Scalar(3, "u8")
    assert " wide" in v.describe()
    v.collect(out=Storage.wrap_device(c, F.U8, n, to.data_ptr(), keep=to), ctx=c)
    assert torch.equal(to, ta + 3)                          # wrapping u8 add, every element
    del ta, to, a, v
    rows, cols = 1 << 16, (1 << 15) + 8                     # rank 2, 2^31 + 2^19 f32 elements, broadcast row vector
    tm = torch.empty(rows * cols, device="cuda", dtype=torch.float32).uniform_(-1, 1)
    tr = torch.empty(cols, device="cuda", dtype=torch.float32).uniform_(-1, 1)
    tout = torch.empty(rows * cols, device="cuda", dtype=torch.float32)
    m = Array.from_device((usize, usize), (rows, cols), tm.data_ptr(), "f32", ctx=c, keep=tm)
    r = Array.from_device(usize, cols, tr.data_ptr(), "f32", ctx=c, keep=tr)
    w = m - r.iso(((), usize))
    assert " wide" in w.describe()
    w.collect(out=Storage.wrap_device(c, F.F32, rows * cols, tout.data_ptr(), keep=tout), ctx=c)
    assert torch.equal(tout.view(rows, cols), tm.view(rows, cols) - tr)
    t = m.transpose((), usize, usize, ())                   # the tile kernels take 32-bit coordinates only: the evaluator's 64-bit path serves this
    assert " wide" in t.describe() and "transpose.tile" not in t.describe(), t.describe()
    t.collect(out=Storage.wrap_device(c, F.F32, rows * cols, tout.data_ptr(), keep=tout), ctx=c)
    assert not c.last_kernel().startswith("k_transpose"), c.last_kernel()
    assert torch.equal(tout.view(cols, rows), tm.view(rows, cols).t())
    torch.cuda.synchronize()
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["1", "2"])
def test_both_fold_kernels_for_both_forms(mode):
    """MDIM_FOLD_MODE forces the shared-memory/TMA form (1) or the register form (2) for fold-only AND fused
    chains (by default each serves the form it is faster for); both must stay bit-exact and sequential."""
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, "tests")
from helpers import assert_same_bits
import multidimension_b200 as P
from multidimension_b200 import usize, Array, Scalar, Add, fold_rows
ctx = P.Context(0); P.set_default_context(ctx)
rng = np.random.default_rng(1)
for rows, n in [(1, 32), (77, 64), (1000, 256), (33, 512), (130, 1024), (64, 96), (9, 2048)]:
    x = rng.uniform(0, 1, rows * n).astype(np.float32)
    a = Array.new((usize, usize), (rows, n), x)
    s = fold_rows(a, usize, usize, Add, np.float32(0))
    seq = np.add.accumulate(x.reshape(rows, n), axis=1, dtype=np.float32)[:, -1]
    assert_same_bits(s.collect(location="device").as_ref(), seq, f"fold {rows}x{n}")
    fused = a - (s / Scalar(float(n), "f32")).iso((usize, ()))
    want = (x.reshape(rows, n) - (seq / np.float32(n))[:, None]).reshape(-1)
    assert_same_bits(fused.collect(location="device").as_ref(), want, f"fused {rows}x{n}")
print("ok")
'''
    env = dict(os.environ, MDIM_FOLD_MODE=mode)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_shape_specialised_kernels_on_first_use():
    """By default a rank-N chain is specialised on its shape the SECOND time it is collected, which most
    tests never reach; MDIM_JIT_SHAPES=1 specialises at once, so the same parity tests then run through the
    shape-specialised kernels (strides, dividers and predicates as immediates)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, MDIM_JIT_SHAPES="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(root, "tests", "test_gpu_parity.py"), "-m", "gpu", "-q", "-x", "-k",
                        "(rank5 or mixed_strides or concat or diagonal_guards or transpose_batched or fold_over_outermost or two_components) and gpu"],
                       env=env, capture_output=True, text=True, cwd=root)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


@pytest.mark.gpu
def test_dependency_aware_launches_respect_raw_war_and_waw_hazards():
    """csrc/launch.cuh: a collect whose buffers are untouched by the kernels still in flight skips the stream-order wait.
    Chains with read-after-write, write-after-read and write-after-write hazards between back-to-back ASYNC launches must
    still give the sequential result (and independent launches in between must not break the chain)."""
    from multidimension_b200.runtime import Storage
    c = P.Context(0)
    rng = np.random.default_rng(12)
    n = 1024
    x0 = rng.uniform(-1, 1, n * n).astype(np.float32)
    bufs = [Storage.device(c, F.F32, n * n) for _ in range(4)]
    c.upload(bufs[0].dptr, x0)
    other_src = [Array.new((usize, usize), (n, n), rng.uniform(-1, 1, n * n).astype(np.float32)).to_device(c) for _ in range(3)]
    other_out = [Storage.device(c, F.F32, n * n) for _ in range(3)]

    def arr(k):
        return Array((usize, usize), (n, n), bufs[k], "f32")
    for rounds in range(20):
        # RAW chain: b1 = t(b0); b2 = t(b1) (= b0); b3 = b2 * b1' ... interleaved with independent transposes
        arr(0).transpose((), usize, usize, ()).collect(out=bufs[1], ctx=c, flags=F.COLLECT_ASYNC)
        other_src[0].transpose((), usize, usize, ()).collect(out=other_out[0], ctx=c, flags=F.COLLECT_ASYNC)       # independent
        arr(1).transpose((), usize, usize, ()).collect(out=bufs[2], ctx=c, flags=F.COLLECT_ASYNC)                     # RAW on b1
        other_src[1].transpose((), usize, usize, ()).collect(out=other_out[1], ctx=c, flags=F.COLLECT_ASYNC)       # independent
        (arr(2) * arr(1) + Scalar(1.0, "f32")).collect(out=bufs[3], ctx=c, flags=F.COLLECT_ASYNC)                   # RAW on b2, b1
        other_src[2].transpose((), usize, usize, ()).collect(out=bufs[1], ctx=c, flags=F.COLLECT_ASYNC)              # WAR on b1 (b3's kernel reads it), WAW on b1
        arr(3).transpose((), usize, usize, ()).collect(out=bufs[2], ctx=c, flags=F.COLLECT_ASYNC)                     # WAW on b2, RAW on b3
    c.sync()
    X = x0.reshape(n, n)
    want3 = (X * X.T + np.float32(1)).astype(np.float32)
    assert np.array_equal(bufs[3].to_numpy().reshape(n, n), want3)
    assert np.array_equal(bufs[2].to_numpy().reshape(n, n), want3.T)
    assert np.array_equal(bufs[1].to_numpy().reshape(n, n), other_src[2].as_ref().reshape(n, n).T)
    for k in range(2):
        assert np.array_equal(other_out[k].to_numpy().reshape(n, n), other_src[k].as_ref().reshape(n, n).T)
    c.close()
