#!/usr/bin/env python
"""Rates of the 1- and 2-byte integer types on one GPU, beside the 4-byte types that stream the same way.

    python scripts/narrow_bench.py [--runs 5] [--out profiles/r4_narrow_dtypes.txt]

Cases: `a * b + 1` (evaluator stream) on i16 and i8 beside f32 and u32 at 2^30 elements; whole-array sums i16 -> i64,
i8 -> i64 and u16 -> u64 (split fold) beside u32 -> u64 at 2^31 elements; a u16 4096 x 4096 transpose (evaluator).  Operands live
on the GPU (torch allocates and fills them) and are larger than the 126 MB L2, except the transpose's 32 MiB.  Each run times
`reps` back-to-back collects with CUDA events on the context's stream, after warm-up collects until the same kernel runs twice
(the run-time specialisations are built by then).  The rate is algorithmic: the bytes the expression must read and write, over
the time of one collect.  Prints the median and the spread (min - max) of the runs and the kernel that ran.
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import multidimension_b200 as P
    from multidimension_b200 import _ffi as F
    from multidimension_b200 import lowering as L
    from multidimension_b200.runtime import Storage

    TT = {F.I8: torch.int8, F.I16: torch.int16, F.U16: torch.int16, F.U32: torch.int32, F.F32: torch.float32, F.I64: torch.int64,
          F.U64: torch.int64}
    ctx = P.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream_handle())
    keep = []

    def operand(dt, n, seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        if dt == F.F32:
            t = torch.rand(n, device="cuda", generator=g)
        else:
            t = torch.randint(-100, 100, (n,), device="cuda", generator=g, dtype=TT[dt])
        keep.append(t)
        return Storage.wrap_device(ctx, dt, n, t.data_ptr(), keep=t)

    def timed(root, axes, n_out, out_dt):
        em = L.emit(root, axes, "device")
        out = torch.empty(max(n_out * F.DTYPE_SIZE[out_dt], 16), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        kernel = None
        for _ in range(4):  # warm up until the same kernel runs twice: a rank-2 chain is specialised for its shape on its 2nd collect
            ctx.collect(em.expr, out.data_ptr(), 0)
            ctx.sync()
            if ctx.last_kernel() == kernel:
                break
            kernel = ctx.last_kernel()
        times = []
        for _ in range(args.runs):
            with torch.cuda.stream(stream):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(args.reps):
                    ctx.collect(em.expr, out.data_ptr(), F.COLLECT_ASYNC)
                e1.record(stream)
            ctx.sync()
            times.append(e0.elapsed_time(e1) / 1e3 / args.reps)
        return times, kernel

    name = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = [f"# scripts/narrow_bench.py --runs {args.runs} --reps {args.reps} on {name}",
             "# case | GB/s median | GB/s min - max | kernel"]

    def report(case, nbytes, times, kernel):
        rates = sorted(nbytes / t / 1e9 for t in times)
        lines.append(f"{case} | {statistics.median(rates):.0f} | {rates[0]:.0f} - {rates[-1]:.0f} | {kernel}")
        print(lines[-1], flush=True)

    n = 1 << 30
    for dt in (F.F32, F.U32, F.I16, F.I8):  # a * b + 1
        o, = ax = [L.Axis(n)]
        a, b = operand(dt, n, 1), operand(dt, n, 2)
        la = L.Node(F.LEAF, dt, buf=a, offset=0, stride={o: 1})
        lb = L.Node(F.LEAF, dt, buf=b, offset=0, stride={o: 1})
        one = L.Node(F.CONST, dt, imm=1.0 if dt == F.F32 else 1)
        root = L.Node(F.BINARY, dt, op=F.ADD, children=(L.Node(F.BINARY, dt, op=F.MUL, children=(la, lb)), one))
        times, k = timed(root, ax, n, dt)
        report(f"a*b+1 {F.DTYPE_NAME[dt]} 2^30", 3 * n * F.DTYPE_SIZE[dt], times, k)
        keep.clear()
    n = 1 << 31
    for src, dst in ((F.U32, F.U64), (F.I16, F.I64), (F.I8, F.I64), (F.U16, F.U64)):  # whole-array sums
        r = L.Axis(n)
        x = operand(src, n, 3)
        lf = L.Node(F.LEAF, src, buf=x, offset=0, stride={r: 1})
        root = L.Node(F.FOLD, dst, op=F.ADD, children=(L.Node(F.UNARY, dst, op=F.CAST, src_dtype=src, children=(lf,)),), red_axes=(r,), imm=0)
        times, k = timed(root, [], 1, dst)
        report(f"sum {F.DTYPE_NAME[src]}->{F.DTYPE_NAME[dst]} 2^31", n * F.DTYPE_SIZE[src], times, k)
        keep.clear()
    m = 4096
    r, c = ax = [L.Axis(m), L.Axis(m)]
    x = operand(F.U16, m * m, 4)
    times, k = timed(L.Node(F.LEAF, F.U16, buf=x, offset=0, stride={r: 1, c: m}), ax, m * m, F.U16)
    report("transpose u16 4096x4096", 2 * m * m * 2, times, k)
    ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
