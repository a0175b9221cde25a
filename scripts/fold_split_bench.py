#!/usr/bin/env python
"""Few-output integer folds on one GPU: the whole-GPU split fold (k_fold_split) against the routes these folds took before it.

    python scripts/fold_split_bench.py --compare A=path/to/libmdim_b200.so B=... [--rounds 3] [--out profiles/x.json]

runs every case once per library per round, alternating the libraries in one call (each run in its own process), writes every
run to --out and prints the median rate per case and library.  `NAME=LIB:small` runs only the reduced sizes on that library;
`--lib PATH` runs one library once and prints one JSON line per case.  Operands live on the GPU (torch allocates and fills them)
and the full sizes are larger than the 126 MB L2.  Each case is timed with CUDA events on the context's stream over repeated
collects, after one warm-up collect.  The rate is algorithmic: the bytes the fold must read, over the time of one collect.

Routes that walk a reduction with one thread (the evaluator) or a few lanes would take minutes at full size, so every headline
case also has a `small` form (2^21 - 2^22 elements), and the threshold grid (outputs x reduction length) is small throughout.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K = 1 << 16


# (name, fold dtype, source dtype, op, out [(len, stride)], red [(len, stride)], fill) — strides in source elements
def cases(full):
    s = (lambda a, b: a) if full else (lambda a, b: b)
    C = [
        ("u64-sum", "u64", "u64", "add", [], [(s(1 << 30, 1 << 21), 1)], "rand"),
        ("u32-to-u64-sum", "u64", "u32", "add", [], [(s(1 << 30, 1 << 21), 1)], "rand"),
        ("bool-count", "u64", "u8", "add", [], [(s(1 << 32, 1 << 22), 1)], "bool"),
        ("bool-any", "u8", "u8", "or", [], [(s(1 << 32, 1 << 22), 1)], "zeros"),
        ("bool-all", "u8", "u8", "and", [], [(s(1 << 32, 1 << 22), 1)], "ones"),
        ("u64-xor", "u64", "u64", "xor", [], [(s(1 << 30, 1 << 21), 1)], "rand"),
        ("u32-4-rows", "u32", "u32", "add", [(4, s(1 << 24, 1 << 20))], [(s(1 << 24, 1 << 20), 1)], "rand"),
        ("u32-4-cols", "u32", "u32", "add", [(4, 1)], [(s(1 << 24, 1 << 20), 4)], "rand"),
    ]
    if full:
        return C
    # both sides of the thresholds: outputs x reduction length (u32 sums of contiguous runs, and of columns)
    for n_out in (1, 64, 1024, 4096, 16384):
        for red in (1 << 12, 1 << 14, K, 1 << 18):
            if n_out * red > (1 << 28):
                continue
            C.append((f"grid-runs-{n_out}x{red}", "u32", "u32", "add", [(n_out, red)] if n_out > 1 else [], [(red, 1)], "rand"))
    for cols in (4, 64, 1024, 4096, 16384):
        for red in (1 << 12, 1 << 14, K, 1 << 18):
            if cols * red > (1 << 28):
                continue
            C.append((f"grid-cols-{cols}x{red}", "u32", "u32", "add", [(cols, 1)], [(red, cols)], "rand"))
    return C


def run_one(lib_path, sizes, reps_target_s=0.3):
    import numpy as np
    import torch
    from multidimension_b200 import _ffi as F
    F.LIB_PATH = lib_path
    import multidimension_b200 as P
    from multidimension_b200 import lowering as L
    from multidimension_b200.runtime import Storage

    DT = {"u8": F.U8, "u32": F.U32, "u64": F.U64}
    TT = {"u8": torch.uint8, "u32": torch.int32, "u64": torch.int64}
    OP = {"add": F.ADD, "or": F.OR, "and": F.AND, "xor": F.XOR}
    ctx = P.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream_handle())
    gen = torch.Generator(device="cuda")
    rows = []
    for full in [{"full": True, "small": False}[x] for x in sizes]:
        for name, T, Ts, op, out, red, fill in cases(full):
            gen.manual_seed(zlib.crc32(f"{name}-{full}".encode()))
            n = 1
            for ln, st in out + red:
                n = max(n, n + (ln - 1) * st)
            if fill == "bool":
                t = torch.randint(0, 2, (n,), device="cuda", dtype=torch.uint8, generator=gen)
            elif fill in ("zeros", "ones"):
                t = torch.full((n,), 0 if fill == "zeros" else 1, device="cuda", dtype=torch.uint8)
                t[n // 2] = 1 - t[n // 2]
            else:
                t = torch.randint(-(1 << 31), (1 << 31) - 1, (n,), device="cuda", dtype=TT[Ts], generator=gen)
            torch.cuda.synchronize()
            buf = Storage.wrap_device(ctx, DT[Ts], n, t.data_ptr(), keep=t)
            ax = [L.Axis(ln) for ln, _ in out + red]
            lf = L.Node(F.LEAF, DT[Ts], buf=buf, offset=0, stride={a: st for a, (_, st) in zip(ax, out + red)})
            body = lf if T == Ts else L.Node(F.UNARY, DT[T], op=F.CAST, src_dtype=DT[Ts], children=(lf,))
            node = L.Node(F.FOLD, DT[T], op=OP[op], children=(body,), red_axes=tuple(ax[len(out):]), imm=0)
            em = L.emit(node, ax[:len(out)], "device")
            o = torch.empty(max(em.out_len, 1) * 8, device="cuda", dtype=torch.uint8)
            expr, optr = em.expr, o.data_ptr()
            t0 = time.perf_counter()
            ctx.collect(expr, optr)  # warm-up (and a first timing to size the timed window)
            first = time.perf_counter() - t0
            reps = max(1, min(200, int(reps_target_s / max(first, 1e-6))))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                ctx.collect(expr, optr, F.COLLECT_ASYNC)
            e1.record(stream)
            ctx.sync()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / reps
            n_red = 1
            for ln, _ in red:
                n_red *= ln
            n_out = 1
            for ln, _ in out:
                n_out *= ln
            nbytes = n_out * n_red * F.DTYPE_SIZE[DT[Ts]]
            res = np.empty(em.out_len, dtype=np.uint8 if T == "u8" else np.uint32 if T == "u32" else np.uint64)
            ctx.download(res, optr)
            rows.append({"case": name, "size": "full" if full else "small", "outs": n_out, "red": n_red, "bytes": nbytes, "reps": reps,
                         "ms": ms, "GBps": nbytes / ms / 1e6, "kernel": ctx.last_kernel(), "route": P.runtime.describe_nodevice(expr)[1],
                         "checksum": int(np.bitwise_xor.reduce(res.view(np.uint8)))})
            print(json.dumps(rows[-1]), flush=True)
            del t, buf, o
            torch.cuda.empty_cache()
    ctx.close()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().split("\n")[0] if q.returncode == 0 else "unknown"


def compare(libs, rounds, out):
    results = {name: [] for name in libs}
    for r in range(rounds):
        for name, path in libs.items():
            path, _, only = path.partition(":")
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--lib", path, "--sizes", only or "full,small"], capture_output=True, text=True, cwd=ROOT)
            if p.returncode != 0:
                sys.exit(f"{name}: {p.stderr[-3000:]}")
            results[name].append([json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith("{")])
    doc = {"card": card(), "rounds": rounds, "libs": libs, "runs": results}
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(doc, f, indent=1)
    print("card:", doc["card"])
    keys = []
    for name in libs:
        keys += [(row["case"], row["size"]) for row in results[name][0] if (row["case"], row["size"]) not in keys]
    print(f"{'case':34s} {'size':5s} " + " ".join(f"{n + ' GB/s':>14s}" for n in libs) + "  kernels")
    for case, size in keys:
        med, kern, sums = [], [], set()
        for name in libs:
            v = sorted(row["GBps"] for run in results[name] for row in run if (row["case"], row["size"]) == (case, size))
            one = [row for row in results[name][0] if (row["case"], row["size"]) == (case, size)]
            med.append(f"{v[len(v) // 2]:14.2f}" if v else f"{'not run':>14s}")
            kern.append(one[0]["kernel"] if one else "-")
            sums |= {one[0]["checksum"]} if one else set()
        print(f"{case:34s} {size:5s} " + " ".join(med) + "  " + " | ".join(kern) + ("" if len(sums) <= 1 else "  RESULTS DIFFER"))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib")
    ap.add_argument("--sizes", default="full,small")
    ap.add_argument("--compare", nargs="+", metavar="NAME=LIB")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="JSON file for the compare mode's raw runs")
    a = ap.parse_args()
    if a.lib:
        run_one(os.path.abspath(a.lib), a.sizes.split(","))
    else:
        compare(dict(x.split("=", 1) for x in a.compare), a.rounds, a.out)
