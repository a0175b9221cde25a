#!/usr/bin/env python
"""bench.py — effective HBM GB/s of View -> collect() (BASELINE.json metric).

A step is ONE collect() of BASELINE config 2 — `a.zip(b).map(|(x,y)| x*y+1)` over two 2^30-element
f32 Arrays per GPU (12 GiB of algorithmic traffic per step per GPU) — through the C ABI.  With N>1
(torchrun, one process per GPU) the global Array is partitioned along its outermost index: every
rank collects its own 2^30-element block, no data-path collective (SURVEY.md §8e), weak scaling.

  value     device-resident: K back-to-back collects, CUDA events on the launching stream, max over ranks
  e2e       the same collect through mdim_collect_host: operands and result in pinned HOST memory,
            H2D/D2H copies inside the timed region (chunked and overlapped by the library)
  roofline  the fused elementwise kernel against the measured HBM copy rate (MEASURED_PEAKS.json)
  ops       the other BASELINE configs (transpose, gather, fold+broadcast-subtract, rank-5 chain), N=1
  scaling_ops  every SURVEY.md §8(e) row as a STRONG-scaling problem (fixed total size cut over the N ranks): ms, aggregate
            GB/s, speed-up against the same problem on ONE GPU measured in the same run, fraction of N x the measured HBM
            peak, NVLink bytes in per GPU where the op has an exchange step (all collectives through the C ABI)
  cpu_baseline   the CPU oracle (a restatement of the reference's single-threaded collect(); the Rust
            crate itself cannot be built here) on a bounded sample of the same workload

`--impl reference` times that CPU restatement alone, as the reference arm.
`--dump-outputs DIR` writes a seeded sample of config 2's result after its timed steps, so that two builds can be
compared output for output (the inputs come from fixed seeds).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np

METRIC = "effective HBM GB/s for View->collect (zip+map x*y+1 over two 2^30-element f32 Arrays per GPU)"
UNIT = "GB/s"
N_ELEMS = 1 << 30
WORKLOAD = "configs[1]: zip+map elementwise collect of two 2^30-element f32 Arrays (a.zip(b).map(|(x,y)| x*y+1))"


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


TRAFFIC_SOURCE = "profiles/traffic.json (dram__bytes_read.sum + dram__bytes_write.sum from the committed ncu --set full captures; a citation, not measured in this run)"


def known_traffic(kernel):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, device):
        self.samples, self.reasons, self.stop_flag, self.max_mhz, self.thread = [], set(), False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def start(self):
        if self.nv:
            self.stop_flag = False
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if self.thread:
            self.stop_flag = True
            self.thread.join()
            self.thread = None

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# ---- the CPU restatement (reference arm and cpu_baseline) -----------------------------------------------
CPU_BUILDS = {"": "gcc -O2 -fno-tree-vectorize -ffp-contract=off (README.md:11-12: 'not SIMD optimized')",
              "_o3": "gcc -O3 -march=x86-64-v3 -ffp-contract=off, vectoriser on (the most `cargo build --release` could do)"}


def cpu_oracle_pass(n, repeat, seed=1, variant=""):
    """Time `repeat` single-threaded passes of config 2 over an n-element sample through
    oracle/ref_shaped.c (the collect() loop as rustc would monomorphise it: bounds asserts, push with
    capacity check, separately rounded mul/add).  Returns (seconds per pass, algorithmic bytes)."""
    from helpers import refshaped_lib
    rng = np.random.default_rng(seed)
    a = rng.uniform(-1, 1, n).astype(np.float32)
    b = rng.uniform(-1, 1, n).astype(np.float32)
    out = np.empty(n, dtype=np.float32)
    lib = refshaped_lib(variant)
    times = []
    for _ in range(repeat):
        t0 = time.perf_counter()
        st = lib.ref_c2_zip_map(a.ctypes.data, b.ctypes.data, n, out.ctypes.data)
        times.append(time.perf_counter() - t0)
        assert st == 0
    want = a * b + np.float32(1)
    assert np.array_equal(out.view(np.uint32), want.view(np.uint32))
    return times, 12 * n


def cpu_ops_table():
    """The other configs on one host core (bounded samples), GB/s on algorithmic bytes."""
    from helpers import refshaped_lib
    lib = refshaped_lib()
    rng = np.random.default_rng(2)
    out = {}

    def timed(fn, nbytes, sample):
        t0 = time.perf_counter()
        assert fn() == 0
        dt = time.perf_counter() - t0
        return {"GB/s": round(nbytes / dt / 1e9, 3), "sample": sample}
    m = 4096
    a = rng.uniform(-1, 1, m * m).astype(np.float32)
    o = np.empty(m * m, np.float32)
    out["c1_transpose_4096x4096_f32"] = timed(lambda: lib.ref_c1_transpose(a.ctypes.data, m, m, o.ctypes.data), 8 * m * m, "full size")
    n3, m3 = 1 << 24, 1 << 28
    src = rng.uniform(-1, 1, m3).astype(np.float32)
    idx = rng.integers(0, m3, n3).astype(np.uint64)
    o3 = np.empty(n3, np.float32)
    out["c3_compose_gather"] = timed(lambda: lib.ref_c3_compose(idx.ctypes.data, n3, src.ctypes.data, m3, o3.ctypes.data), 16 * n3,
                                     "2^24 indices into a 2^28-element source (full: 2^28 into 2^30)")
    I, J, K = 256, 256, 256
    a4 = src[: I * J * K]
    sums = np.empty(I * J, np.float32)
    out["c4a_fold_sum_last_axis"] = timed(lambda: lib.ref_c4_fold(a4.ctypes.data, I, J, K, sums.ctypes.data), 4 * I * J * K + 4 * I * J,
                                          "(256,256,256) of (1024,1024,256)")
    mean = (sums / np.float32(K)).astype(np.float32)
    o4 = np.empty(I * J * K, np.float32)
    out["c4b_broadcast_subtract"] = timed(lambda: lib.ref_c4_sub(a4.ctypes.data, mean.ctypes.data, I, J, K, o4.ctypes.data), 8 * I * J * K + 4 * I * J,
                                          "(256,256,256) of (1024,1024,256)")
    P_, Q, R = 16, 16, 64
    a5 = src[: P_ * Q]
    w5 = src[1000: 1000 + R]
    o5 = np.empty(Q * P_ * Q * P_ * R, np.float32)
    out["c5_rank5_chain"] = timed(lambda: lib.ref_c5_chain(a5.ctypes.data, P_, Q, w5.ctypes.data, R, o5.ctypes.data), 4 * o5.size,
                                  "P=Q=16, R=64 (2^22 outputs) of P=Q=R=64 (2^30)")
    return out


def pin_to_one_core():
    try:
        cores = sorted(os.sched_getaffinity(0))
        os.sched_setaffinity(0, {cores[-1]})
    except Exception:
        pass


def run_reference(args, rank):
    if rank != 0:
        return
    pin_to_one_core()
    n = 1 << 26  # bounded sample: 2^26 of the 2^30 elements per step
    best = None
    for variant in CPU_BUILDS:  # the reference arm is the FASTER of the two builds of the same loops
        times, nbytes = cpu_oracle_pass(n, args.warmup + args.steps, variant=variant)
        timed = times[args.warmup:]
        sec_v = sum(timed) / len(timed)
        if best is None or sec_v < best[0]:
            best = (sec_v, variant)
    sec, variant = best
    v = nbytes / sec / 1e9
    sample = (f"{n} of {N_ELEMS} elements per step (same expression, same generator), single thread pinned to one core "
              f"(the reference is single-threaded by construction); build: {CPU_BUILDS[variant]}")
    emit_line({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample,
                   "note": "CPU restatement of the reference's single-threaded collect() as monomorphic loops (oracle/ref_shaped.c); the Rust crate cannot be built in this image"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample, "flags": CPU_BUILDS[variant]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ---- the B200 arm ------------------------------------------------------------------------------------------------------------
def host_memory_available():
    """Bytes of host RAM this process may still take: MemAvailable, capped by the cgroup limit when there is one."""
    avail = 1 << 62
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable:"):
                    avail = int(ln.split()[1]) * 1024
    except OSError:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            with open(lim) as f:
                v = f.read().strip()
            if v != "max":
                with open(cur) as f:
                    avail = min(avail, int(v) - int(f.read().strip()))
        except (OSError, ValueError):
            pass
    return max(avail, 0)


def bind_near_gpu(local):
    """Run this rank (and therefore first-touch its pinned staging buffers) on the NUMA node its GPU hangs off.
    -> what was found, for the e2e record."""
    info = {"numa_node": None, "cpus": None, "nodes_online": None}
    try:
        with open("/sys/devices/system/node/online") as f:
            info["nodes_online"] = f.read().strip()
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        with open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node") as f:
            node = int(f.read().strip())
        info["numa_node"] = node
        if node >= 0:
            with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
                cpus = set()
                for part in f.read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
            allowed = os.sched_getaffinity(0) & cpus
            if allowed:
                os.sched_setaffinity(0, allowed)
                info["cpus"] = len(allowed)
    except Exception as e:  # not fatal: the numbers are then whatever the default placement gives
        info["error"] = str(e)[:120]
    return info


_json_fd = None


def keep_stdout_for_json():
    """Libraries print to fd 1 (NCCL writes its version banner there): point fd 1 at stderr for the rest of
    the run and keep the original for the ONE JSON line the driver parses."""
    global _json_fd
    sys.stdout.flush()
    _json_fd = os.dup(1)
    os.dup2(2, 1)


def emit_line(obj):
    sys.stdout.flush()
    os.write(_json_fd if _json_fd is not None else 1, (json.dumps(obj) + "\n").encode())


DUMP_SAMPLE = 1 << 21  # over all ranks: 8 MiB of f32 results + 16 MiB of f64 positions


def dump_outputs(out_dir, tout, rank, world):
    """Config 2's result as the last timed collect left it: DIR/zip_map_out.npy (float32) and the positions it was read at,
    DIR/zip_map_out_index.npy (float64, exact below 2^53).  All of it when it has at most DUMP_SAMPLE / world elements,
    otherwise that many positions drawn with a fixed seed.  Under torchrun every rank writes its own block, suffixed _rank<r>."""
    import torch
    n, k = tout.numel(), DUMP_SAMPLE // world
    if n <= k:
        idx = np.arange(n)
    else:
        idx = np.unique(np.random.default_rng(0x5EED00D0).integers(0, n, k))
    got = tout[torch.from_numpy(idx).to(tout.device)].cpu().numpy()
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"zip_map_out{suffix}.npy"), got)
    np.save(os.path.join(out_dir, f"zip_map_out_index{suffix}.npy"), idx.astype(np.float64))


class Bench:
    """What every section needs: the context and its stream, the communicator, timing, buffers."""

    def __init__(self, args, rank, world, local):
        import torch
        import torch.distributed as dist
        import multidimension_b200 as P
        from multidimension_b200 import sharding
        self.args, self.rank, self.world, self.local = args, rank, world, local
        self.torch, self.dist, self.P = torch, dist, P
        torch.cuda.set_device(local)
        self.numa = bind_near_gpu(local)
        if world > 1:  # torch.distributed is plumbing only: barriers and the max over ranks of the device times
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        self.ctx = P.Context(local)
        P.set_default_context(self.ctx)
        # The collects run on the context's OWN stream (dependency-aware launches need it, csrc/launch.cuh); torch only
        # wraps it to record CUDA events there.  torch's own kernels stay on torch's stream, fenced by device syncs.
        self.stream = torch.cuda.ExternalStream(self.ctx.stream_handle(), device=local)
        self.comm = sharding.Comm.from_env(self.ctx) if world > 1 else None  # NCCL behind the C ABI (mdim_comm_init)
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world > 1:
            t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def dev_array(self, I, size, t, T):
        return self.P.Array.from_device(I, size, t.data_ptr(), T, ctx=self.ctx, keep=t)

    def out_storage(self, t, dtype):
        from multidimension_b200.runtime import Storage
        return Storage.wrap_device(self.ctx, dtype, t.numel(), t.data_ptr(), keep=t)

    def time_launches(self, fn, steps, warmup, collective=True):
        """ms per call of fn (device time, CUDA events on the launching stream, max over ranks) and kernels launched.
        collective=False: every rank times the same thing on its own (no barrier), e.g. the one-GPU reference of an op."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        if collective:
            self.barrier()
        else:
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = self.ctx.launch_count()
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        if collective:
            self.barrier()
        else:
            torch.cuda.synchronize()
        self.ctx.sync()
        ms = e0.elapsed_time(e1)
        return self.max_over_ranks(ms) / steps, self.ctx.launch_count() - l0


def main():
    keep_stdout_for_json()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every GPU measurement (the 4096x4096 transpose counts "
                                                          "one pass over its 16 rotating buffers as a step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-elems", type=int, default=30, help="elements per GPU (default 2^30 = the BASELINE config)")
    ap.add_argument("--no-ops", action="store_true", help="skip the per-op tables (configs 1, 3, 4, 5; scaling_ops)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of config 2's result "
                                                          "(float32) and its positions (float64) to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    B = Bench(args, rank, world, local)
    torch, dist, P, ctx = B.torch, B.dist, B.P, B.ctx
    from multidimension_b200 import usize, Array, _ffi as F
    from multidimension_b200.runtime import Storage
    n = 1 << args.log2_elems

    # ---- config 2, device-resident ---------------------------------------------------------------------
    g = torch.Generator(device="cuda")
    g.manual_seed(0x5EED0001 + rank)
    ta = torch.empty(n, device="cuda", dtype=torch.float32).uniform_(-1, 1, generator=g)
    tb = torch.empty(n, device="cuda", dtype=torch.float32).uniform_(-1, 1, generator=g)
    tout = torch.empty(n, device="cuda", dtype=torch.float32)
    torch.cuda.synchronize()
    a, b = B.dev_array(usize, n, ta, "f32"), B.dev_array(usize, n, tb, "f32")
    view = a.zip(b).map(lambda p: p[0] * p[1] + np.float32(1))
    plan_text = view.describe()
    st_out = B.out_storage(tout, F.F32)
    # parity gate before any number: bit-exact against separately rounded mul and add
    view.collect(out=st_out)
    want = ta * tb
    want += 1.0
    assert torch.equal(tout.view(torch.int32), want.view(torch.int32)), "config 2 result is not bit-exact"
    del want

    clocks = ClockSampler(local)
    clocks.start()
    ms_step, launches = B.time_launches(lambda: view.collect(out=st_out, flags=F.COLLECT_ASYNC), args.steps, args.warmup)
    clocks.stop()
    kernel_ran = ctx.last_kernel()
    if args.dump_outputs:  # before the sections below overwrite tout and ta
        dump_outputs(args.dump_outputs, tout, rank, world)
    alg_bytes = 12 * n
    per_gpu = alg_bytes / (ms_step * 1e-3) / 1e9
    value = per_gpu * world
    peak, peak_src = B.peak, B.peak_src

    result = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "elements_per_gpu": n, "algorithmic_bytes_per_step_per_gpu": alg_bytes,
                   "parallelism": f"outermost-index shards x{world}, no collective", "kernel": plan_text,
                   "l2": "operands (8 GiB) and result (4 GiB) are far larger than the 126 MB L2; no flush needed",
                   "parity": "bit-exact vs separately rounded f32 mul/add, checked in this run",
                   "note": "the weak-scaling headline cannot fail (no exchange); the rows that can are in scaling_ops"},
        "clocks": clocks.summary(),
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": per_gpu, "peak": peak, "unit": "GB/s", "frac": per_gpu / peak,
                     "frac_of_nominal_8000": per_gpu / 8000.0, "peak_source": peak_src,
                     "kernel": "k_eval<SigMulAddCF32, u32, V=8, R1>", "kernel_ran": kernel_ran, "traffic": known_traffic("k_eval_SigMulAddCF32"),
                     "traffic_source": TRAFFIC_SOURCE},
    }

    # ---- e2e: host buffers through mdim_collect_host ---------------------------------------------------------------------
    if not args.no_e2e:
        result["e2e"] = bench_e2e(B, ta, tb, tout, n)

    # ---- the other BASELINE configs, one line each (N=1 only) ------------------------------------------------------------------
    if not args.no_ops and world == 1:
        result["ops"] = bench_ops(B, ta, tout)

    # ---- every SURVEY §8(e) row as a strong-scaling problem, any N ------------------------------------------------------------------
    if not args.no_ops:
        del tb, b, view
        torch.cuda.empty_cache()
        so = bench_scaling_ops(B, ta, tout)
        if rank == 0:
            result["scaling_ops"] = so

    # ---- CPU restatement beside it (rank 0, N=1) -----------------------------------------------------------------------------------
    if not args.no_cpu and world == 1 and rank == 0:
        pin_to_one_core()
        sample_n = 1 << 28
        best = None
        per_build = {}
        for variant, flags in CPU_BUILDS.items():
            times, nbytes = cpu_oracle_pass(sample_n, 2, variant=variant)
            v = nbytes / min(times) / 1e9
            per_build[flags] = round(v, 3)
            if best is None or v > best[0]:
                best = (v, flags)
        result["cpu_baseline"] = {"value": best[0], "unit": UNIT, "cores": 1, "kind": "port", "flags": best[1], "GB/s_per_build": per_build,
                                  "sample": f"{sample_n} of {N_ELEMS} elements of config 2, 2 passes (best) per build, the faster build reported, single thread; "
                                            f"oracle/ref_shaped.c restates the reference's collect() loop (no Rust toolchain in this image; "
                                            f"the reference is single-threaded by construction)",
                                  "host_cores_available": os.cpu_count(), "ops": cpu_ops_table()}

    if rank == 0:
        emit_line(result)
    if B.comm is not None:
        B.comm.close()
    if world > 1:
        dist.destroy_process_group()


def bench_e2e(B, ta, tb, tout, n):
    """Config 2 through mdim_collect_host: operands and result in pinned HOST memory, copies inside the timed region.
    Beside it, the raw ceiling of this box for the same bytes: plain concurrent cudaMemcpyAsync H2D + D2H of the same
    buffers on every rank at once (what PCIe and the host memory system give N GPUs at the same time)."""
    import gc
    from multidimension_b200 import usize, Array, _ffi as F
    from multidimension_b200.runtime import Storage
    torch, ctx, world, args = B.torch, B.ctx, B.world, B.args
    # Every rank pins 12 bytes per element: the full 2^30-element config when the box's RAM allows it for ALL ranks.
    ne, avail = n, host_memory_available()
    while ne > (1 << 24) and 12 * ne * world * 1.25 > avail:
        ne //= 2
    ha, hb, ho = (Storage.pinned(ctx, F.F32, ne) for _ in range(3))
    ctx.download(ha.host, ta.data_ptr())
    ctx.download(hb.host, tb.data_ptr())
    hview = Array(usize, ne, ha, "f32").zip(Array(usize, ne, hb, "f32")).map(lambda p: p[0] * p[1] + np.float32(1))
    e2e_steps = args.e2e_steps or max(1, min(args.steps, 5))
    hview.collect(out=ho)  # warm-up: grows the staging arena
    B.barrier()
    l0 = ctx.launch_count()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        hview.collect(out=ho)
    B.barrier()
    sec = B.max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    chk = torch.from_numpy(ho.host[: 1 << 22]).cuda()
    assert torch.equal(chk.view(torch.int32), tout[: 1 << 22].view(torch.int32)), "e2e result differs from the device-resident result"
    out = {"value": 12 * ne * world / sec / 1e9, "unit": UNIT, "h2d_bytes_per_step": 8 * ne, "d2h_bytes_per_step": 4 * ne,
           "ms_per_step": sec * 1e3, "steps": e2e_steps, "kernels_per_step": (ctx.launch_count() - l0) // e2e_steps,
           "pcie_gbs": 12 * ne / sec / 1e9, "elements_per_gpu": ne, "full_config": ne == n, "numa": B.numa,
           "host_ram_available_gb": round(avail / 2**30, 1)}
    # raw copy ceiling, same buffers, same concurrency: H2D of both operands on one stream, D2H of the result on another
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
    t_ha, t_hb, t_ho = (torch.from_numpy(s.host) for s in (ha, hb, ho))
    da, db = ta[:ne], tb[:ne]

    def raw():
        with torch.cuda.stream(s_up):
            da.copy_(t_ha, non_blocking=True)
            db.copy_(t_hb, non_blocking=True)
        with torch.cuda.stream(s_dn):
            t_ho.copy_(tout[:ne], non_blocking=True)
    raw()
    B.barrier()
    t0 = time.perf_counter()
    for _ in range(2):
        raw()
    B.barrier()
    raw_sec = B.max_over_ranks((time.perf_counter() - t0) / 2)
    out["raw_copy_ceiling_pcie_gbs"] = 12 * ne / raw_sec / 1e9
    out["frac_of_raw_copy_ceiling"] = out["pcie_gbs"] / out["raw_copy_ceiling_pcie_gbs"]
    out["note"] = ("pcie_gbs = bytes crossing PCIe per second per GPU through mdim_collect_host; raw_copy_ceiling = the same bytes as bare "
                   "cudaMemcpyAsync H2D+D2H on all ranks at once (no kernel): the host-memory / PCIe ceiling of this box at this N")
    del ha, hb, ho, hview, t_ha, t_hb, t_ho
    gc.collect()  # the pinned memory must be released now, not inside a later timed region
    torch.cuda.synchronize()
    return out


def bench_ops(B, ta, tout):
    """Configs 1, 3, 4, 5 of BASELINE.json at full size on one GPU: GB/s on algorithmic bytes, each parity-gated."""
    import multidimension_b200 as P
    from multidimension_b200 import usize, Array, Scalar, Add, fold_rows, _ffi as F
    torch, ctx, peak, args = B.torch, B.ctx, B.peak, B.args
    dev_array, out_storage, time_launches = B.dev_array, B.out_storage, B.time_launches
    ops = {}
    steps = args.steps

    def line(name, alg_bytes, ms, plan, **extra):
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        ops[name] = dict({"GB/s": round(gbs, 1), "frac_of_measured_peak": round(gbs / peak, 4), "frac_of_nominal_8000": round(gbs / 8000.0, 4),
                          "ms": round(ms, 5), "algorithmic_bytes": alg_bytes, "kernel": plan, "kernel_ran": ctx.last_kernel()}, **extra)

    # C1: 4096x4096 f32 transpose; 16 rotating source/destination pairs (2 GiB) keep it out of L2
    R = 16
    n1 = 4096
    srcs = ta[: R * n1 * n1].view(R, n1 * n1)
    dsts = tout[: R * n1 * n1].view(R, n1 * n1)
    views = [dev_array((usize, usize), (n1, n1), srcs[k], "f32").transpose((), usize, usize, ()) for k in range(R)]
    outs = [out_storage(dsts[k], F.F32) for k in range(R)]
    views[0].collect(out=outs[0])
    assert torch.equal(dsts[0].view(n1, n1), srcs[0].view(n1, n1).t()), "transpose mismatch"
    state = {"k": 0}
    prepared = [views[k].prepare(out=outs[k], flags=F.COLLECT_ASYNC) for k in range(R)]  # lowered once: a 20 us kernel must not wait for Python

    def tr():
        k = state["k"] = (state["k"] + 1) % R
        prepared[k].run()
    ms, _ = time_launches(tr, steps * R, R)
    line("c1_transpose_4096x4096_f32", 2 * 4 * n1 * n1, ms, views[0].describe(), l2="16 rotating buffer pairs (2 GiB total)",
         launch="independent launches overlap their neighbours' tails (dependency-aware programmatic launch, csrc/launch.cuh)")
    for k in range(R):  # every pair is still a correct transpose after the overlapped launches
        assert torch.equal(dsts[k].view(n1, n1), srcs[k].view(n1, n1).t()), "transpose mismatch after back-to-back launches"
    n16 = 16384
    v16 = dev_array((usize, usize), (n16, n16), ta[: n16 * n16], "f32").transpose((), usize, usize, ())
    p16 = v16.prepare(out=out_storage(tout[: n16 * n16], F.F32), flags=F.COLLECT_ASYNC)
    p16.run()
    ctx.sync()
    assert torch.equal(tout[: n16 * n16].view(n16, n16), ta[: n16 * n16].view(n16, n16).t()), "transpose 16384 mismatch"
    ms, _ = time_launches(p16.run, steps, 3)
    line("c1_transpose_16384x16384_f32", 2 * 4 * n16 * n16, ms, v16.describe())

    # C3: compose — 2^28 uniform random usize indices into the 2^30-element f32 Array
    n3 = 1 << 28
    g = torch.Generator(device="cuda")
    g.manual_seed(0x5EED0003)
    tidx = torch.randint(0, ta.numel(), (n3,), device="cuda", dtype=torch.int64, generator=g)
    torch.cuda.synchronize()
    idx = dev_array(usize, n3, tidx, usize)
    src = dev_array(usize, ta.numel(), ta, "f32")
    v3 = idx.compose(src)
    o3 = out_storage(tout[:n3], F.F32)
    v3.collect(out=o3)
    assert torch.equal(tout[:n3], ta[tidx]), "gather mismatch"
    torch.cuda.synchronize()
    ms, _ = time_launches(lambda: v3.collect(out=o3, flags=F.COLLECT_ASYNC), steps, 3)
    line("c3_compose_gather_2^28_from_2^30", 8 * n3 + 4 * n3 + 4 * n3, ms, v3.describe(),
         dram_line_model_bytes=8 * n3 + 4 * n3 + 128 * n3, dram_line_model_GBs=round((8 + 4 + 128) * n3 / (ms * 1e-3) / 1e9, 1),
         note="a uniform-random 4-byte read over a 4 GiB source moves a whole 128-byte line from DRAM (ncu: 134 B per element, profiles/r2_gather_probe.md); "
              "the algorithmic 16 B per element can therefore reach at most 16/140 of the DRAM rate")
    del tidx, idx, v3
    torch.cuda.empty_cache()

    # C4: (1024,1024,256) f32: sum over the last index (sequential order) and subtract the mean
    shape = (1024, 1024, 256)
    n4 = shape[0] * shape[1] * shape[2]
    t4 = ta[:n4]
    t4.uniform_(0, 1)
    torch.cuda.synchronize()
    a4 = dev_array((usize, usize, usize), shape, t4, "f32")
    sums = fold_rows(a4, (usize, usize), usize, Add, np.float32(0))
    tsum = torch.empty(shape[0] * shape[1], device="cuda", dtype=torch.float32)
    osum = out_storage(tsum, F.F32)
    sums.collect(out=osum)
    ref64 = t4.view(-1, 256).double().sum(dim=1)
    rel = ((tsum.double() - ref64).abs() / ref64.abs()).max().item()  # informational: error of the SEQUENTIAL f32 sum itself
    rows = torch.arange(0, shape[0] * shape[1], 251, device="cuda")      # parity: bit-exact vs a sequential f32 sum on the host
    seq = np.add.accumulate(t4.view(-1, 256)[rows].cpu().numpy(), axis=1, dtype=np.float32)[:, -1]
    assert np.array_equal(seq.view(np.uint32), tsum[rows].cpu().numpy().view(np.uint32)), "fold is not in sequential order"
    torch.cuda.synchronize()
    ms, _ = time_launches(lambda: sums.collect(out=osum, flags=F.COLLECT_ASYNC), steps, 3)
    line("c4a_fold_sum_last_axis", 4 * n4 + 4 * shape[0] * shape[1], ms, sums.describe(), max_rel_err_vs_f64=rel)
    fused = a4 - (sums / Scalar(256.0, "f32")).iso((usize, usize, ()))
    o4 = out_storage(tout[:n4], F.F32)
    fused.collect(out=o4)
    want = t4.view(-1, 256) - (tsum / 256.0).unsqueeze(1)
    assert torch.equal(tout[:n4].view(-1, 256), want), "fused fold+subtract mismatch"
    del want
    torch.cuda.synchronize()
    ms, _ = time_launches(lambda: fused.collect(out=o4, flags=F.COLLECT_ASYNC), steps, 3)
    line("c4c_fold_mean_subtract_fused", 8 * n4, ms, fused.describe())
    means = dev_array((usize, usize), shape[:2], tsum, "f32")
    sub = a4 - means.iso((usize, usize, ()))
    ms, _ = time_launches(lambda: sub.collect(out=o4, flags=F.COLLECT_ASYNC), steps, 3)
    line("c4b_broadcast_subtract", 8 * n4 + 4 * shape[0] * shape[1], ms, sub.describe(flags=0))

    # C5: rank-5 chain transpose -> diagonal -> broadcast -> map, P=Q=R=64: 2^30 outputs, write-bound
    Pn = Qn = Rn = 64
    ta5 = torch.empty(Pn * Qn, device="cuda", dtype=torch.float32).uniform_(-1, 1)
    tw5 = torch.empty(Rn, device="cuda", dtype=torch.float32).uniform_(-1, 1)
    torch.cuda.synchronize()
    a5 = dev_array((usize, usize), (Pn, Qn), ta5, "f32")
    w5 = dev_array(usize, Rn, tw5, "f32")
    v5 = (a5.transpose((), usize, usize, ()).diagonal(np.float32(0)).iso((((usize, usize), (usize, usize)), ()))
          .zip(w5.iso(((), usize))).map(lambda p: p[0] * p[1] + np.float32(1)))
    o5 = out_storage(tout, F.F32)
    v5.collect(out=o5)
    eye = torch.eye(Pn * Qn, device="cuda", dtype=torch.float32)
    t_qp = ta5.view(Pn, Qn).t().reshape(-1)
    d = (eye * t_qp.unsqueeze(0))  # [(q,p),(q',p')]
    want5 = d.reshape(-1, 1) * tw5.view(1, Rn)
    want5 += 1.0
    assert torch.equal(tout.view(-1, Rn), want5), "rank-5 chain mismatch"
    del want5, d, eye
    torch.cuda.synchronize()
    ms, _ = time_launches(lambda: v5.collect(out=o5, flags=F.COLLECT_ASYNC), steps, 3)
    line("c5_rank5_transpose_diagonal_broadcast_map", 4 * (1 << 30) + 4 * Pn * Qn + 4 * Rn, ms, v5.describe())
    ms, _ = time_launches(lambda: v5.collect(out=o5, flags=F.COLLECT_ASYNC | F.COLLECT_NO_JIT), steps, 3)
    line("c5_rank5_chain_prebuilt_signature_only", 4 * (1 << 30) + 4 * Pn * Qn + 4 * Rn, ms, v5.describe(flags=F.COLLECT_NO_JIT),
         note="MDIM_COLLECT_NO_JIT: the pre-built kernel, without the NVRTC shape specialisation")
    return ops


def bench_scaling_ops(B, ta, tout):
    """Every SURVEY.md §8(e) row as a strong-scaling problem: a FIXED total problem cut over the N ranks along the outermost
    index.  Per row: ms (device time, max over ranks, any collective included), aggregate GB/s on algorithmic bytes, the
    same problem on ONE GPU timed in the same run (`n1_ms`) and the speed-up against it, the fraction of N x the measured
    HBM peak, and the NVLink bytes each GPU pulls in where there is an exchange.  Every collective goes through the C ABI."""
    import multidimension_b200 as P
    from multidimension_b200 import usize, Array, Scalar, Add, fold_rows, sharding, _ffi as F
    from multidimension_b200.runtime import Storage
    torch, ctx, comm, world, rank, peak = B.torch, B.ctx, B.comm, B.world, B.rank, B.peak
    dev_array, out_storage, time_launches = B.dev_array, B.out_storage, B.time_launches
    rows = {}
    steps = B.args.steps

    def row(name, alg_bytes, ms, n1_ms, kernel, nvlink_in_bytes=0, **extra):
        gbs = alg_bytes / (ms * 1e-3) / 1e9
        r = {"ms": round(ms, 5), "GB/s": round(gbs, 1), "n1_ms": round(n1_ms, 5), "speedup_vs_n1": round(n1_ms / ms, 3),
             "frac_of_measured_peak": round(gbs / (peak * world), 4), "algorithmic_bytes": alg_bytes, "kernel": kernel, "kernel_ran": ctx.last_kernel()}
        if nvlink_in_bytes:
            r["nvlink_in_gbs_per_gpu"] = round(nvlink_in_bytes / (ms * 1e-3) / 1e9, 1)
        r.update(extra)
        rows[name] = r

    # replicated operands: the same bits on every rank (fixed seed), so every parity check is local
    g = torch.Generator(device="cuda")
    g.manual_seed(0x5EED00AA)
    rep = ta
    rep.uniform_(-1, 1, generator=g)
    torch.cuda.synchronize()
    full_buf = torch.empty(1 << 30, device="cuda", dtype=torch.float32)

    # ---- C1: 16384^2 transpose, each rank collecting its block of the transposed rows ------------------------------------------
    M = 16384
    whole = dev_array((usize, usize), (M, M), rep[: M * M], "f32").transpose((), usize, usize, ())
    lo, hi = sharding.shard_bounds(M, world, rank)
    want_t = rep[: M * M].view(M, M).t()[lo:hi]
    ot = out_storage(tout[: (hi - lo) * M], F.F32)
    p1 = whole.prepare(out=out_storage(tout[: M * M], F.F32), flags=F.COLLECT_ASYNC)
    n1_ms, _ = time_launches(p1.run, steps, 3, collective=False)
    mine = sharding.shard_view(whole, rank, world)
    pm = mine.prepare(out=ot, flags=F.COLLECT_ASYNC)
    pm.run(); ctx.sync()
    assert torch.equal(tout[: (hi - lo) * M].view(hi - lo, M), want_t), "sharded transpose (replicated source) mismatch"
    ms, _ = time_launches(pm.run, steps, 3)
    row("c1_transpose_16384_source_replicated", 8 * M * M, ms, n1_ms, mine.describe(), note="no exchange: every rank reads its columns of its own replica")
    if world > 1:
        tblock = M * M // world  # row-sharded: this rank owns rows [rank*M/world, ...) = a slice of `rep` (same global matrix)
        mine_rows = rep[rank * tblock:(rank + 1) * tblock]
        local = Storage.wrap_device(ctx, F.F32, tblock, mine_rows.data_ptr(), keep=rep)
        tpeers = sharding.PeerStorage(F.F32, M * M, comm.peer_table(local.dptr, local.nbytes), tblock, keep=rep, ctx=ctx)
        vt = sharding.shard_view(Array((usize, usize), (M, M), tpeers, "f32").transpose((), usize, usize, ()), rank, world)
        pt = vt.prepare(out=ot, flags=F.COLLECT_ASYNC)
        pt.run(); ctx.sync()
        assert torch.equal(tout[: (hi - lo) * M].view(hi - lo, M), want_t), "peer-mapped transpose mismatch"
        ms, _ = time_launches(pt.run, steps, 3)
        remote = 4 * M * M // world * (world - 1) // world
        row("c1_transpose_16384_source_row_sharded_peer_mapped", 8 * M * M, ms, n1_ms, vt.describe(), nvlink_in_bytes=remote,
            note="the all-to-all is inside the kernel: every tile is fetched by TMA from the GPU that owns those rows")
        whole_ag = full_buf[: M * M]
        vt2 = sharding.shard_view(dev_array((usize, usize), (M, M), whole_ag, "f32").transpose((), usize, usize, ()), rank, world)
        pt2 = vt2.prepare(out=ot, flags=F.COLLECT_ASYNC)
        blk_st, full_st = out_storage(mine_rows, F.F32), out_storage(whole_ag, F.F32)

        def ag_then_transpose():
            comm.all_gather_into(full_st, blk_st)
            pt2.run()
        ag_then_transpose(); ctx.sync()
        assert torch.equal(tout[: (hi - lo) * M].view(hi - lo, M), want_t), "all-gather + transpose mismatch"
        ms, _ = time_launches(ag_then_transpose, steps, 3)
        row("c1_transpose_16384_source_row_sharded_allgather_first", 8 * M * M, ms, n1_ms, vt2.describe(), nvlink_in_bytes=4 * M * M // world * (world - 1),
            note="mdim_allgather (NCCL) of the 1 GiB source, then the local block transpose: the north star's baseline route")

    # ---- C3: compose, 2^28 indices (sharded) into the 2^30-element source ------------------------------------------------------------
    n_src, n3 = 1 << 30, 1 << 28
    gi = torch.Generator(device="cuda")
    gi.manual_seed(0x5EED0003)
    tidx_all = torch.randint(0, n_src, (n3,), device="cuda", dtype=torch.int64, generator=gi)  # same indices on every rank
    torch.cuda.synchronize()
    src_rep = dev_array(usize, n_src, rep, "f32")
    v_all = dev_array(usize, n3, tidx_all, usize).compose(src_rep)
    p_all = v_all.prepare(out=out_storage(tout[:n3], F.F32), flags=F.COLLECT_ASYNC)
    n1_ms, _ = time_launches(p_all.run, steps, 2, collective=False)
    ilo, ihi = sharding.shard_bounds(n3, world, rank)
    tidx = tidx_all[ilo:ihi]
    idx = dev_array(usize, ihi - ilo, tidx, usize)
    o3 = out_storage(tout[: ihi - ilo], F.F32)
    want3 = rep[tidx]
    v3 = idx.compose(src_rep)
    p3 = v3.prepare(out=o3, flags=F.COLLECT_ASYNC)
    p3.run(); ctx.sync()
    assert torch.equal(tout[: ihi - ilo], want3), "sharded gather (replicated source) mismatch"
    ms, _ = time_launches(p3.run, steps, 2)
    row("c3_compose_source_replicated", 16 * n3, ms, n1_ms, v3.describe(), note="indices and result sharded, 4 GiB source replicated: no exchange")
    if world > 1:
        block = n_src // world
        local = Storage.wrap_device(ctx, F.F32, block, rep[rank * block:(rank + 1) * block].data_ptr(), keep=rep)
        peers = sharding.PeerStorage(F.F32, n_src, comm.peer_table(local.dptr, local.nbytes), block, keep=rep, ctx=ctx)
        vp = idx.compose(Array(usize, n_src, peers, "f32"))
        pp = vp.prepare(out=o3, flags=F.COLLECT_ASYNC)
        pp.run(); ctx.sync()
        assert torch.equal(tout[: ihi - ilo], want3), "peer-mapped gather mismatch"
        ms_peer, _ = time_launches(pp.run, steps, 2)
        row("c3_compose_source_sharded_peer_mapped", 16 * n3, ms_peer, n1_ms, vp.describe(), nvlink_in_bytes=4 * (ihi - ilo) * (world - 1) // world,
            note="the gather kernel reads each element from the owning GPU over NVLink (32-byte sectors on the wire)")
        v2 = idx.compose(dev_array(usize, n_src, full_buf, "f32"))
        p2 = v2.prepare(out=o3, flags=F.COLLECT_ASYNC)
        blk_st, full_st = out_storage(rep[rank * block:(rank + 1) * block], F.F32), out_storage(full_buf, F.F32)

        def ag_then_gather():
            comm.all_gather_into(full_st, blk_st)
            p2.run()
        ag_then_gather(); ctx.sync()
        assert torch.equal(tout[: ihi - ilo], want3), "all-gather + gather mismatch"
        ms_ag, _ = time_launches(ag_then_gather, steps, 2)
        row("c3_compose_source_sharded_allgather_first", 16 * n3, ms_ag, n1_ms, v2.describe(), nvlink_in_bytes=4 * block * (world - 1),
            note="mdim_allgather (NCCL) of the 4 GiB source, then a local gather: the north star's route")
        route = sharding.choose_compose_route(ihi - ilo, 4 * n_src, world)
        row("c3_compose_source_sharded_planner_choice", 16 * n3, ms_peer if route == "peer" else ms_ag, n1_ms, f"route={route}",
            note="sharding.choose_compose_route: cost model from the measured rates (random reads over NVLink vs NCCL all-gather + local gather)",
            chose_the_faster=bool((route == "peer") == (ms_peer <= ms_ag)))
    del tidx_all, tidx, idx, want3, v_all, p_all
    torch.cuda.empty_cache()

    # ---- C4: (1024,1024,256): fold over the LAST axis + broadcast-subtract of the mean, rows sharded (no exchange) ---------------------
    shape = (1024, 1024, 256)
    n4 = shape[0] * shape[1] * shape[2]
    t4 = rep[:n4]
    g4 = torch.Generator(device="cuda")
    g4.manual_seed(0x5EED0004)
    t4.uniform_(0, 1, generator=g4)  # sums far from zero, so that a relative error means something
    torch.cuda.synchronize()

    def fused_of(arr):
        s = fold_rows(arr, (usize, usize), usize, Add, np.float32(0))
        return arr - (s / Scalar(256.0, "f32")).iso((usize, usize, ()))
    f_all = fused_of(dev_array((usize, usize, usize), shape, t4, "f32"))
    pf_all = f_all.prepare(out=out_storage(tout[:n4], F.F32), flags=F.COLLECT_ASYNC)
    n1_ms, _ = time_launches(pf_all.run, steps, 3, collective=False)
    rlo, rhi = sharding.shard_bounds(shape[0], world, rank)
    nb = (rhi - rlo) * shape[1] * shape[2]
    blk4 = t4[rlo * shape[1] * shape[2]: rhi * shape[1] * shape[2]]
    f_mine = fused_of(dev_array((usize, usize, usize), (rhi - rlo, shape[1], shape[2]), blk4, "f32"))
    pf = f_mine.prepare(out=out_storage(tout[:nb], F.F32), flags=F.COLLECT_ASYNC)
    pf.run(); ctx.sync()
    some = torch.arange(0, (rhi - rlo) * shape[1], 997, device="cuda")
    seq = np.add.accumulate(blk4.view(-1, 256)[some].cpu().numpy(), axis=1, dtype=np.float32)[:, -1]
    want = blk4.view(-1, 256)[some].cpu().numpy() - (seq / np.float32(256.0))[:, None]
    assert np.array_equal(tout[:nb].view(-1, 256)[some].cpu().numpy().view(np.uint32), want.view(np.uint32)), "sharded fused fold+subtract mismatch"
    torch.cuda.synchronize()
    ms, _ = time_launches(pf.run, steps, 3)
    row("c4_fold_last_axis_mean_subtract_rows_sharded", 8 * n4, ms, n1_ms, f_mine.describe(), note="the folded axis is local to every row: no exchange")

    # ---- C4': fold over the SHARDED (outermost) axis of the same Array -----------------------------------------------------------------
    I, J, K = shape
    fold0_all = fold_rows(dev_array((usize, usize, usize), shape, t4, "f32").transpose((), (usize, usize), usize, ()).iso(((usize, usize), usize)),
                          (usize, usize), usize, Add, np.float32(0))
    tfull = torch.empty(J * K, device="cuda", dtype=torch.float32)
    p0 = fold0_all.prepare(out=out_storage(tfull, F.F32), flags=F.COLLECT_ASYNC)
    n1_ms, _ = time_launches(p0.run, steps, 3, collective=False)
    alg0 = 4 * n4 + 4 * J * K
    if world == 1:
        row("c4_fold_sharded_axis", alg0, n1_ms, n1_ms, fold0_all.describe(), note="one GPU: a sequential fold over the outermost axis (strided rows)")
    else:
        ib = I // world
        a_blk = dev_array((usize, usize, usize), (ib, J, K), t4[rank * ib * J * K:(rank + 1) * ib * J * K], "f32")
        part_view = fold_rows(a_blk.transpose((), (usize, usize), usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, Add, np.float32(0))
        tpart = torch.empty(J * K, device="cuda", dtype=torch.float32)
        spart = out_storage(tpart, F.F32)
        ppart = part_view.prepare(out=spart, flags=F.COLLECT_ASYNC)

        def fold_allreduce():
            ppart.run()
            comm.all_reduce(spart, "sum")
        fold_allreduce(); ctx.sync()
        ref = t4.view(I, J * K).double().sum(dim=0)
        rel = ((tpart.double() - ref).abs() / ref.abs()).max().item()
        p0.run(); ctx.sync()  # the reference's order: ONE sequential f32 chain over the whole axis
        rel_seq = ((tfull.double() - ref).abs() / ref.abs()).max().item()
        diff = (tpart.double() - tfull.double()).abs() / tfull.double().abs()
        # Parity contract (north star): within 1e-6 relative of the reference's collect() for f32 reductions.  The sequential
        # f32 chain itself is ~1.1e-6 away from the exact sum on the worst of 2^18 columns, so the reassociated sum is held to
        # its ACCURACY (error vs the exact sum no worse than the reference order's own), and the distance between the two orders is
        # reported: max over the 2^18 columns and the fraction of columns beyond 1e-6.  The peer-mapped route below is bit-exact.
        assert rel <= max(1.5 * rel_seq, 2e-6), f"sharded-axis fold: error vs f64 {rel}, the sequential order's own is {rel_seq}"
        ms, _ = time_launches(fold_allreduce, steps, 3)
        row("c4_fold_sharded_axis_allreduce", alg0, ms, n1_ms, part_view.describe(), nvlink_in_bytes=4 * J * K, max_rel_err_vs_f64=rel,
            reference_order_max_rel_err_vs_f64=rel_seq, max_rel_diff_vs_reference_order=diff.max().item(),
            fraction_of_outputs_beyond_1e_6=(diff > 1e-6).double().mean().item(),
            note="per-rank partial fold + mdim_allreduce (NCCL) of 1 MiB: reassociated across ranks (1e-6 tolerance); latency-bound")
        fpeers = sharding.PeerStorage(F.F32, n4, comm.peer_table(t4[rank * ib * J * K:].data_ptr(), 4 * ib * J * K), ib * J * K, keep=rep, ctx=ctx)
        whole3 = Array((usize, usize, usize), shape, fpeers, "f32")
        exact = sharding.shard_view(fold_rows(whole3.transpose((), (usize, usize), usize, ()).iso(((usize, usize), usize)), (usize, usize), usize, Add, np.float32(0)), rank, world)
        j_lo, j_hi = sharding.shard_bounds(J, world, rank)
        texact = torch.empty((j_hi - j_lo) * K, device="cuda", dtype=torch.float32)
        px = exact.prepare(out=out_storage(texact, F.F32), flags=F.COLLECT_ASYNC)
        px.run(); ctx.sync()
        p0.run(); ctx.sync()  # the one-GPU sequential fold of the same (replicated) data is the bit-exact reference
        assert torch.equal(texact, tfull.view(J, K)[j_lo:j_hi].reshape(-1)), "peer-mapped fold over the sharded axis is not bit-exact"
        ms, _ = time_launches(px.run, steps, 3)
        row("c4_fold_sharded_axis_peer_mapped_bit_exact", alg0, ms, n1_ms, exact.describe(), nvlink_in_bytes=4 * n4 // world * (world - 1) // world,
            note="every rank folds ITS block of the result over all ranks' rows in index order, reading the peers over NVLink: bit-identical to the reference")

    if world > 1:
        # the same bit-exact fold as ONE fused kernel per GPU: the running values travel rank to rank over NVLink, pipelined
        # over column slices (csrc/k_fold_ring.cu); the result lands on EVERY rank
        tring = torch.empty(J * K, device="cuda", dtype=torch.float32)
        sring = out_storage(tring, F.F32)
        blk_rows = out_storage(t4[rank * ib * J * K:(rank + 1) * ib * J * K], F.F32)

        ring, _ = comm.prepare_fold_sharded_axis(blk_rows, ib, J * K, P.Add, np.float32(0), out=sring)
        ring(); ctx.sync(); comm.fold_status()
        assert torch.equal(tring, tfull), "pipelined ring fold over the sharded axis is not bit-exact"
        ms, _ = time_launches(ring, steps, 3)
        comm.fold_status()
        row("c4_fold_sharded_axis_ring_pipelined_bit_exact", alg0, ms, n1_ms, "k_fold_ring (mdim_fold_sharded_axis)", nvlink_in_bytes=4 * J * K,
            note="ONE fused kernel per GPU: rank r continues rank r-1's running values slice by slice (TMA row tiles, flags in peer memory); "
                 "bit-identical to the reference's sequential chain, replicated result, no NCCL call")

    if world > 1:
        # the all-reduce route as ONE fused kernel per GPU (csrc/k_fold_xchg.cu): sequential per-rank partial folds, combined in
        # RANK ORDER inside the kernel from flag-in-data packets in peer memory — deterministic, checked bit for bit against that order
        tblk = torch.empty(J * K, device="cuda", dtype=torch.float32)
        blocked, _ = comm.prepare_fold_sharded_axis(blk_rows, ib, J * K, P.Add, np.float32(0), out=out_storage(tblk, F.F32), blocked=True)
        blocked(); ctx.sync(); comm.fold_status()
        want_blk = None
        for r in range(world):
            pr = torch.full((J * K,), 0.0 if r == 0 else -0.0, device="cuda", dtype=torch.float32)
            for i in range(r * ib, (r + 1) * ib):
                pr = pr + t4.view(I, J * K)[i]
            want_blk = pr if r == 0 else want_blk + pr
        assert torch.equal(tblk.view(torch.int32), want_blk.view(torch.int32)), "blocked fold over the sharded axis differs from the rank-ordered combination"
        diff_b = (tblk.double() - tfull.double()).abs() / tfull.double().abs()
        ms, _ = time_launches(blocked, steps, 3)
        comm.fold_status()
        row("c4_fold_sharded_axis_blocked_in_kernel_allreduce", alg0, ms, n1_ms, "k_fold_xchg (mdim_fold_sharded_axis_blocked)", nvlink_in_bytes=8 * J * K * (world - 1),
            max_rel_diff_vs_reference_order=diff_b.max().item(), fraction_of_outputs_beyond_1e_6=(diff_b > 1e-6).double().mean().item(),
            note="ONE fused kernel per GPU: sequential per-rank partial folds + an all-reduce in rank order inside the kernel (16-byte "
                 "flag-in-data packets into peer HBM, no fence, no NCCL call); reassociated at the rank boundaries only, deterministic")

    # ---- C5: the rank-5 chain, 2^30 outputs cut into N blocks of the outermost index -------------------------------------------------
    Pn = Qn = Rn = 64
    g5 = torch.Generator(device="cuda")
    g5.manual_seed(0x5EED0005)
    ta5 = torch.empty(Pn * Qn, device="cuda", dtype=torch.float32).uniform_(-1, 1, generator=g5)
    tw5 = torch.empty(Rn, device="cuda", dtype=torch.float32).uniform_(-1, 1, generator=g5)
    torch.cuda.synchronize()
    v5 = (dev_array((usize, usize), (Pn, Qn), ta5, "f32").transpose((), usize, usize, ()).diagonal(np.float32(0))
          .iso((((usize, usize), (usize, usize)), ())).zip(dev_array(usize, Rn, tw5, "f32").iso(((), usize))).map(lambda p: p[0] * p[1] + np.float32(1)))
    p5_all = v5.prepare(out=out_storage(full_buf, F.F32), flags=F.COLLECT_ASYNC)
    n1_ms, _ = time_launches(p5_all.run, steps, 3, collective=False)
    mine5 = sharding.shard_view(v5, rank, world)
    n5 = mine5.len()
    p5 = mine5.prepare(out=out_storage(tout[:n5], F.F32), flags=F.COLLECT_ASYNC)
    p5.run(); ctx.sync()
    q_lo, q_hi = sharding.shard_bounds(Qn, world, rank)
    eye = torch.eye(Pn * Qn, device="cuda", dtype=torch.float32)[q_lo * Pn:q_hi * Pn]
    want5 = (eye * ta5.view(Pn, Qn).t().reshape(-1).unsqueeze(0)).reshape(-1, 1) * tw5.view(1, Rn)
    want5 += 1.0
    assert torch.equal(tout[:n5].view(-1, Rn), want5), "sharded rank-5 chain mismatch"
    del want5, eye
    torch.cuda.synchronize()
    ms, _ = time_launches(p5.run, steps, 3)
    row("c5_rank5_chain_outermost_sharded", 4 * (1 << 30), ms, n1_ms, mine5.describe(), note="BASELINE configs[4]: write-bound, tiny replicated operands, no exchange")
    if comm is not None:
        comm.close_peers()
    return rows


if __name__ == "__main__":
    main()
