"""bench.py's output contract, checked on the CPU-runnable arm (`--impl reference`): exactly ONE line on
stdout, valid JSON, carrying the keys the driver reads.  The B200 arm prints through the same function."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return p.stdout


def test_reference_arm_prints_one_json_line():
    out = _run()
    lines = out.splitlines()
    assert len(lines) == 1, out
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    """Under torchrun (N > 1) rank 0 alone runs the CPU arm; the other ranks exit 0 without output."""
    out = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29533"})
    assert out.strip() == ""


def test_zero_steps_is_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode == 2 and "--steps" in p.stderr, p.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_step_the_same_every_run(tmp_path):
    """--dump-outputs: config 2's result (x*y+1 of the seeded inputs) at seeded positions, float32 beside float64
    positions, and the same files from a second run with the same arguments."""
    import numpy as np
    import torch
    log2 = 22  # above the 2^21-element sample: the positions are drawn
    runs = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--log2-elems", str(log2),
                            "--no-ops", "--no-e2e", "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, cwd=ROOT, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout)["steps"] == 2
        runs.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    assert list(runs[0]) == ["zip_map_out.npy", "zip_map_out_index.npy"]
    for name, arr in runs[0].items():
        assert np.array_equal(arr.view(np.uint8), runs[1][name].view(np.uint8)), name
    got, pos = runs[0]["zip_map_out.npy"], runs[0]["zip_map_out_index.npy"]
    assert got.dtype == np.float32 and pos.dtype == np.float64 and got.shape == pos.shape
    assert 0 < got.size <= 1 << 21 and np.all(np.diff(pos) > 0) and pos[-1] < 1 << log2
    g = torch.Generator(device="cuda")
    g.manual_seed(0x5EED0001)  # bench.py's seed for rank 0
    ta = torch.empty(1 << log2, device="cuda", dtype=torch.float32).uniform_(-1, 1, generator=g)
    tb = torch.empty(1 << log2, device="cuda", dtype=torch.float32).uniform_(-1, 1, generator=g)
    at = torch.from_numpy(pos.astype(np.int64)).cuda()
    want = (ta[at] * tb[at] + 1.0).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
