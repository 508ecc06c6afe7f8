"""bench.py's contract: the reference arm prints ONE JSON line with the keys a caller reads, the GPU
arm refuses to run without a GPU (no CPU fallback), and ``--dump-outputs`` writes the state the
timed steps leave."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, env=e, timeout=600)


def test_reference_arm_prints_one_json_line():
    # bounded: 1 step, 1 warm-up (the arm extends itself to ~10 s of CPU work)
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GDoF/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "GDoF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "demo_linear_box" in d["config"]["workload"]


def test_reference_arm_only_rank0_works_under_torchrun():
    r = _run("--impl", "reference", "--steps", "1", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    r = _run("--steps", "1")
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_dump_outputs_write_a_fixed_sample_within_64_mb_over_all_ranks(tmp_path):
    import torch

    import bench

    n = 3_000_000
    u = torch.arange(n + 7, dtype=torch.float64)  # entries hold their own index; 7 trailing ghosts
    v = torch.arange(n + 7, dtype=torch.float32)  # exact below 2^24
    for world in (1, 2, 8):
        d = tmp_path / f"world{world}"
        for rank in range(world):
            idx = bench.dump_indices(n, 8, 2, rank, world)
            assert np.array_equal(idx, bench.dump_indices(n, 8, 2, rank, world))
            bench.dump_outputs(str(d), {"u": u[torch.from_numpy(idx)], "v": v[torch.from_numpy(idx)]}, rank, world)
        files = sorted(os.listdir(d))
        assert files == (["u.npy", "v.npy"] if world == 1 else
                         sorted(f"{k}_rank{r}.npy" for k in "uv" for r in range(world)))
        assert sum(os.path.getsize(d / f) for f in files) <= 64 * 10**6
        for f in files:
            if f.startswith("u"):
                du, dv = np.load(d / f), np.load(d / ("v" + f[1:]))
                assert du.dtype == np.float64 and dv.dtype == np.float32
                assert np.array_equal(dv, du.astype(np.float32))  # u and v at the same indices
                assert np.all(np.diff(du) > 0) and 0 <= du[0] and du[-1] < n  # distinct, in order, owned
                assert du[0] < n // du.size and du[-1] >= n - n // du.size - 1  # spread over all n
    assert np.array_equal(bench.dump_indices(1000, 8, 2, 1, 2), np.arange(1000))


@pytest.mark.gpu
def test_dump_outputs_hold_the_state_after_the_timed_steps(tmp_path):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = {}
    for steps, warmup in ((2, 3), (1, 4), (3, 3)):
        d = tmp_path / f"s{steps}w{warmup}"
        r = _run("--n-per-gpu", "6", "--no-cpu", "--no-extras", "--steps", str(steps), "--warmup", str(warmup),
                 "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["warmup"] == warmup
        out[steps, warmup] = [np.load(d / f"{k}.npy") for k in ("u", "v")]
    rel = lambda a, b: np.linalg.norm(a - b) / np.linalg.norm(b)  # noqa: E731
    for x, y, z in zip(out[2, 3], out[1, 4], out[3, 3]):
        assert x.dtype == np.float64 and np.linalg.norm(x) > 0
        assert rel(x, y) < 1e-12  # 3 + 2 steps == 4 + 1 steps
        assert rel(x, z) > 1e-3  # one timed step more
