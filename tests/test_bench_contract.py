"""bench.py's reference arm (the CPU port on the host cores) prints one JSON line with the contract's keys; the GPU arm has
no CPU fallback; --dump-outputs writes what the last timed step returned."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    # (a 256-scenario cut of the batch keeps the CPU suite short; the driver runs the whole 4096 x 64 every step)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--scenarios", "256"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "participant_steps_per_sec" and d["unit"] == "participant-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("C2 256x64") and d["config"]["scenarios_per_gpu"] == 256 and d["config"]["participants"] == 64


def test_gpu_arm_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from tactics2d_b200 import BatchedWorld, TypeTable

    with pytest.raises(RuntimeError, match="CUDA"):
        BatchedWorld(2, 2, TypeTable.vehicles())


def test_dump_outputs_writes_float_arrays_and_samples_one_row_set(tmp_path, monkeypatch):
    """bench.dump_outputs: every array as float32 (integers converted exactly); above the size limit one seeded set of
    scenario rows, the same in every array and in every run, recorded in scenario_index.npy."""
    import bench

    rng = np.random.default_rng(0)
    n, m = 300, 16
    arrays = {"x": rng.random((n, m), dtype=np.float32), "hit_index": rng.integers(-1, m, (n, m)).astype(np.int16),
              "done": rng.integers(0, 2, n).astype(np.uint8)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert np.array_equal(np.load(tmp_path / "all" / "scenario_index.npy"), np.arange(n))
    monkeypatch.setattr(bench, "DUMP_BYTES", (64 << 10) + 100 * ((2 * m + 1) * 4 + 8))   # room for 100 scenario rows
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    rows = np.load(tmp_path / "a" / "scenario_index.npy")
    assert rows.dtype == np.float64 and len(rows) == 100 and (np.diff(rows) > 0).all()
    assert np.array_equal(np.load(tmp_path / "b" / "scenario_index.npy"), rows)
    for k, a in arrays.items():
        got = np.load(tmp_path / "a" / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, a[rows.astype(np.int64)].astype(np.float32))
        assert np.array_equal(np.load(tmp_path / "b" / f"{k}.npy"), got)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(cuda_device, tmp_path):
    """--dump-outputs writes what the last timed step returned: with 2 replicas and 3 steps that is replica 0 after its
    second tick (steps 0 and 2), which a world built from the same seeds reproduces bit for bit."""
    import torch

    import bench
    from tactics2d_b200 import BatchedWorld, synthetic

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--scenarios", "64",
                        "--replicas", "2", "--min-reps", "2", "--min-seconds", "0", "--no-e2e", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    sc = bench.make_scene("c2", seed=1, n=64)
    w = BatchedWorld(*sc.shape, sc.table, device=cuda_device, max_step=0)
    w.set_map(sc.segments, sc.bounds)
    w.set_state(sc.x, sc.y, sc.heading, sc.speed, vx=sc.vx, vy=sc.vy, type_id=sc.type_id)
    act = torch.from_numpy(synthetic.random_actions(9000, sc.shape)).to(cuda_device)
    for _ in range(2):
        res = w.step(act)
    torch.cuda.synchronize()
    want = w.state_numpy()
    want.update({k: getattr(res, k).cpu().numpy() for k in ("flags", "hit_index", "hit_segment", "status", "done")})
    w.close()
    assert np.array_equal(np.load(tmp_path / "scenario_index.npy"), np.arange(64))
    for k, v in want.items():
        assert np.array_equal(np.load(tmp_path / f"{k}.npy"), v.astype(np.float32), equal_nan=True), k
    assert want["flags"].any()
