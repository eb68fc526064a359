"""bench.py contract checks: the reference arm's JSON line (the CPU port of the reference's path, a bounded sample
per step), the command-line surface the driver uses, and (on a GPU) the arrays --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT, env=e)


def test_reference_arm_prints_the_contract_line():
    out = _run("--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "stream-s/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("stream-seconds of 48 kHz stereo analysed/sec")
    assert line["value"] > 0 and line["steps"] == 1 and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "cpu" in cb and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "stream-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    out = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1",
               env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_product_arm_refuses_to_run_without_a_gpu():
    try:
        import torch
        if torch.cuda.is_available():
            return
    except Exception:
        pass
    out = _run("--steps", "1", "--no-cpu", "--no-e2e")
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def test_steps_must_be_positive():
    for impl in ("b200", "reference"):
        out = _run("--impl", impl, "--steps", "0")
        assert out.returncode != 0 and "--steps must be at least 1" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_step_computed(tmp_path):
    """3 stereo streams x 2 s = 6 x 187 rows, fewer than the sample size: the dump is every row, in order, and equals
    a separate analysis of the same seeded signal."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "audio-analyzer-omega_b200"))
    from omega4_b200.batch.driver import analyze_resident, device_synth
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    out = _run("--steps", "2", "--streams", "3", "--seconds", "2", "--no-cpu", "--no-e2e", "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["combined.npy", "meters.npy"]
    comb, met = np.load(tmp_path / "combined.npy"), np.load(tmp_path / "meters.npy")
    n_ch, n_hops = 6, 2 * 48000 // 512
    assert comb.dtype == met.dtype == np.float32 and comb.shape == (n_ch * n_hops, 512) and met.shape == (n_ch * n_hops, 5)
    plan = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
    x = device_synth(3, 2, n_hops * 512)
    want_c = torch.empty((n_ch, n_hops, 512), device="cuda")
    want_m = torch.empty((n_ch, n_hops, 5), device="cuda")
    analyze_resident(plan, x, combined=want_c, meters=want_m)
    torch.cuda.synchronize()
    assert np.array_equal(comb, want_c.reshape(-1, 512).cpu().numpy())
    assert np.array_equal(met, want_m.reshape(-1, 5).cpu().numpy())
    plan.close()


def test_numa_binding_helper_is_harmless_without_topology():
    sys.path.insert(0, ROOT)
    import bench
    before = os.sched_getaffinity(0)
    try:
        info = bench.bind_to_gpu_numa_node(0, 1)
        assert set(info) >= {"node", "cpus", "how"} and info["cpus"] >= 1
        assert bench._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    finally:
        os.sched_setaffinity(0, before)
