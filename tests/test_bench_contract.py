"""bench.py's reference arm and JSON contract, on the CPU with a tiny workload; its output dump on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--n-env", "4", "--n-dot", "4", "--res", "16", "--cpu-scans", "6"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ground_state_pixels_per_s" and d["unit"] == "pixels/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_flop_models_match_the_survey_figures():
    sys.path.insert(0, ROOT)
    import bench
    assert [bench.flops_reference_formulation(n) for n in (2, 4, 6, 8)] == [402.0, 1450.0, 6850.0, 39210.0]
    assert bench.flops_factored(8) < bench.flops_reference_formulation(8) / 30


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(engine, tmp_path):
    """--dump-outputs writes float .npy files within 64 MB, equal to what the same launches compute here for the same
    seeded workloads; --steps sets the number of timed launches of both blocks."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_F32, N_U8
    steps, flags = 3, FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                          "--n-env", "64", "--n-dot", "4", "--res", "16", "--no-cpu-baseline", "--parity-scans", "0",
                          "--no-compact", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    names = {p + f for p in ("", "tunnel_") for f in ("z.npy", "n.npy", "scan_index.npy")}
    assert {f.name for f in tmp_path.iterdir()} == names
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64_000_000
    got = {f: np.load(tmp_path / f) for f in names}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())

    def run(mb, scans, n_type, n_dtype):
        """Host-buffer outputs of ``scans`` and the kernel launches of one device-resident step over them."""
        engine.set_models(mb)
        z, n = engine.scan_open_host(scans, n_type=n_type, flags=flags)
        st = torch.cuda.current_stream()
        zd = torch.empty(z.size, dtype=torch.float32, device="cuda")
        nd = torch.empty(n.shape, dtype=n_dtype, device="cuda")
        engine.scan_upload(scans, st)
        l0 = engine.launch_count
        engine.scan_launch(zd, nd, n_type, flags, st)
        torch.cuda.synchronize()
        return z.reshape(-1, 16, 16), n.reshape(-1, 16, 16, 4).astype(np.float32), engine.launch_count - l0

    _, mb, sets = bench.build_workload(64, 4, 16, 0, 1)
    z, n, per_step = run(mb, sets[0], N_U8, torch.uint8)
    assert d["gpu_launches"] == steps * per_step
    assert np.array_equal(got["scan_index.npy"], np.arange(len(sets[0])))       # the whole batch fits the budget
    assert np.array_equal(got["z.npy"], z) and np.array_equal(got["n.npy"], n)
    _, mb, sets = bench.build_workload(512, 4, 16, 0, 1, "B")                   # the tunnel-path block's workload
    z, n, per_step = run(mb, sets[0], N_F32, torch.float32)
    assert d["env_step_tunnel_path"]["gpu_launches"] == steps * per_step
    pick = got["tunnel_scan_index.npy"].astype(np.int64)
    assert len(pick) > 0 and np.array_equal(pick, np.unique(pick)) and pick[-1] < len(sets[0])
    np.testing.assert_allclose(got["tunnel_z.npy"], z[pick], rtol=0, atol=1e-5)
    np.testing.assert_allclose(got["tunnel_n.npy"], n[pick], rtol=0, atol=1e-5)


def test_tunnel_cpu_baseline_block():
    """The CPU comparator of bench.py's tunnel-path block runs on its own (no GPU) and reports the contract's keys."""
    import bench
    from qdsim import synth
    dev = synth.sample_barrier_devices(2, 4, seed=3)
    mb = synth.tunnel_batch(dev)
    scans = synth.env_step_scans(mb, dev, res=8, seed=4)
    out = bench.tunnel_cpu_baseline(mb, scans, budget_s=0.2)
    assert out["kind"] == "port" and out["unit"] == "pixels/s" and out["value"] > 0 and out["cores"] >= 1
