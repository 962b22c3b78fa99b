"""What more charge sensors cost: the scan rate of one batch at 1, 2 and 4 sensors.

One JSON line per case, each with the card's name and power limit read in the same run:
  * Path A, 8 dots, 64 x 64 scans of one env.step (7 per env), 4096 envs, latching + white / telegraph + radial noise:
    S = 1 on the fast kernel and on the generic kernel (QDSIM_GENERIC_SCAN=1), S = 2 and S = 4 (the QD_MSENSOR instances);
  * the tunnel path, 4 dots with barriers, 64 x 64, 256 envs, latching + noise: S = 1 and S = 2.
Rates are Mpixel/s of qd_scan_open into device buffers, CUDA events around ``--reps`` launches after a warm-up launch.
Sensors 1.. of the multi-sensor devices are synth.sample_devices's extra sensors; sensor 0 and the dots are the
one-sensor device's.

    python tools/multisensor_bench.py [--reps 5] [--envs 4096] [--tunnel-envs 256]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "rl-agent-for-qubit-array-tuning_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def rate(fn, pixels, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return pixels * reps / (e0.elapsed_time(e1) * 1e-3) / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--tunnel-envs", type=int, default=256)
    args = ap.parse_args()
    import torch
    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_F64, N_U8, Engine, synth
    name, power = card()
    eng = Engine(0)

    def run(case, mb, scans, flags, n_type, generic=False, **extra):
        eng.set_models(mb)
        pixels = int(scans["nx"][0]) * int(scans["ny"][0]) * len(scans)
        z = torch.empty((pixels, mb.n_sensor), dtype=torch.float32, device="cuda")
        n = torch.empty((pixels, mb.n_dot), dtype=torch.uint8 if n_type == N_U8 else torch.float64, device="cuda")
        if generic:
            os.environ["QDSIM_GENERIC_SCAN"] = "1"
        try:
            launches0 = eng.launch_count
            r = rate(lambda: eng.scan_open(scans, z, n, n_type, flags), pixels, args.reps)
            per_call = (eng.launch_count - launches0) // (args.reps + 1)
        finally:
            os.environ.pop("QDSIM_GENERIC_SCAN", None)
        del z, n
        torch.cuda.empty_cache()
        print(json.dumps({"case": case, "n_dot": mb.n_dot, "n_sensor": mb.n_sensor, "scans": len(scans), "scan": "64x64",
                          "mpix_s": round(r, 2), "launches_per_call": per_call, **extra, "gpu": name,
                          "power_limit": power}), flush=True)

    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    for s in (1, 2, 4):
        dev = synth.sample_devices(args.envs, 8, seed=2024, n_sensor=s)
        mb = synth.model_batch(dev, latching=True, noise=True)
        scans = synth.env_step_scans(mb, dev, res=64, seed=7)
        if s == 1:
            run("pathA_8dot_S1_fast", mb, scans, flags, N_U8, kernel="qd_scan_fast_kernel")
            run("pathA_8dot_S1_generic", mb, scans, flags, N_U8, generic=True, kernel="qd_scan_kernel")
        else:
            run(f"pathA_8dot_S{s}", mb, scans, flags, N_U8, kernel="qd_scan_kernel QD_MSENSOR")
    for s in (1, 2):
        dev = synth.sample_barrier_devices(args.tunnel_envs, 4, seed=2025, n_sensor=s)
        mb = synth.tunnel_batch(dev)
        scans = synth.env_step_scans(mb, dev, res=64, seed=8, radial=False)
        run(f"tunnel_4dot_S{s}", mb, scans, FLAG_LATCH | FLAG_NOISE, N_F64)
    eng.close()


if __name__ == "__main__":
    main()
