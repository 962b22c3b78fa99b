"""Throughput of the closed-array path (qd_scan_closed) next to the open path on the same batch and the C restatement.

One JSON line per case: 2 / 4 / 6 / 8 dots, 64 x 64 scans (one per env), 1024 and 4096 envs, ``default`` and
``brute_force``, total charge N // 2 + 2 on every scan, latching + white / telegraph noise on.  For each case the Mpixel/s of
  * ``closed``: qd_scan_closed into device buffers (CUDA events around the launches, after a warm-up launch);
  * ``open``: qd_scan_open of the same batch through the same generic kernel (QDSIM_GENERIC_SCAN=1);
  * ``cport``: the plain-C restatement's closed scans (OpenMP, all cores) on the first few scans of the batch.
Every line carries the card's name and power limit, read in the same run.

    python tools/closed_bench.py [--reps 3] [--cport-scans 4]
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

import numpy as np  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def batch(n_dot, n_env, algorithm, res=64):
    from qdsim import synth
    dev = synth.sample_devices(n_env, n_dot, seed=17 + n_dot)
    mb = synth.model_batch(dev, algorithm=algorithm, latching=True, noise=True, max_charge_carriers=4)
    scans = synth.env_step_scans(mb, dev, res=res, seed=5, offset_range=2.0, radial=False)[:: n_dot - 1].copy()
    scans["pix_offset"] = np.arange(len(scans), dtype=np.int64) * res * res
    return mb, scans


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
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cport-scans", type=int, default=4)
    args = ap.parse_args()
    import torch
    from oracle.cport import closed as cport
    from qdsim import FLAG_LATCH, FLAG_NOISE, N_U8, Engine
    name, power = card()
    eng = Engine(0)
    flags = FLAG_LATCH | FLAG_NOISE
    for algorithm in ("default", "brute_force"):
        for n_dot in (2, 4, 6, 8):
            for n_env in (1024, 4096):
                mb, scans = batch(n_dot, n_env, algorithm)
                q = n_dot // 2 + 2
                pixels = len(scans) * 64 * 64
                eng.set_models(mb)
                z = torch.empty(pixels, dtype=torch.float32, device="cuda")
                n = torch.empty((pixels, n_dot), dtype=torch.uint8, device="cuda")
                closed = rate(lambda: eng.scan_closed(scans, q, z, n, N_U8, flags), pixels, args.reps)
                os.environ["QDSIM_GENERIC_SCAN"] = "1"
                try:
                    opened = rate(lambda: eng.scan_open(scans, z, n, N_U8, flags), pixels, args.reps)
                finally:
                    del os.environ["QDSIM_GENERIC_SCAN"]
                sub = scans[: args.cport_scans].copy()
                _, _, dt = cport.run_scans_closed(mb, sub, q, flags, want_n=False)
                print(json.dumps({
                    "case": f"{algorithm}_{n_dot}dot_{n_env}env", "algorithm": algorithm, "n_dot": n_dot, "n_env": n_env,
                    "scan": "64x64", "n_charge": q, "flags": "latch+noise",
                    "closed_mpix_s": round(closed, 2), "open_generic_mpix_s": round(opened, 2),
                    "cport_closed_mpix_s": round(len(sub) * 64 * 64 / dt / 1e6, 4), "cport_threads": os.cpu_count(),
                    "gpu": name, "power_limit": power}), flush=True)
    eng.close()


if __name__ == "__main__":
    main()
