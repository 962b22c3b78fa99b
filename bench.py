#!/usr/bin/env python
"""bench.py -- ground-state pixels/s and env steps/s of the charge-stability hot path (BASELINE.json metric).

A "step" is one pass of the hot path over one batch of env.step calls: for every env, the N-1 adjacent-pair scan
windows (res x res pixels each) through ground-state solve -> latching -> sensor -> noise.  Workload at N GPUs:
BASELINE config 4 -- 8-dot latched array, 16384 envs PER GPU (weak scaling: envs shard by contiguous env id, no
collective on the step path), 64x64 scans, full sensor-noise model.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Prints ONE JSON line on rank 0.  `value` = pixels/s with descriptors and models resident in HBM; `e2e` = the same
through the host-buffer path (descriptors H2D from pinned memory + sensor images D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "rl-agent-for-qubit-array-tuning_b200")
for _p in (ROOT, PKG, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402


# ---------------------------------------------------------------------------------------------------------------
# Algorithmic work per pixel (DESIGN.md "Roofline").  SURVEY.md 8d counts the reference formulation (every candidate a
# full N^2 quadratic form); the kernel evaluates the same argmin through the factorisation
#   E(delta) = r.h + sum_j delta_j 2h_j + Q[delta],  Q precomputed per env,
# whose fp64 work is what the FP64 pipe actually has to do.  Both are reported.
# ---------------------------------------------------------------------------------------------------------------
def flops_reference_formulation(n: int) -> float:
    g, d = n + 1, n + 1
    return 2.0 * (n * g + (2 ** n) * n * (n + 1) + d * g + 11 * d * (d + 1)) + 60


def flops_factored(n: int) -> float:
    """fp64 operations of the factored search, FMA = 2 flop, add / compare = 1 flop, no relaxation."""
    nlo = min(n, 4)
    nhi = n - nlo
    pot = 2 * (2 * n) + 4                    # g = g0 + ix gx + iy gy, sensor potential
    lin = n + 2 * n * n + n                  # r = f - g, h = Cinv r, 2h
    llo = (1 << nlo) - 1
    search = (1 << nhi) * (nhi + 2 * (1 << nlo) + 2)
    sensor = 3 * n + 8 + 10 * 4
    return float(pot + lin + llo + search + sensor)


def fp64_pipe_ops_factored(n: int) -> float:
    """fp64-pipe instruction slots per pixel (FMA, add, compare each occupy one slot)."""
    nlo = min(n, 4)
    nhi = n - nlo
    return float(2 * n + 2 + n + n * n + n + ((1 << nlo) - 1) + (1 << nhi) * (nhi + 2 * (1 << nlo) + 2) + 2 * n + 8 + 20)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except OSError:
        return {"hbm_gbs": 6650.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the restated reference path on the host cores (oracle/), bounded sample of the same workload.
# ---------------------------------------------------------------------------------------------------------------
def _cpu_worker(job):
    mb_fields, rec, flags = job
    from util import oracle_batch
    from qdsim.engine import ModelBatch
    mb = ModelBatch(**mb_fields)
    oracle_batch(mb, rec, flags)
    return int(rec["nx"][0]) * int(rec["ny"][0]) * len(rec)


def cpu_reference_pixels_per_s(mb, scans, flags, n_sample_scans: int, cores: int, budget_s: float = 10.0):
    """Pixels/s of the CPU restatement (reference formulation) over a bounded sample of ``scans`` on ``cores`` threads.

    Preferred: the plain-C restatement with OpenMP (oracle/cport).  ``n_sample_scans == 0`` sizes the sample for about
    ``budget_s`` seconds from a short calibration run.  Fallback if gcc is missing: the NumPy oracle, one process/core.
    """
    import multiprocessing as mp
    try:
        from oracle import cport
        if cport.available():
            cal = min(len(scans), 4 * cores)
            cport.time_scans(mb, scans[:cal], flags, threads=cores)              # spin the thread pool up
            rate, cpix, cdt = cport.time_scans(mb, scans[:cal], flags, threads=cores)
            n = n_sample_scans or int(min(len(scans), max(cal, budget_s * rate / (cpix / cal))))
            pps, pixels, dt = cport.time_scans(mb, scans[:n], flags, threads=cores)
            return pps, pixels, dt, "port: plain-C restatement of the reference formulation, OpenMP over scans"
    except ImportError:
        pass
    n_sample_scans = n_sample_scans or max(2 * cores, 16)
    sample = scans[:n_sample_scans]
    envs = np.unique(sample["env_id"])
    remap = {int(e): i for i, e in enumerate(envs)}
    fields = dict(algorithm=mb.algorithm, n_gate=mb.n_gate, cdd_inv_gs=mb.cdd_inv_gs[envs], cdd_gs=mb.cdd_gs[envs],
                  cdd_inv_full=mb.cdd_inv_full[envs], cgd_full=mb.cgd_full[envs], params=mb.params[envs])
    sample = sample.copy()
    sample["env_id"] = [remap[int(e)] for e in sample["env_id"]]
    jobs = [(fields, sample[i:i + 1], flags) for i in range(len(sample))]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        pixels = sum(pool.map(_cpu_worker, jobs, chunksize=1))
    dt = time.perf_counter() - t0
    return pixels / dt, pixels, dt, "port: NumPy restatement, one process per core"


def cpu_reference_scan_seconds(mb, scans, flags, threads: int) -> float:
    """Wall time of ONE pass of the C restatement over ``scans`` on ``threads`` threads (latency of small cases; the
    first call spins the thread pool up and is discarded)."""
    from oracle import cport
    cport.run_scans(mb, scans, flags, threads=threads)
    return cport.run_scans(mb, scans, flags, threads=threads)[2]


def parity_sample(mb, scans, flags, z, n, pick, res: int, threads: int = 0):
    """CHECKER leg (the only use of oracle/ here besides the CPU baselines): re-run the scans ``pick`` of the timed batch
    with the plain-C restatement and compare -- charge maps bit for bit on rows without near-ties, images at 5e-6.
    ``z`` [pixels] / ``n`` [pixels, N]: this run's outputs (NumPy or CUDA tensors)."""
    from util import cport_parity
    pick = np.asarray(pick)
    pp = res * res
    if hasattr(z, "is_cuda"):
        import torch
        idx = torch.from_numpy(pick).to(z.device)
        zs = z.view(-1, pp)[idx].cpu().numpy().reshape(-1)
        ns = n.view(-1, pp, n.shape[-1])[idx].cpu().numpy().reshape(-1, n.shape[-1])
    else:
        zs = np.asarray(z).reshape(-1, pp)[pick].reshape(-1)
        ns = np.asarray(n).reshape(-1, pp, np.asarray(n).shape[-1])[pick].reshape(-1, np.asarray(n).shape[-1])
    sub = scans[pick].copy()
    sub["pix_offset"] = np.arange(len(sub), dtype=np.int64) * pp
    rep = cport_parity(mb, sub, flags, zs, ns, threads=threads or (os.cpu_count() or 1))
    rep["what"] = ("random scans of the timed batch re-run by the plain-C restatement (oracle/cport): n bit-exact on rows "
                   "whose best/second-best margin > 1e-9, z abs 5e-6")
    return rep


def source_sha() -> str:
    """sha256 over the kernel sources: keys the committed ncu figures (profiles/ncu_figures.json) to the code they were
    captured from, so a stale figure is reported as stale instead of silently reused."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(PKG, "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(open(os.path.join(csrc, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_figure(kernel: str):
    """Per-kernel figures taken from a committed ncu capture (profiles/ncu_figures.json, written by tools/ncu_figures.py
    from a .ncu-rep): warp instructions and DRAM bytes per pixel, with the source hash they belong to."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_figures.json")) as f:
            fig = json.load(f).get(kernel)
    except (OSError, ValueError):
        return None
    if fig is not None:
        fig = dict(fig)
        fig["stale"] = fig.get("source_sha") != source_sha()
    return fig


def build_workload(n_env: int, n_dot: int, res: int, rank: int, n_sets: int, path: str = "A"):
    from qdsim import synth
    if path == "B":
        dev = synth.sample_barrier_devices(n_env, n_dot, seed=1234 + rank)
        mb = synth.tunnel_batch(dev, latching=True, noise=True)
    else:
        dev = synth.sample_devices(n_env, n_dot, seed=1234 + rank)
        mb = synth.model_batch(dev, algorithm="default", thermal=False, latching=True, noise=True)
    sets = [synth.env_step_scans(mb, dev, res=res, seed=99 + rank, step=s) for s in range(n_sets)]
    return dev, mb, sets


def tunnel_cpu_baseline(mb, scans, budget_s: float = 8.0):
    """The tunnel path's reference formulation in plain C (all 4^N candidates as full quadratic forms, 32 x 32
    eigen-solve; oracle/cport/qd_cport_b.c, checked against the reference-made fixtures in tests/), OpenMP over the pixels
    of env 0's scan windows on every host core, about ``budget_s`` seconds."""
    from oracle import composer, cport
    from util import oracle_model, oracle_scan
    cores = os.cpu_count() or 1
    m = oracle_model(mb, 0, 0)
    grids = []
    for rec in scans[scans["env_id"] == 0]:              # every window of env 0 (N-1 scans)
        s0 = oracle_scan(rec, mb.n_volt, 0)
        grids.append(composer.affine_grid(s0.v0, s0.dx, s0.dy, s0.nx, s0.ny).reshape(-1, mb.n_volt))
    v = np.concatenate(grids)
    cal = v[: 8 * cores]
    _, _, dt = cport.tunnel_ground_state(m, cal, threads=cores)
    n_pix = int(min(len(v), max(len(cal), budget_s * len(cal) / max(dt, 1e-6))))
    _, _, dt = cport.tunnel_ground_state(m, v[:n_pix], threads=cores)
    return {"value": n_pix / dt, "unit": "pixels/s", "cores": cores, "kind": "port",
            "sample": f"{n_pix} pixels of one env's scan windows (ground state only), {dt:.1f} s",
            "what": "plain-C restatement of qarray_latched._ground_state_open in the reference's formulation, "
                    "OpenMP over pixels"}


def issue_roofline(kernels, pixels_per_s: float, sm_count: int, sm_mhz: float):
    """Issue-slot roofline of kernels with data-dependent control flow (no flop model): warp instructions per pixel from
    the committed ncu captures of THIS source (profiles/ncu_figures.json, keyed by source hash), summed over the kernels of
    the pipeline, against 4 issue slots per SM per clock at the measured SM clock."""
    if isinstance(kernels, str):
        kernels = [kernels]
    figs = {k: ncu_figure(k) for k in kernels}
    missing = [k for k, f in figs.items() if not f or not f.get("warp_instr_per_pixel")]
    name = " + ".join(kernels)
    if missing:
        return {"kernel": name, "bound": "issue", "achieved": None, "peak": None, "frac": None,
                "note": f"no ncu figure committed for {missing} (profiles/ncu_figures.json)"}
    instr = sum(f["warp_instr_per_pixel"] for f in figs.values())
    traffic = sum((f.get("dram_bytes_per_pixel") or 0.0) for f in figs.values())
    peak = sm_count * 4 * sm_mhz * 1e6
    ach = pixels_per_s * instr
    return {"kernel": name, "bound": "issue", "achieved": ach, "peak": peak, "unit": "warp-instr/s", "frac": ach / peak,
            "warp_instr_per_pixel": instr, "per_kernel": {k: {"warp_instr_per_pixel": f["warp_instr_per_pixel"],
                                                               "ncu_issue_active_pct": f.get("issue_active_pct"),
                                                               "registers": f.get("registers")} for k, f in figs.items()},
            "source": "ncu --set full captures listed in profiles/ncu_figures.json",
            "figure_source_sha": sorted({f.get("source_sha") for f in figs.values()}),
            "stale": any(f["stale"] for f in figs.values()), "traffic": traffic,
            "traffic_note": "DRAM bytes per pixel of the listed kernels (dram__bytes_read.sum + dram__bytes_write.sum)"}


def dump_outputs(out_dir: str, prefix: str, z, n, res: int, budget_bytes: int, seed: int):
    """Write what a timed launch returned, for output-for-output comparison of two builds: a fixed, seeded sample of
    whole scans as ``<prefix>z.npy`` (scans, res, res) float32 sensor images, ``<prefix>n.npy`` (scans, res, res, N)
    float32 charge occupations and ``<prefix>scan_index.npy`` (float64), the sampled scans' positions in the batch.
    The three files together stay within ``budget_bytes``."""
    import torch
    pp = res * res
    n_dot = n.shape[-1]
    n_scan = z.numel() // pp
    count = min(n_scan, (budget_bytes - 3 * 128) // (pp * 4 * (1 + n_dot) + 8))       # 128 B: one .npy header
    if count < 1:
        raise SystemExit(f"--dump-outputs: one {res}x{res} scan exceeds the {budget_bytes}-byte budget of '{prefix}'")
    pick = np.sort(np.random.default_rng(seed).choice(n_scan, size=count, replace=False))
    idx = torch.from_numpy(pick).to(z.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, prefix + "z.npy"), z.view(n_scan, res, res)[idx].float().cpu().numpy())
    np.save(os.path.join(out_dir, prefix + "n.npy"), n.view(n_scan, res, res, n_dot)[idx].float().cpu().numpy())
    np.save(os.path.join(out_dir, prefix + "scan_index.npy"), pick.astype(np.float64))


# --dump-outputs budgets (bytes): the headline launch and the tunnel-path block, under 64 MB in all
DUMP_BYTES_MAIN, DUMP_BYTES_TUNNEL = 45_900_000, 17_900_000


def tunnel_kernels(n_dot: int):
    # (the fix-up passes of the block-walk select kernel and of the Householder eigen kernel over the pixels the
    # enumeration / Noda kernels gave up on, < 0.5 % of them, are not counted)
    sel = "qd_tunnel_select2_kernel" if n_dot >= 4 else "qd_tunnel_select_kernel"
    return [f"{sel}<{n_dot}>", f"qd_tunnel_eigen2_kernel<{n_dot}>"]


def tunnel_path_block(eng, n_dot: int, res: int, flags: int, with_cpu: bool, n_env: int = 512, steps: int = 5,
                      warmup: int = 5, sm_mhz: float = 1965.0, dump_dir: str | None = None):
    """Path B on the same GPU (what env.step runs in barrier mode): device-resident timing (CUDA events, warmed) AND the
    end-to-end host-buffer call, the issue-slot roofline from the committed ncu figure, and the C restatement of the
    reference's formulation on the host cores.  ``dump_dir``: write a sample of the last timed launch's outputs there."""
    import torch
    from qdsim import N_F32, N_NONE
    dev, mb, sets = build_workload(n_env, n_dot, res, 0, 1, "B")
    eng.set_models(mb)
    scans = sets[0]
    pixels = len(scans) * res * res
    st = torch.cuda.current_stream()
    z = torch.empty(pixels, dtype=torch.float32, device="cuda")
    n = torch.empty((pixels, n_dot), dtype=torch.float32, device="cuda")
    eng.scan_upload(scans, st)
    for _ in range(warmup):
        eng.scan_launch(z, n, N_F32, flags, st)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = eng.launch_count
    e0.record(st)
    for _ in range(steps):
        eng.scan_launch(z, n, N_F32, flags, st)
    e1.record(st)
    torch.cuda.synchronize()
    launches = eng.launch_count - l0
    ms = e0.elapsed_time(e1) / steps
    if dump_dir:
        dump_outputs(dump_dir, "tunnel_", z, n, res, DUMP_BYTES_TUNNEL, seed=2027)
    z_host = torch.empty(pixels, dtype=torch.float32).pin_memory().numpy()
    pin = torch.empty(scans.nbytes, dtype=torch.uint8).pin_memory()
    pin.numpy()[:] = scans.view(np.uint8)
    sp = pin.numpy().view(scans.dtype)
    for _ in range(2):
        eng.scan_open_host(sp, n_type=N_NONE, flags=flags, z_out=z_host)
    t0 = time.perf_counter()
    for _ in range(steps):
        eng.scan_open_host(sp, n_type=N_NONE, flags=flags, z_out=z_host)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / steps
    props = torch.cuda.get_device_properties(0)
    blk = {"workload": f"{n_dot}-dot tunnel-coupled array (TunnelCoupledChargeSensed, 32-state basis, barrier voltages), "
                       f"{n_env} envs, {n_dot - 1} scans/env of {res}x{res}, latching + noise",
           "kernels": f"qd_tunnel_relax_kernel<{n_dot}> + qd_tunnel_select2_kernel<{n_dot}> + qd_tunnel_eigen2_kernel<{n_dot}> "
                      f"(+ qd_tunnel_select_kernel / qd_tunnel_eigen_kernel<{n_dot}> as fix-up passes) "
                      f"+ qd_scan_kernel<{n_dot},tunnel>",
           "value": pixels / (ms * 1e-3), "unit": "pixels/s", "env_steps_per_s": n_env / (ms * 1e-3),
           "ms_per_step": ms, "steps": steps, "warmup": warmup, "gpu_launches": int(launches),
           "e2e": {"value": pixels / (e2e_ms * 1e-3), "unit": "pixels/s", "env_steps_per_s": n_env / (e2e_ms * 1e-3),
                   "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(scans.nbytes), "d2h_bytes_per_step": int(pixels * 4)},
           "roofline": issue_roofline(tunnel_kernels(n_dot), pixels / (ms * 1e-3), props.multi_processor_count, sm_mhz),
           "cpu_baseline": None}
    if with_cpu:
        blk["cpu_baseline"] = tunnel_cpu_baseline(mb, scans)
    return blk


_REAL_STDOUT = None


def _claim_stdout():
    """Everything any library prints to fd 1 during the run (NCCL prints its version line there) goes to stderr; the ONE
    JSON line is written to the real stdout by ``_emit``."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    sys.stdout.flush()
    line = (json.dumps(obj) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-env", type=int, default=16384, help="envs per GPU")
    ap.add_argument("--n-dot", type=int, default=8)
    ap.add_argument("--res", type=int, default=64)
    ap.add_argument("--cpu-scans", type=int, default=0, help="scans in the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-path-b", action="store_true", help="skip the secondary tunnel-coupled measurement")
    ap.add_argument("--no-compact", action="store_true", help="skip the compact-format (uint8 / half) end-to-end runs")
    ap.add_argument("--parity-scans", type=int, default=2048,
                    help="scans of the timed batch re-run by the C restatement and compared (0 = skip)")
    ap.add_argument("--path", default="A", choices=["A", "B"],
                    help="A: constant-interaction ChargeSensedDotArray path (headline); B: tunnel-coupled path of "
                         "env.step in barrier mode (secondary; use e.g. --n-dot 4 --n-env 1024)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed, seeded sample of the last timed step's sensor images and charge occupations "
                         "(and of the tunnel-path block's) to DIR as .npy files, 64 MB at most")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from qdsim import FLAG_LATCH, FLAG_NOISE, FLAG_RADIAL, N_NONE, N_U8
    flags = FLAG_LATCH | FLAG_NOISE | FLAG_RADIAL
    N, res = args.n_dot, args.res
    pix_per_env = (N - 1) * res * res
    workload = (f"{N}-dot latched array, {args.n_env} envs/GPU, {N - 1} scans/env of {res}x{res}, default algorithm, "
                f"T=0, latching + white/telegraph/radial noise")
    if args.path == "B":
        workload = (f"{N}-dot tunnel-coupled array (32-state basis, barrier voltages), {args.n_env} envs/GPU, {N - 1} "
                    f"scans/env of {res}x{res}, latching + white/telegraph/radial noise")
    config = {"workload": workload, "n_dot": N, "n_env_per_gpu": args.n_env, "res": res,
              "scans_per_env": N - 1, "l2": "inputs+outputs per step >> L2 (outputs alone 12 B/pixel)",
              "value_inputs": "model records and scan descriptors resident in HBM when the timed region starts; "
                              "e2e includes the per-step descriptor H2D and the image D2H"}

    # ---------------------------------------------------------------- reference arm: CPU only, rank 0 only
    if args.impl == "reference":
        if rank != 0:
            return
        cores = os.cpu_count() or 1
        dev, mb, sets = build_workload(min(args.n_env, 512), N, res, 0, 1)
        n_scans = args.cpu_scans
        if not n_scans:                       # ~3 s of CPU work per step
            _, cpix, cdt, _ = cpu_reference_pixels_per_s(mb, sets[0], flags, 4 * cores, cores)
            n_scans = int(min(len(sets[0]), max(4 * cores, 3.0 * (cpix / cdt) / (res * res))))
        per_step = []
        kind = ""
        for _ in range(args.warmup + args.steps):
            pps, pixels, dt, kind = cpu_reference_pixels_per_s(mb, sets[0], flags, n_scans, cores)
            per_step.append((pixels, dt))
        timed = per_step[args.warmup:]
        pixels = sum(p for p, _ in timed)
        dt = sum(t for _, t in timed)
        value = pixels / dt
        sample = f"{n_scans} scans ({timed[0][0]} pixels) of the workload per step"
        _emit(({
            "impl": "reference", "metric": "ground_state_pixels_per_s", "value": value, "unit": "pixels/s",
            "env_steps_per_s": value / pix_per_env, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / max(1, len(timed)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": "pixels/s", "cores": cores, "kind": "port", "sample": sample,
                             "what": kind},
            "e2e": {"value": value, "unit": "pixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist
    from qdsim import Engine

    torch.cuda.set_device(local_rank)
    numa_bound = False
    if world > 1 and os.environ.get("QDSIM_NO_NUMA_BIND") != "1":
        from qdsim import parallel as _par
        numa_bound = _par.bind_to_gpu_numa_node(local_rank)      # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = Engine(local_rank)
    n_sets = 2
    dev, mb, sets = build_workload(args.n_env, N, res, rank, n_sets, args.path)
    eng.set_models(mb)
    n_scan = len(sets[0])
    pixels = n_scan * res * res
    stream = torch.cuda.current_stream()
    z_dev = torch.empty(pixels, dtype=torch.float32, device="cuda")
    n_dev = torch.empty((pixels, N), dtype=torch.uint8, device="cuda")
    if args.path == "B":
        n_dev = torch.empty((pixels, N), dtype=torch.float32, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) device-resident timing: `value` and the kernel's roofline ----
    eng.scan_upload(sets[0], stream)
    N_OUT = N_U8
    if args.path == "B":
        from qdsim import N_F32
        N_OUT = N_F32
    for _ in range(warmup):
        eng.scan_launch(z_dev, n_dev, N_OUT, flags, stream)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record(stream)
    for k in range(args.steps):
        eng.scan_launch(z_dev, n_dev, N_OUT, flags, stream)
        ev[k + 1].record(stream)
    barrier()
    launches = eng.launch_count - launches0
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_ms = max_over_ranks(ev[0].elapsed_time(ev[-1]))
    ms_per_step = total_ms / args.steps
    value = world * pixels / (ms_per_step * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, "", z_dev, n_dev, res, DUMP_BYTES_MAIN, seed=2026)

    # ---- parity on the timed batch itself (outside every timed region; rank 0) ----
    parity = None
    if rank == 0 and args.path == "A" and args.parity_scans > 0:
        rng = np.random.default_rng(2026)
        pick = np.sort(rng.choice(n_scan, size=min(args.parity_scans, n_scan), replace=False))
        parity = parity_sample(mb, sets[0], flags, z_dev, n_dev, pick, res)

    # ---- (2) end to end through the host-buffer path ----
    pinned_scans = [torch.empty(s.nbytes, dtype=torch.uint8).pin_memory() for s in sets]
    for t, s in zip(pinned_scans, sets):
        t.numpy()[:] = s.view(np.uint8)
    z_host = torch.empty(pixels, dtype=torch.float32).pin_memory()
    z_host_np = z_host.numpy()
    obs_u8 = torch.empty(pixels, dtype=torch.uint8).pin_memory().numpy()
    obs_f16 = torch.empty(pixels, dtype=torch.float16).pin_memory().numpy()
    from qdsim import Z_F16, Z_U8

    def e2e_step(k):
        # the reference-facing host-buffer call: descriptors H2D from pinned memory, compute, sensor images D2H into
        # pinned memory, all inside qd_scan_open_host (chunked: compute overlaps the copy-back)
        s = pinned_scans[k % n_sets].numpy().view(sets[0].dtype)
        eng.scan_open_host(s, n_type=N_NONE, flags=flags, z_out=z_host_np)

    def e2e_obs_u8(k):
        # compact observation: percentile-normalised per env on the device, uint8, one quarter of the bytes
        s = pinned_scans[k % n_sets].numpy().view(sets[0].dtype)
        eng.scan_obs_host(s, z_type=Z_U8, flags=flags, normalise=True, out=obs_u8)

    def e2e_obs_f16(k):
        s = pinned_scans[k % n_sets].numpy().view(sets[0].dtype)
        eng.scan_obs_host(s, z_type=Z_F16, flags=flags, normalise=False, out=obs_f16)

    def time_e2e(fn):
        for k in range(2):
            fn(k)
        barrier()
        # the call is synchronous (returns with the images in host memory), so the host clock brackets exactly the device
        # work + copies; barrier + synchronize on both sides, max over ranks
        t0 = time.perf_counter()
        for k in range(args.steps):
            fn(k)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        barrier()
        per_rank = [wall / args.steps]
        if world > 1:
            t = torch.tensor([wall / args.steps], dtype=torch.float64, device="cuda")
            allr = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allr, t)
            per_rank = [float(x.item()) for x in allr]
        return max(per_rank), per_rank

    e2e_ms, e2e_ranks = time_e2e(e2e_step)
    # the measured host ceiling of this copy (profiles/r02_d2h_ceiling.json: every rank of one box copying at once)
    ceiling = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_d2h_ceiling.json")) as f:
            c = json.load(f)["by_ranks"].get(str(world))
        if c:
            ms_c = pixels * 4 / (min(c["d2h_per_rank_gbs"]) * 1e9) * 1e3
            ceiling = {"d2h_gbs_slowest_rank": min(c["d2h_per_rank_gbs"]), "ms_per_step_copy_only": ms_c,
                       "frac_of_ceiling": ms_c / e2e_ms,
                       "source": "profiles/r02_d2h_ceiling.json (tools/pcie_bw.py, all ranks copying concurrently)"}
    except (OSError, ValueError, KeyError):
        pass
    clocks = sampler.stop() if rank == 0 else None          # sampled across the device-resident and the fp32 e2e regions
    e2e_value = world * pixels / (e2e_ms * 1e-3)
    compact = {}
    if args.path == "A" and not args.no_compact:
        for name, fn, bpp, what in (("obs_u8", e2e_obs_u8, 1, "per-env percentile-normalised observation, uint8 (what the policy is fed, env.py:471-509)"),
                                    ("raw_f16", e2e_obs_f16, 2, "raw sensor signal, IEEE half")):
            ms_c, ranks_c = time_e2e(fn)
            compact[name] = {"value": world * pixels / (ms_c * 1e-3), "unit": "pixels/s", "ms_per_step": ms_c,
                             "per_rank_ms": ranks_c, "d2h_bytes_per_step": int(pixels * bpp),
                             "h2d_bytes_per_step": int(sets[0].nbytes), "format": what}
    # the host-buffer path returns the very images of the device-resident launch (same descriptors -> same pixels)
    e2e_step(0)
    e2e_same = bool(torch.equal(z_host.cuda(), z_dev)) if args.path == "A" else None

    # ---- (3) roofline of the dominant kernel (rank 0) ----
    out = None
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        fp64_peak = eng.fp64_peak_tflops(8192)
        fp32_peak = eng.fp32_peak_tflops(8192)
        k_ms = sum(kernel_ms) / len(kernel_ms)
        pix_s_kernel = pixels / (k_ms * 1e-3)
        f_exec, f_ref = flops_factored(N), flops_reference_formulation(N)
        achieved = pix_s_kernel * f_exec * 1e-12
        bytes_per_pixel = 4 + N
        hbm_achieved = pix_s_kernel * bytes_per_pixel * 1e-9
        kname = f"qd_scan_kernel<{N},default>"
        fig = ncu_figure(kname)
        sm_mhz = float((clocks or {}).get("sm_mhz") or 1965.0)
        sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
        roofline = {
            "bound": "fp64_pipe", "kernel": kname,
            "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
            # two numerators, both against the measured FP64 FMA peak: the factored search the kernel has to execute, and
            # SURVEY 8(d)'s count of the REFERENCE formulation (every candidate a full quadratic form).  The second exceeds
            # 1: the kernel does not do that work -- exact dominance pruning + Gray-code walk reach the same argmin.
            "frac_factored": achieved / fp64_peak,
            "frac_survey_formulation": pix_s_kernel * f_ref * 1e-12 / fp64_peak,
            "peak_kind": "fp64 FMA micro-benchmark run inside this bench (qd_measure_fp64_peak); "
                         "MEASURED_PEAKS.json has no CUDA-core figure",
            "flop_per_pixel": f_exec, "flop_per_pixel_reference_formulation": f_ref,
            "binding": "instruction issue (see `issue`): a per-pixel 8 x 8 fp64 quadratic form with data-dependent control "
                       "flow -- no tensor-core shape, HBM at a few percent",
            "issue": issue_roofline(kname, pix_s_kernel, sm_count, sm_mhz),
            "pipe_slot_frac": pix_s_kernel * fp64_pipe_ops_factored(N) * 2e-12 / fp64_peak,
            "kernel_ms": k_ms, "fp32_peak": fp32_peak,
            # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu capture of THIS source
            # (profiles/ncu_figures.json; `traffic_stale` says when the kernel sources changed since)
            "traffic": (fig["dram_bytes_per_pixel"] * pixels) if fig and fig.get("dram_bytes_per_pixel") else None,
            "traffic_stale": fig["stale"] if fig else None,
            "traffic_source": (fig or {}).get("source"),
            "hbm": {"achieved": hbm_achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": hbm_achieved / peaks["hbm_gbs"], "peak_kind": peak_kind,
                    "algorithmic_bytes_per_pixel": bytes_per_pixel},
        }
        cpu = None
        if args.path == "B":
            roofline = issue_roofline(tunnel_kernels(N), pix_s_kernel, sm_count, sm_mhz)
            roofline["kernel_ms"] = k_ms
            if world == 1 and not args.no_cpu_baseline:
                cpu = tunnel_cpu_baseline(mb, sets[0])
        if world == 1 and not args.no_cpu_baseline and args.path == "A":
            cores = os.cpu_count() or 1
            pps, cpix, cdt, kind = cpu_reference_pixels_per_s(mb, sets[0], flags, args.cpu_scans, cores)
            cpu = {"value": pps, "unit": "pixels/s", "cores": cores, "kind": "port",
                   "sample": f"{cpix // (res * res)} scans ({cpix} pixels) of the same workload, {cdt:.1f} s",
                   "what": kind}
            # BASELINE.md section 3 variant 1, once: the literal NumPy restatement -- vectorised over the pixels of a scan,
            # host Python loops for latching and telegraph noise exactly where the reference has them -- single process
            from util import oracle_batch
            n_lit = 6
            t0 = time.perf_counter()
            oracle_batch(mb, sets[0][:n_lit], flags)
            dt_lit = time.perf_counter() - t0
            cpu["variants"] = {"literal_numpy_single_process": {
                "value": n_lit * res * res / dt_lit, "unit": "pixels/s", "cores": 1,
                "sample": f"{n_lit} scans, {dt_lit:.1f} s",
                "what": "oracle/scan.py: NumPy fp64 over the pixels of a scan, Python loops along the latching / telegraph "
                        "chains (how the reference's host code is written)"}}
        out = {
            "metric": "ground_state_pixels_per_s", "value": value, "unit": "pixels/s",
            "env_steps_per_s": value / pix_per_env,
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "pixels/s", "env_steps_per_s": e2e_value / pix_per_env,
                    "ms_per_step": e2e_ms, "per_rank_ms": e2e_ranks, "format": "fp32 sensor images (the parity format)",
                    "h2d_bytes_per_step": int(sets[0].nbytes), "d2h_bytes_per_step": int(pixels * 4),
                    "matches_device_resident_launch": e2e_same, "host_d2h_ceiling": ceiling},
            "e2e_compact": compact or None,
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "parity_sample": parity,
            "parity_note": "latching / noise semantics are the restatement's (qarray wheel absent: parity unpinned there, "
                           "DESIGN.md section 2); the check above pins the CUDA path to that restatement on the benched batch",
            "source_sha": source_sha(),
        }
    # ---- (4) secondary: the tunnel-coupled path that QADAPT's env.step executes in barrier mode (Path B) ----
    if rank == 0 and world == 1 and args.path == "A" and not args.no_path_b:
        out["env_step_tunnel_path"] = tunnel_path_block(eng, N, res, flags, not args.no_cpu_baseline, steps=args.steps,
                                                        sm_mhz=float((clocks or {}).get("sm_mhz") or 1965.0),
                                                        dump_dir=args.dump_outputs)
    # the one collective of the design, OFF the step path: per-env episode statistics to every rank (NCCL all-gather)
    if world > 1:
        from qdsim import parallel
        stats = torch.stack([z_dev.view(args.n_env, -1).mean(dim=1),
                             torch.full((args.n_env,), float(rank), device="cuda")], dim=1)
        full = parallel.gather_episode_stats(stats, args.n_env * world)
        assert full.shape == (args.n_env * world, 2)
        if rank == 0:
            out["episode_stats_allgather"] = {"shape": list(full.shape), "ranks_seen": int(full[:, 1].unique().numel())}
            out["numa_bound"] = bool(numa_bound)
    barrier()
    if world > 1:
        dist.destroy_process_group()
    if rank == 0:
        _emit(out)


if __name__ == "__main__":
    main()
