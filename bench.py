#!/usr/bin/env python
"""Benchmark of the DESMO fused train step (BASELINE.json metric: train iters/s + HBM GB/s of the fused residual+grad pass).

  python bench.py --gpus N --steps K --warmup W            # this framework, N GPUs of one node (torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle/torch_port.py) on the host cores

Default workload (config.workload): "aneurysm-scale" -- n = 3 * 2^20 mesh points per GPU x m = 1000 snapshots, r = 4, polyorder = 2
(K = 27 library terms), fp32, synthetic pulsatile data generated on the device (12.6 GB per GPU, >> L2), POD init on the device.
Weak scaling by default (every rank owns an equally sized slab of points; only the (K*m + 29)-float `red` buffer is all-reduced);
`--scaling strong --total-points P` fixes the total instead.  One step = build_w + fused residual/grad pass + partial reduction +
(all-reduce) + regulariser/Adamax update, with the host-side ReduceLROnPlateau stepped at the reference script's cadence
(every epoch for the aneurysm / channel scripts, ANEU:613 / TURB:672; every 10th for the cylinder scripts, CYL:776-778).
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)
os.environ.setdefault("DESMO_KERNEL_EVENTS", "1")  # lets the library time its dominant kernel with CUDA events

WORKLOADS = {
    # name: (points per GPU, m, r, polyorder, nF, scheduler cadence of the script, patience, beta)
    "aneurysm-scale": (3 * 2 ** 20, 1000, 4, 2, 0, 1, 200, 1e-3),       # ANEU script's model at BASELINE's "millions of points"
    "aneurysm-script": (27000, 1000, 4, 2, 0, 1, 200, 1e-3),             # ANEU:551,613
    "cylinder-script": (3961, 1001, 4, 3, 0, 10, 1000, 1e-3),            # CYL:614,778
    "cylinder-8modes": (3961, 1001, 8, 2, 0, 10, 1000, 1e-3),            # BASELINE configs[0] ("8 modes"): K = 69
    "cylinder-8modes-p3": (3961, 1001, 8, 3, 0, 10, 1000, 1e-3),         # ... with the script's polyorder 3: K = 189
    "cylinder-fourier": (3961, 1001, 2, 2, 10, 10, 1000, 1e-3),          # FCYL
    "channel-script": (16384, 1000, 4, 2, 0, 1, 2000, 1e-6),             # TURB:612,672
    "channel-32modes": (16384, 1000, 32, 2, 0, 1, 2000, 1e-6),           # BASELINE configs[2] ("32 modes"): T = 561, K = 657
    "sweep": (10 ** 7, 1000, 8, 1, 0, 1, 2000, 1e-3),                    # BASELINE configs[4]; override with --points / --modes / --polyorder
}
METRIC = "train_iters_per_s"  # weak scaling: slab-iterations per second (N slabs per step at N GPUs); strong: whole-job iterations per second
UNIT = "it/s"
DUMP_BYTES = 64 * 2 ** 20  # --dump-outputs writes at most this much


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 0.0)), float(d.get("bf16_tflops_sustained", 0.0)), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: NVML polled every 2 ms (nvidia-smi as a fallback, ~10 Hz)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index: int):
        self.index, self.samples, self._stop = index, [], threading.Event()  # samples: (sm_mhz, sm_max_mhz, {reasons})
        self.power_w, self.power_limit_w = [], None
        self._ready = threading.Event()  # set after the first sample: NVML initialisation must not eat a short timed region
        self.th = threading.Thread(target=self._run, daemon=True)
        self.source = "nvml"

    def _run_nvml(self):
        import pynvml as nv

        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        try:
            self.power_limit_w = nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
        except Exception:
            pass
        k = 0
        while not self._stop.is_set():
            mask = int(get_reasons(h))
            self.samples.append((int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(mx), {n for n, b in self.BITS if mask & b}))
            self._ready.set()
            if k % 8 == 0:  # board power: a slow sensor, sampled every ~16 ms
                try:
                    self.power_w.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
            k += 1
            self._stop.wait(0.002)

    def _run_smi(self):
        self.source = "nvidia-smi"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                c = [v.strip() for v in out.split(",")]
                if len(c) >= 6 and c[0].isdigit():
                    names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
                    self.samples.append((int(c[0]), int(c[1]), {n for n, v in zip(names, c[2:6]) if v.lower().startswith("active")}))
                    self._ready.set()
            except Exception:
                pass
            self._stop.wait(0.05)

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def __enter__(self):
        self.th.start()
        self._ready.wait(timeout=10.0)  # the sampler is running before the timed region starts
        return self

    def __exit__(self, *a):
        self._stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(s[0] for s in self.samples)
        reasons = set().union(*[s[2] for s in self.samples]) if self.samples else set()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(s[1] for s in self.samples) if self.samples else None, "reasons": sorted(reasons),
                "samples": len(self.samples), "source": self.source,
                "power_w": round(sorted(self.power_w)[len(self.power_w) // 2], 1) if self.power_w else None,
                "power_limit_w": self.power_limit_w}


def synth_on_device(torch, n, m, dev, seed, x_offset=0, n_global=None):
    """Synthetic snapshots generated on the device straight into the padded time-major layout (SURVEY.md 8d C4 / C5): 8 smooth spatial
    fields x 5 temporal harmonics (pulsatile, aneurysm-like) + a counter-based hash noise that depends only on (global point,
    snapshot, seed) -- every world size sees the same global data --, temporal mean removed (CYL:136-149), scaled by 1/sqrt(m)
    (ANEU:143)."""
    ld = (n + 255) // 256 * 256
    n_global = n_global or n
    g = torch.Generator(device="cpu").manual_seed(seed)
    U = torch.zeros(m, ld, dtype=torch.float32, device=dev)
    rows = torch.arange(n, device=dev, dtype=torch.int64) + x_offset
    x = rows.to(torch.float64) / max(n_global - 1, 1)
    t = torch.arange(m, device=dev, dtype=torch.float64)
    for q in range(8):
        c = torch.randn(4, generator=g, dtype=torch.float64)
        ph = torch.rand(4, generator=g, dtype=torch.float64) * 3.141592653589793
        gq = sum(c[j] * torch.sin(3.141592653589793 * (j + 1) * (q + 1) * x + ph[j]) / (j + 1) for j in range(4))
        a = torch.randn(6, generator=g, dtype=torch.float64)
        psi = torch.rand(6, generator=g, dtype=torch.float64) * 6.283185307179586
        aq = (a[0] * 0 + sum(a[h] / h * torch.cos(6.283185307179586 * h * t / m + psi[h]) for h in range(1, 6))).to(torch.float32) / (q + 1)
        gq = gq.to(torch.float32)
        for t0 in range(0, m, 128):  # outer product in slabs: no m x n temporary
            U[t0:t0 + 128, :n].addcmul_(aq[t0:t0 + 128, None], gq[None, :])
    chunk = 32
    for t0 in range(0, m, chunk):
        tt = torch.arange(t0, min(t0 + chunk, m), device=dev, dtype=torch.int64)
        h = (rows[None, :] * 0x9E3779B1 + tt[:, None] * 0x85EBCA77 + (seed * 0xC2B2AE3D + 0x27D4EB2F)) & 0xFFFFFFFF
        h = ((h ^ (h >> 15)) * 0x2C1B3C6D) & 0xFFFFFFFF
        h = ((h ^ (h >> 12)) * 0x297A2D39) & 0xFFFFFFFF
        h = h ^ (h >> 15)
        U[t0:t0 + chunk, :n].add_(0.02 * 3.4641 * ((h & 0xFFFFFF).to(torch.float32) / 16777216.0 - 0.5))  # uniform, std 0.02
    U[:, :n].sub_(U[:, :n].mean(dim=0, keepdim=True))
    U.mul_(1.0 / m ** 0.5)
    return U


def cpu_reference_leg(kind, n_full, m, r, p, nF, steps, warmup, sample_points):
    """The reference's CPU implementation of the step (oracle/torch_port.py, all host threads) on a slab of `sample_points` points of
    the workload; `value` is scaled to the full slab only when the sample is smaller than it (then `extrapolated` says so)."""
    import numpy as np
    import torch

    from oracle import desmo_oracle as orc
    from oracle.torch_port import time_steps

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ns = min(n_full, sample_points)
    X = orc.synthetic_snapshots(kind, ns, m, seed=2)
    modes, _, _, _ = orc.pod_analysis(X, r)
    prm = orc.init_params(ns, m, p, r, nF=nF or None)
    sec, _ = time_steps(prm, modes, np.ascontiguousarray(X.T), steps, warmup)
    its_sample = 1.0 / sec
    extrap = ns < n_full
    return {"value": its_sample * ns / n_full, "unit": UNIT, "cores": cores, "kind": "port", "extrapolated": extrap,
            "extrapolation_factor": ns / n_full, "steps_run": steps, "warmup_run": warmup, "sample_ms_per_step": 1000.0 * sec,
            "sample_points": ns,
            "sample": f"{ns} of {n_full} points x {m} snapshots, {steps} steps after {warmup} warm-up, torch CPU fp32 "
                      f"{torch.get_num_threads()} threads, incl. the per-epoch fp64->fp32 re-collation (CYL:707-708); "
                      f"{its_sample:.3f} it/s on the sample" + (f", scaled by {ns}/{n_full} (cost is linear in the number of points)" if extrap else
                                                                " (the full workload, measured, not extrapolated)")}


def count_graph_kernels(torch, engine):
    """Kernel nodes of one captured train step (the launches a CUDA-graph replay performs), counted with the runtime's graph API."""
    try:
        from cuda.bindings import runtime as rt

        state = {k: getattr(engine, k).clone() for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u",
                                                         "omega", "omega_m", "omega_u", "step_dev", "hyper")}
        if engine.plateau_state is not None:  # the device scheduler's state: its kernel is one of the step's launches
            state["plateau_state"] = engine.plateau_state.clone()
        side = torch.cuda.Stream(device=engine.device)  # one eager step first: function attributes, NCCL communicator
        side.wait_stream(torch.cuda.current_stream(engine.device))
        with torch.cuda.stream(side):
            engine.train_step()
        torch.cuda.current_stream(engine.device).wait_stream(side)
        torch.cuda.synchronize(engine.device)
        g = torch.cuda.CUDAGraph(keep_graph=True)
        with torch.cuda.graph(g):
            engine.train_step()
        raw = g.raw_cuda_graph()
        err, _, n = rt.cudaGraphGetNodes(raw, 0)
        err, nodes, n = rt.cudaGraphGetNodes(raw, n)
        kernels = 0
        for nd in nodes:
            err, ty = rt.cudaGraphNodeGetType(nd)
            kernels += int(ty == rt.cudaGraphNodeType.cudaGraphNodeTypeKernel)
        for k, v in state.items():
            getattr(engine, k).copy_(v)
        return kernels, "counted (kernel nodes of the captured step)"
    except Exception as ex:  # older runtime bindings: fall back to the known launch sequence
        per = {1: 4, 2: 5}.get(engine.path_used)
        if per is None:
            chunks = -(-engine.ld // 16384)
            per = 2 + 4 * chunks + 3 + 2 + (1 if engine.r > 8 else 0)
        return per, f"formula ({type(ex).__name__})"


def step_outputs(torch, engine, budget=DUMP_BYTES):
    """What a caller of the train step holds after it, as host float32 arrays: the updated parameters in the packed layout, the losses
    the step computed (mse, ortho, l1, total) and the learning rates the scheduler left.  phi (r x points) is the only array that grows
    with the mesh: when everything does not fit in `budget` bytes, phi is cut to a fixed, seeded sample of points (same sample for the
    same shape in every run), whose indices are written beside it as phi_points (float64)."""
    import numpy as np

    e = engine
    out = {"losses": e.losses, "gates": e.gates, "omega": e.omega, "lrs": e.hyper[:5 if e.nF else 4]}
    if e.nF:
        out.update(coefs=e.coefs, periods=e.periods)
    else:
        out["rows"] = e.rows[:, :e.m]
    out = {k: v.detach().cpu().numpy() for k, v in out.items()}
    room = budget - sum(v.nbytes for v in out.values())
    if 4 * e.r * e.n <= room:
        out["phi"] = e.phi[:, :e.n].cpu().numpy()
    else:
        idx = np.sort(np.random.default_rng(0).choice(e.n, room // (4 * e.r + 8), replace=False))
        out["phi"] = e.phi[:, torch.from_numpy(idx).to(e.device)].cpu().numpy()
        out["phi_points"] = idx.astype(np.float64)
    return out


def sharded_parity(torch, dist, dev, rank, world, m, r, p, nF, path):
    """One small sharded fused pass (slabs of points + all-reduce of `red`) against the unsharded pass over the same global data on rank 0."""
    from desmo_b200 import DesmoEngine
    from desmo_b200.dist import shard_bounds

    n_g = 128 * 23 * world + 77
    lo, hi = shard_bounds(n_g, world, rank)

    def make(n, x_off, n_global, pg_active):
        e = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF or None, device=dev, n_global=n_global, path=path)
        rows = torch.arange(n, device=dev, dtype=torch.float64) + x_off
        for i in range(r):
            e.P[i, :n] = (torch.sin(0.37 * (i + 1) * rows / n_g * 6.283 + 0.2 * i) * (2.0 / n_g) ** 0.5).float()
            e.phi[i, :n] = (1.0 + 0.05 * torch.cos(0.11 * rows + i)).float()
        tt = torch.arange(m, device=dev, dtype=torch.float64)
        if not nF:
            for k in range(e.K):
                e.rows[k, :m] = (1.0 + 0.1 * torch.sin(0.05 * (k + 1) * tt)).float()
        e.U = synth_on_device(torch, n, m, dev, seed=7, x_offset=x_off, n_global=n_g)
        return e

    e = make(hi - lo, lo, n_g, True)
    e.build_w(False)
    e.fused_residual_grad()
    e.all_reduce()
    torch.cuda.synchronize()
    out = None
    if rank == 0:
        f = make(n_g, 0, n_g, False)
        f.build_w(False)
        f.fused_residual_grad()
        torch.cuda.synchronize()
        a, b = e.red.double(), f.red.double()
        out = {"rel_err": float((a - b).norm() / b.norm()), "points": n_g, "ranks": world}
    dist.barrier()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="desmo_b200", choices=["desmo_b200", "reference"])
    ap.add_argument("--workload", default="aneurysm-scale", choices=sorted(WORKLOADS))
    ap.add_argument("--points", type=int, default=0, help="override points per GPU (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--total-points", type=int, default=0, help="strong scaling: total mesh points over all GPUs (default: the workload's per-GPU size)")
    ap.add_argument("--modes", type=int, default=0, help="override r")
    ap.add_argument("--polyorder", type=int, default=-1, help="override polyorder")
    ap.add_argument("--path", type=int, default=0, help="0 auto, 1 fp32 FFMA, 2 fused tcgen05, 3 tcgen05 GEMM path")
    ap.add_argument("--allreduce", default="peer", choices=["peer", "nccl"],
                    help="N > 1: inter-rank sum of the partials -- one-shot exchange over NVLink peer memory (csrc/peer.cu) or NCCL")
    ap.add_argument("--host-scheduler", action="store_true",
                    help="step ReduceLROnPlateau on the host like the reference (one D2H sync per scheduler epoch) instead of inside the captured step")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pod", action="store_true", help="profiling runs: random orthonormal-scale modes instead of the POD init")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the parameters, losses and learning rates of the last timed step as DIR/<name>.npy "
                         "(at most 64 MB; rank 0's slab of phi): the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    n, m, r, p, nF, sched_every, patience, beta = WORKLOADS[args.workload]
    if args.modes:
        r = args.modes
    if args.polyorder >= 0:
        p = args.polyorder
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.points:
        n = args.points
    if args.scaling == "strong":
        total = args.total_points or n
        n_global = total
    else:
        n_global = n * world
    kind = "aneurysm" if args.workload.startswith(("aneurysm", "sweep")) else "channel" if args.workload.startswith("channel") else "cylinder"

    def config(n_local):
        return {"workload": f"{args.workload}: {n_local} points/GPU x {m} snapshots, r={r}, polyorder={p}" + (f", nF={nF}" if nF else "") +
                f", fp32, point-sharded, {args.scaling} scaling", "points_per_gpu": n_local, "points_total": n_global, "snapshots": m, "r": r,
                "polyorder": p, "scheduler_every": sched_every,
                "scheduler": ("ReduceLROnPlateau on the host (one D2H sync per scheduler epoch)" if getattr(args, "host_scheduler", False) else
                              "ReduceLROnPlateau inside the captured step (desmo_plateau_step): same schedule, no host round trip"),
                "cache": "inputs larger than L2 (streamed from HBM every step)" if n_local * m * 4 > 4e8 else "L2 flushed between steps"}

    if args.impl == "reference":
        if rank != 0:
            return
        # unit of `value` (both arms): weak scaling -- slab-iterations per second, a slab being one GPU's share (n points x m snapshots): the
        # host cores process slabs at the same rate whatever N is, the GPUs process N of them per step; strong -- whole-job iterations/s
        n_ref = n if args.scaling == "weak" else n_global
        leg = cpu_reference_leg(kind, n_ref, m, r, p, nF, args.steps, args.warmup, args.cpu_sample or 2 ** 15)
        line = {"impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1000.0 / leg["value"], "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config(n if args.scaling == "weak" else n_global // max(args.gpus, 1)),
                "extrapolated": leg["extrapolated"], "extrapolation_factor": leg["extrapolation_factor"],
                "sample_ms_per_step": leg["sample_ms_per_step"], "cpu_baseline": leg,
                "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if not args.no_cpu and n_ref > 27000:
            # a second, fully measured point: the aneurysm script's own shape (27000 x 1000, r = 4, p = 2) run in full on the host cores
            line["measured_pair_reference"] = cpu_reference_leg("aneurysm", 27000, 1000, 4, 2, 0, 5, 2, 27000)
        print(json.dumps(line))
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (desmo_b200 has no CPU fallback)")
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from desmo_b200 import DESMO, DesmoTrainer, _lib
    from desmo_b200.dist import shard_bounds

    if args.scaling == "strong":
        lo, hi = shard_bounds(n_global, world, rank)
        n, x_off = hi - lo, lo
    else:
        x_off = rank * n
    cfg = config(n)

    parity = sharded_parity(torch, dist, dev, rank, world, 200, r, p, nF, args.path) if world > 1 else None

    with contextlib.redirect_stdout(sys.stderr):  # the module prints the reference's banner (CYL:510); keep stdout = one JSON line
        model = DESMO(n, m, p, r, 10000, device=dev, n_global=n_global, path=args.path)
    e = model.engine
    e.U = synth_on_device(torch, n, m, dev, seed=2, x_offset=x_off, n_global=n_global)
    pod_info = None
    if args.no_pod or r > 14:
        # r > 14 exceeds the on-device eigensolver's block size: orthonormal-scale modes from a QR of smooth fields (setup only, not timed)
        rows = (torch.arange(n, device=dev, dtype=torch.float64) + x_off) / max(n_global - 1, 1)
        e.P[:, :n] = torch.stack([torch.sin(3.141592653589793 * (i + 1) * rows + 0.3 * i) for i in range(r)]).float() * (2.0 / n_global) ** 0.5
        sigma = torch.zeros(r)
        if not args.no_pod:
            pod_info = {"skipped": "r > 14: on-device eigensolver covers r <= 14; smooth orthonormal-scale modes used"}
    else:
        sigma = e.pod_from_snapshot()  # POD init on the device (method of snapshots)
        pod_info = dict(e.pod_timing)
        pod_info["err_pod_rank_r"] = e.pod_error  # POD_analysis' printed rank-r error (CYL:208-211)
        nt = (m + 127) // 128
        pod_info["gram_tflops_fp32_equiv"] = 2.0 * n * m * m / (pod_info["gram_ms"] * 1e-3) / 1e12
        # executed on the tensor pipe as 6 bf16 passes over 128-padded tiles of the upper triangle
        pod_info["gram_tensor_tflops_bf16_executed"] = 6 * 2.0 * n * (nt * (nt + 1) // 2) * 128 * 128 / (pod_info["gram_ms"] * 1e-3) / 1e12
    torch.cuda.synchronize()
    if world > 1 and args.allreduce == "peer":
        e.enable_peer_allreduce()  # collective; falls back to NCCL (peer_status says why) when peer-mapped memory is unavailable
    trainer = DesmoTrainer(model, beta=beta, patience=patience, sched_every=sched_every, use_cuda_graph=True,
                           device_scheduler=not args.host_scheduler)
    launches_per_step, launches_src = count_graph_kernels(torch, e)  # after the trainer: its device scheduler is part of the step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    l2_flush = None if n * m * 4 > 4e8 else torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for _ in range(args.warmup):
        trainer.step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    have_dom = e.path_used in (_lib.PATH_FP32, _lib.PATH_TC)  # the fused kernels are bracketed by CUDA events inside the library
    gk = ctypes.c_float(0.0)
    graph_samples = []  # dominant kernel inside replays of the captured step (external event nodes of the graph)

    def sample_graph_kernel():
        if have_dom and e.lib.desmo_graph_fused_kernel_ms(ctypes.byref(gk)) == 0:
            graph_samples.append(float(gk.value))

    with ClockSampler(local_rank) as clk:
        barrier()
        if l2_flush is None:
            ev0.record()
            for _ in range(args.steps):
                trainer.step()
            ev1.record()
            barrier()
            ms_total = ev0.elapsed_time(ev1)
            sample_graph_kernel()  # the dominant kernel inside the last step of the timed region
        else:
            ms_total = 0.0
            for _ in range(args.steps):
                l2_flush.fill_(1)
                ev0.record()
                trainer.step()
                ev1.record()
                torch.cuda.synchronize()
                ms_total += ev0.elapsed_time(ev1)
                sample_graph_kernel()
            barrier()
    # the measurements below run more steps: keep the state of the last timed one
    dumped = step_outputs(torch, e) if args.dump_outputs and rank == 0 else None
    # The dominant kernel's launch durations over a SECOND timed region of the same K steps (the 64 most recent at most), launched eagerly and back to back
    # (the library brackets the kernel with one CUDA event pair per launch on the launching stream; the events of a captured
    # step can only keep the last replay).  The region starts from the same state as the first one: synchronised, after a pause
    # that lets the board's power average decay -- under load the step time drifts upwards as the 1000 W limit is approached,
    # so a kernel timed in isolated, synchronised launches is not the kernel of the timed region.
    kms_series, eager_ms_step, clk_b = [], None, None
    n_eager = max(1, min(args.steps, 64))
    if have_dom:
        time.sleep(1.5)
        trainer.use_cuda_graph = False
        for _ in range(args.warmup):
            trainer.step()
        clk_b = ClockSampler(local_rank)
        clk_b.__enter__()
        barrier()
        e.lib.desmo_fused_kernel_ms_mean(None, None, 1)  # start a new series
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if l2_flush is None:
            r0.record()
            for _ in range(n_eager):
                trainer.step()
            r1.record()
            torch.cuda.synchronize()
            eager_ms_step = r0.elapsed_time(r1) / n_eager
        else:
            for _ in range(n_eager):
                l2_flush.fill_(1)
                trainer.step()
            torch.cuda.synchronize()
        clk_b.__exit__(None, None, None)
        trainer.use_cuda_graph = True
        buf, cnt = (ctypes.c_float * 64)(), ctypes.c_int32(0)
        _lib.check(e.lib.desmo_fused_kernel_ms_series(buf, 64, ctypes.byref(cnt)), "desmo_fused_kernel_ms_series")
        kms_series = [float(buf[i]) for i in range(cnt.value)]
    # the whole fused call (dominant kernel + chain rule + partial reduction), eager launches back to back, torch events
    e.build_w(False)
    torch.cuda.synchronize()
    pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_eager)]
    for k0, k1 in pairs:
        if l2_flush is not None:
            l2_flush.fill_(1)
        k0.record()
        e.fused_residual_grad()
        k1.record()
    torch.cuda.synchronize()
    kms = sum(k0.elapsed_time(k1) for k0, k1 in pairs) / n_eager
    if kms_series:
        kms_dom = sum(kms_series) / len(kms_series)
        kms_src = (f"mean of {len(kms_series)} launches: one CUDA event pair per launch around the kernel on its launching stream, over a "
                   "second timed region of back-to-back eager steps (region_ms_per_step beside it); kernel_ms_graph_last_step = the same "
                   "kernel inside the last replay of the first (graph) region")
    else:
        kms_dom, kms_src = kms, "the whole fused call (torch events, eager launches back to back)"
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    losses = [float(v) for v in e.losses.tolist()]

    # ---- e2e: the reference-facing C-ABI call with HOST buffers (H2D of the batch + sharded step + D2H of the losses, every step) ----
    e2e = None
    if not args.no_e2e:
        try:
            lib = _lib.load()
            import numpy as np
            import psutil

            local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
            if 4.0 * n * m * local_world > 0.6 * psutil.virtual_memory().available:  # never drive the box out of memory
                raise RuntimeError(f"host memory too small for {local_world} pinned batches of {4.0 * n * m / 1e9:.1f} GB")
            host = torch.empty(m, n, dtype=torch.float32, pin_memory=True)
            host.copy_(e.U[:, :n])
            ss = ctypes.c_void_p()
            _lib.check(lib.desmo_session_create_sharded(n, n_global, m, r, p, nF, args.path, ctypes.byref(ss)), "session_create_sharded")
            hook = _lib.torch_allreduce_hook() if world > 1 else None
            if hook is not None:
                _lib.check(lib.desmo_session_set_allreduce(ss, ctypes.cast(hook, ctypes.c_void_p), None), "session_set_allreduce")
            pod = np.ascontiguousarray(e.P[:, :n].t().double().cpu().numpy())
            K = e.K
            phi0 = np.ones((r, n), np.float32); gates0 = np.ones(K, np.float32)
            rows0 = np.ones((K, 2 * nF + 1 if nF else m), np.float32); per0 = np.full(K, 60.0, np.float32)
            om0 = np.full(3 * r, 1e4, np.float32); lrs = np.array([1e-2, 1e-3, 1e-2, 1e3, 1e-2], np.float32)
            cp = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
            _lib.check(lib.desmo_session_set_pod_host(ss, cp(pod)), "set_pod")
            _lib.check(lib.desmo_session_set_params_host(ss, cp(phi0), cp(gates0), cp(rows0), cp(per0) if nF else None, cp(om0)), "set_params")
            _lib.check(lib.desmo_session_set_hyper(ss, cp(lrs), beta, 1e-4), "set_hyper")
            lo_ = np.zeros(4, np.float32)
            e_steps = max(2, min(args.steps, 5 if n * m * 4 > 4e8 else 50))
            _lib.check(lib.desmo_session_step_host(ss, ctypes.c_void_p(host.data_ptr()), cp(lo_)), "step_host")  # warm-up
            barrier()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                _lib.check(lib.desmo_session_step_host(ss, ctypes.c_void_p(host.data_ptr()), cp(lo_)), "step_host")
            torch.cuda.synchronize()
            dt = torch.tensor([(time.perf_counter() - t0) / e_steps], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            lib.desmo_session_destroy(ss)
            units = world if args.scaling == "weak" else 1
            e2e = {"value": units / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": int(n * m * 4), "d2h_bytes_per_step": 16,
                   "steps": e_steps, "mse_last_step": float(lo_[0]),
                   "call": "desmo_session_step_host (pinned host batch -> device, fused step" +
                           (", NCCL all-reduce of red through the session's hook" if world > 1 else "") + ", losses -> host)",
                   "bound": "PCIe: the reference re-sends the whole batch every epoch (CYL:707-708); pass NULL to keep the resident copy"}
            del host
        except Exception as ex:  # keep the device-resident number even if the host leg cannot run (e.g. pinned alloc)
            e2e = {"value": None, "unit": UNIT, "error": str(ex)[:200]}

    if rank == 0:
        peak, tpeak, tpeak_sus, peak_src = load_peaks()
        units = world if args.scaling == "weak" else 1
        alg_bytes = 4.0 * n * m + 12.0 * n * r + 8.0 * e.K * m  # U once; phi, P in, dphi out; W in, E out
        achieved = alg_bytes / (kms_dom * 1e-3) / 1e9
        kernel_name = {1: "fused_fp32_kernel", 2: "fused_tc_kernel", 3: "gemm_planes_kernel x3 per chunk (GEMM path, whole fused call)"}[e.path_used]
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": kernel_name, "kernel_ms": kms_dom, "kernel_ms_source": kms_src,
                "kernel_ms_series": [round(v, 4) for v in kms_series], "region_ms_per_step": eager_ms_step,
                "region_clocks": clk_b.summary() if clk_b is not None else None,
                "kernel_ms_graph_last_step": [round(v, 4) for v in graph_samples][-1:] if l2_flush is None else
                [round(sum(graph_samples) / max(len(graph_samples), 1), 4)], "fused_call_ms": kms, "peak_source": peak_src,
                "algorithmic_bytes": alg_bytes}
        if e.path_used == _lib.PATH_GEMM:
            # K > 32: 6 K n m flop on 4 n m bytes -- bound by the tensor pipe (SURVEY.md 8d); report both roofs, name the binding one
            flop_alg = 6.0 * e.K * n * m
            # bf16 MMA flops executed: GEMM 1 six plane products, GEMM 3 / 4 three each, on K padded to 64 (contraction) / 16 (N)
            flop_exec = 2.0 * n * m * (6 * (-(-e.K // 64) * 64) + 2 * 3 * (-(-e.K // 16) * 16))
            roof = {"bound": "tensor", "achieved": flop_exec / (kms * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                    "frac": flop_exec / (kms * 1e-3) / 1e12 / tpeak, "traffic": None, "kernel": kernel_name, "kernel_ms": kms,
                    "fused_call_ms": kms, "peak_source": peak_src, "algorithmic_flops": flop_alg, "executed_bf16_flops": flop_exec,
                    "fp32_equivalent_tflops": flop_alg / (kms * 1e-3) / 1e12, "hbm_frac": achieved / peak, "algorithmic_bytes": alg_bytes}
        line = {"metric": METRIC, "value": units / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": cfg,
                "global_iters_per_s": 1.0 / (ms_step * 1e-3),
                "snapshot_gbs": 4.0 * n_global * m / (ms_step * 1e-3) / 1e9,
                "roofline": roof, "clocks": clk.summary(), "e2e": e2e,
                "gpu_launches": launches_per_step * args.steps + (args.steps if world > 1 and e._peer is None else 0),
                "gpu_launches_per_step": launches_per_step, "gpu_launches_source": launches_src,
                "losses_last_step": losses, "pod_sigma": [float(v) for v in sigma.tolist()], "pod_init": pod_info,
                "path": _lib.PATH_NAMES[e.path_used],
                "allreduce": ("none (single GPU)" if world == 1 else
                              "peer memory, one-shot, rank-ordered (csrc/peer.cu)" if e._peer is not None else
                              f"NCCL (peer exchange {e.peer_status})")}
        if parity is not None:
            line["sharded_parity"] = parity
        try:
            with open(os.path.join(ROOT, "profiles", "traffic_r02.json")) as fh:
                tr = json.load(fh)
            if tr.get("points_per_gpu") == n and tr.get("path") == e.path_used:
                line["roofline"]["traffic"] = tr["dram_bytes_per_launch"]
                line["roofline"]["traffic_source"] = "static: ncu capture committed under profiles/ (not measured in this run)"
        except Exception:
            pass
        if not args.no_cpu and world == 1:
            try:
                line["cpu_baseline"] = cpu_reference_leg(kind, n, m, r, p, nF, 5, 2, args.cpu_sample or 2 ** 14)
                if n > 27000:
                    # a fully measured pair (no extrapolation): the aneurysm script's own shape on the host cores vs this GPU
                    line["measured_pair"] = {"workload": "aneurysm-script 27000 x 1000, r=4, polyorder=2",
                                             "cpu": cpu_reference_leg("aneurysm", 27000, 1000, 4, 2, 0, 5, 2, 27000),
                                             "gpu": small_gpu_pair(torch, dev, 27000, 1000, 4, 2)}
            except Exception as ex:
                line["cpu_baseline"] = {"value": None, "error": str(ex)[:200]}
        if dumped is not None:
            import numpy as np

            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line), flush=True)
    if world > 1:
        # tear-down of a process group whose collectives were captured in a CUDA graph can block; everything is measured and
        # printed, so leave without the destructor dance (exit code 0 for torchrun)
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def small_gpu_pair(torch, dev, n, m, r, p):
    """Device-resident and host-fed (e2e) train rate of this framework at a script-sized workload, L2 flushed between steps."""
    import numpy as np

    from desmo_b200 import DESMO, DesmoTrainer, _lib

    with contextlib.redirect_stdout(sys.stderr):
        model = DESMO(n, m, p, r, 10000, device=dev)
    e = model.engine
    e.U = synth_on_device(torch, n, m, dev, seed=2)
    e.pod_from_snapshot()
    tr = DesmoTrainer(model, patience=200, sched_every=1)
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for _ in range(5):
        tr.step()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = 0.0
    for _ in range(50):
        flush.fill_(1)
        ev0.record()
        tr.step()
        ev1.record()
        torch.cuda.synchronize()
        ms += ev0.elapsed_time(ev1)
    lib = _lib.load()
    host = torch.empty(m, n, dtype=torch.float32, pin_memory=True)
    host.copy_(e.U[:, :n])
    ss = ctypes.c_void_p()
    _lib.check(lib.desmo_session_create(n, m, r, p, 0, 0, ctypes.byref(ss)), "session_create")
    cp = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    pod = np.ascontiguousarray(e.P[:, :n].t().double().cpu().numpy())
    K = e.K
    _lib.check(lib.desmo_session_set_pod_host(ss, cp(pod)), "set_pod")
    _lib.check(lib.desmo_session_set_params_host(ss, cp(np.ones((r, n), np.float32)), cp(np.ones(K, np.float32)), cp(np.ones((K, m), np.float32)),
                                                 None, cp(np.full(3 * r, 1e4, np.float32))), "set_params")
    _lib.check(lib.desmo_session_set_hyper(ss, cp(np.array([1e-2, 1e-3, 1e-2, 1e3, 1e-2], np.float32)), 1e-3, 1e-4), "set_hyper")
    lo_ = np.zeros(4, np.float32)
    for _ in range(3):
        _lib.check(lib.desmo_session_step_host(ss, ctypes.c_void_p(host.data_ptr()), cp(lo_)), "step_host")
    t0 = time.perf_counter()
    for _ in range(50):
        _lib.check(lib.desmo_session_step_host(ss, ctypes.c_void_p(host.data_ptr()), cp(lo_)), "step_host")
    dt = (time.perf_counter() - t0) / 50
    lib.desmo_session_destroy(ss)
    return {"value": 1000.0 / (ms / 50), "e2e_value": 1.0 / dt, "unit": UNIT, "steps": 50,
            "note": "device-resident: CUDA-graph replay + per-epoch loss fetch, L2 flushed between steps; e2e: desmo_session_step_host with the "
                    "108 MB batch re-sent from pinned host memory every step"}


if __name__ == "__main__":
    main()
