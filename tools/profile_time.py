"""Residual profile (DesmoEngine.residual_profile) against the graph-replayed training step, fp32 and bf16 storage of U alternated in
ONE process, at the headline shape; then the channel "32 modes" shape (r = 32, p = 2, K = 657).

    python tools/profile_time.py [--n 3145728] [--m 1000] [--reps 20] [--rounds 3] [--out FILE]

Per storage and shape: ms per graph-replayed DesmoTrainer step and per residual_profile() call (CUDA events after warm-up; U is far
larger than the 126 MB L2, so every call streams it from HBM), the algorithmic bytes of a profile call (U once, phi and P, W, the
outputs) and their share of the HBM peak that bench.py's load_peaks() returns (MEASURED_PEAKS.json when present, else its fallback;
the JSON says which), and a per-kernel device-time breakdown of one profile call from torch.profiler (a separate pass, so tracing does
not disturb the timed numbers).  The card's name and power limit are read in the same run.  One JSON object is printed (and written
to --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import load_peaks  # noqa: E402
from desmo_b200 import DesmoEngine, DesmoTrainer  # noqa: E402

LRS = (1e-2, 1e-3, 1e-2, 1e-2)


def smi(fields):
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, timeout=20)
    return [v.strip() for v in out.stdout.strip().split(",")]


def make_engines(n, m, r, p, dev):
    """One engine per storage with the same parameters; U = a few travelling modes + 2 % noise, U_q.float() for the fp32 engine."""
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.linspace(0, 1, n, device=dev)
    P = torch.stack([torch.sin(3.1416 * (k + 1) * x + 0.3 * k) for k in range(r)]) * (2.0 / n) ** 0.5
    eng = {}
    for dt in (torch.bfloat16, torch.float32):
        e = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev, snapshot_dtype=dt)
        e.P[:, :n] = P
        e.rows[:, :m] = 1.0
        e.U = torch.zeros(m, e.ld, dtype=dt, device=dev)
        eng[dt] = e
    eb, ef = eng[torch.bfloat16], eng[torch.float32]
    for t0 in range(0, m, 100):
        t = torch.linspace(0, 1, m, device=dev)[t0:t0 + 100]
        Us = sum(torch.cos(6.2832 * (k + 1) * t + k)[:, None] * torch.sin(3.1416 * (k + 1) * x + 0.3 * k)[None, :] / (k + 1) for k in range(5))
        src = (Us + 0.02 * torch.randn(Us.shape, device=dev, generator=g)).contiguous()
        eb.lib.desmo_snapshot_to_bf16(C.byref(eb.shape), src.data_ptr(), src.stride(0), t0, src.shape[0], eb.U.data_ptr(), None,
                                      torch.cuda.current_stream().cuda_stream)
        ef.U[t0:t0 + src.shape[0], :n] = src.bfloat16().float()
        del Us, src
    torch.cuda.synchronize()
    return eng


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_breakdown(e):
    """Device time per kernel of one residual_profile() call (torch.profiler, CUDA activities), summed over its launches."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e.residual_profile()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t and ev.count:
            name = ev.key
            for short in ("library_planes_kernel", "w_planes_kernel", "term_table_kernel", "profile_points_kernel", "profile_snapshots_kernel",
                          "gemm_planes_kernel", "Memset"):
                if short in name:
                    name = short
            out[name] = {"ms": round(t / 1000.0, 4), "launches": ev.count}
    return out


def run_shape(label, n, m, r, p, dev, reps, rounds, hbm_gbs):
    eng = make_engines(n, m, r, p, dev)
    trainers = {dt: DesmoTrainer(e, lrs=LRS, beta=1e-3, l1_lambda=1e-4, use_cuda_graph=True) for dt, e in eng.items()}
    for dt, tr in trainers.items():  # warm-up: graph capture, first launches, the allocator's pool for the profile's scratch
        for _ in range(5):
            tr.step()
        for _ in range(3):
            eng[dt].residual_profile()
    torch.cuda.synchronize()
    res = {}
    for rnd in range(rounds):
        for dt in ((torch.float32, torch.bfloat16) if rnd % 2 == 0 else (torch.bfloat16, torch.float32)):
            key = str(dt).replace("torch.", "")
            out = res.setdefault(key, {"step_ms": [], "profile_ms": []})
            out["step_ms"].append(round(timed(trainers[dt].step, reps), 4))
            out["profile_ms"].append(round(timed(eng[dt].residual_profile, reps), 4))
    a, b = eng[torch.bfloat16].residual_profile(), eng[torch.float32].residual_profile()
    parity = all(torch.equal(a[k], b[k]) for k in a)
    for dt, e in eng.items():
        key = str(dt).replace("torch.", "")
        out = res[key]
        alg = (2 if dt == torch.bfloat16 else 4) * n * m + 8 * n * r + 4 * e.Kp * e.mld + 16 * m + 8 * e.ld
        best = min(out["profile_ms"])
        out["profile_algorithmic_bytes"] = alg
        out["profile_hbm_floor_ms"] = round(alg / hbm_gbs / 1e6, 4)
        out["profile_share_of_hbm_floor"] = round(alg / hbm_gbs / 1e6 / best, 4)
        out["profile_kernels"] = kernel_breakdown(e)
    del trainers, eng
    torch.cuda.empty_cache()
    return {"shape": label, "n": n, "m": m, "r": r, "p": p, "bitwise_bf16_vs_fp32_of_uq": parity, "storages": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3 << 20)
    ap.add_argument("--m", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("profile_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    name, plim = smi("name,power.limit")
    hbm_gbs, _, _, peak_src = load_peaks()
    shapes = [run_shape("headline r4p2", a.n, a.m, 4, 2, dev, a.reps, a.rounds, hbm_gbs),
              run_shape("channel-32modes", 262144, 1000, 32, 2, dev, max(3, a.reps // 4), a.rounds, hbm_gbs)]
    rep = {"card": name, "power_limit_w": float(plim), "hbm_peak_gbs": hbm_gbs, "hbm_peak_source": peak_src, "shapes": shapes}
    txt = json.dumps(rep, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
