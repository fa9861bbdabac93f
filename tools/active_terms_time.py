"""Training step on an active set of library terms (DesmoEngine.set_active_terms) against the unmasked step, in ONE process: at each
shape the unmasked step and masked steps at Ka = K, K/2, K/4, K/10 (seeded random sets) are each captured in a CUDA graph and their
replays alternated, `--reps` steps per timed window (CUDA events, after a warm-up), `--rounds` windows per configuration; the median
window is reported.  Shapes (fp32 storage, U far larger than the 126 MB L2):
  channel-32modes  262144 x 1000, r = 32, p = 2, K = 657 (GEMM path)
  cylinder-gemm    1048576 x 1000, r = 4, p = 3, K = 47 (the cylinder library, GEMM path)
  headline         3 * 2^20 x 1000, r = 4, p = 2, K = 27 (fused tcgen05 path)
A separate torch.profiler pass gives the device time per kernel of one unmasked and one Ka = K/10 step at each shape.  The card's name,
power limit and maximum SM clock are read in the same run.  One JSON object is printed (and written to --out).

    python tools/active_terms_time.py [--rounds 5] [--reps 50] [--out FILE] [--shapes a,b]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from desmo_b200 import DesmoEngine  # noqa: E402

SHAPES = {"channel-32modes": (262144, 1000, 32, 2), "cylinder-gemm": (1048576, 1000, 4, 3), "headline": (3 * 2 ** 20, 1000, 4, 2)}


def smi(fields):
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, timeout=20)
    return [v.strip() for v in out.stdout.strip().split(",")]


def make_engine(n, m, r, p, dev):
    """U = a few travelling modes + 2 % noise (fp32), smooth modes in P, learning rates small enough to keep the state finite."""
    g = torch.Generator(device=dev).manual_seed(0)
    e = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev)
    x = torch.linspace(0, 1, n, device=dev)
    e.P[:, :n] = torch.stack([torch.sin(3.1416 * (k + 1) * x + 0.3 * k) for k in range(r)]) * (2.0 / n) ** 0.5
    e.U = torch.zeros(m, e.ld, dtype=torch.float32, device=dev)
    for t0 in range(0, m, 100):
        t = torch.linspace(0, 1, m, device=dev)[t0:t0 + 100]
        Us = sum(torch.cos(6.2832 * (k + 1) * t + k)[:, None] * torch.sin(3.1416 * (k + 1) * x + 0.3 * k)[None, :] / (k + 1) for k in range(5))
        e.U[t0:t0 + Us.shape[0], :n] = Us + 0.02 * torch.randn(Us.shape, device=dev, generator=g)
        del Us
    e.set_hyper([1e-6] * 5, 1e-3, 1e-4)
    torch.cuda.synchronize()
    return e


def masks(K, seed=0):
    rng = np.random.default_rng(seed)
    out = {"unmasked": None, "Ka=K": np.ones(K, bool)}
    for div in (2, 4, 10):
        m = np.zeros(K, bool)
        m[np.sort(rng.choice(K, size=max(1, round(K / div)), replace=False))] = True
        out[f"Ka=K/{div}"] = m
    return out


def capture(e):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        e.train_step()  # warm-up outside the capture (function attributes, first launches)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        e.train_step()
    return g


def window_ms(g, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_breakdown(e):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e.train_step()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t and ev.count:
            name = ev.key.split("(")[0].replace("void ", "")
            out[name] = {"ms": round(out.get(name, {}).get("ms", 0.0) + t / 1000.0, 4), "launches": out.get(name, {}).get("launches", 0) + ev.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms"]))


def run_shape(label, n, m, r, p, dev, rounds, reps):
    e = make_engine(n, m, r, p, dev)
    cfg = masks(e.K)
    graphs, keep = {}, []
    for name, mk in cfg.items():
        e.set_active_terms(mk)
        keep.append(e._active)  # each graph holds its own table's address
        graphs[name] = capture(e)
    for g in graphs.values():  # warm-up of every graph
        window_ms(g, 5)
    times = {name: [] for name in graphs}
    for _ in range(rounds):
        for name, g in graphs.items():  # alternated: drift of clocks and co-tenants hits every configuration alike
            times[name].append(window_ms(g, reps))
    med = {k: statistics.median(v) for k, v in times.items()}
    base = med["unmasked"]
    res = {"n": n, "m": m, "r": r, "polyorder": p, "K": e.K, "path_used": e.path_used,
           "Ka": {k: (e.K if v is None else int(v.sum())) for k, v in cfg.items()},
           "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
           "ms_per_step_windows": {k: [round(x, 4) for x in v] for k, v in times.items()},
           "speedup_vs_unmasked": {k: round(base / v, 3) for k, v in med.items()},
           "spread_unmasked_pct": round(100.0 * (max(times["unmasked"]) - min(times["unmasked"])) / base, 2)}
    e.set_active_terms(None)
    res["kernels_unmasked"] = kernel_breakdown(e)
    e.set_active_terms(cfg["Ka=K/10"])
    res["kernels_Ka=K/10"] = kernel_breakdown(e)
    del graphs, keep, e
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device (sm_100a); nothing is measured without one")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, plimit, maxclk = smi("name,power.limit,clocks.max.sm")
    out = {"gpu": name, "power_limit_w": plimit, "max_sm_clock_mhz": maxclk, "rounds": args.rounds, "reps": args.reps,
           "method": "CUDA-graph replays of one train_step, reps per event-timed window, configurations alternated, median window",
           "shapes": {}}
    for label in args.shapes.split(","):
        out["shapes"][label] = run_shape(label, *SHAPES[label], dev, args.rounds, args.reps)
        print(label, json.dumps(out["shapes"][label]["ms_per_step_median"]), flush=True)
    txt = json.dumps(out, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
