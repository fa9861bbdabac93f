"""Training step of a Fourier model at a caller-given time table (DesmoEngine.set_time_points) against the same step on the grid, in ONE
process: at each shape the step without a table and the step with a table (sorted random times in [0, m)) are each captured in a CUDA
graph and their replays alternated, `--reps` steps per timed window (CUDA events, after a warm-up), `--rounds` windows per configuration;
the median window is reported.  The table changes one operand of build_w and of the Fourier gradients in the update (a load per column
instead of t_point's arithmetic), so the expectation is no difference beyond noise.  Shapes (fp32 storage, U far larger than the 126 MB
L2), 3 * 2^20 points x 1000 snapshots:
  fcyl   r = 2, p = 2, nF = 10, K = 12 (the FCYL library, fused tcgen05 path)
  faneu  r = 2, p = 2, nF = 30, K = 12 (FANEU's nF, fused tcgen05 path)
  gemm   r = 4, p = 3, nF = 10, K = 47 (GEMM path)
A separate torch.profiler pass gives the device time per kernel of one step of each kind.  The card's name, power limit and maximum SM
clock are read in the same run.  One JSON object is printed (and written to --out).

    python tools/time_points_time.py [--rounds 7] [--reps 50] [--out FILE] [--shapes a,b]"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from active_terms_time import capture, kernel_breakdown, smi, window_ms  # noqa: E402
from desmo_b200 import DesmoEngine  # noqa: E402

N = 3 * 2 ** 20
SHAPES = {"fcyl": (N, 1000, 2, 2, 10, 0), "faneu": (N, 1000, 2, 2, 30, 0), "gemm": (N, 1000, 4, 3, 10, 3)}


def make_engine(n, m, r, p, nF, path, dev):
    """U = a few travelling modes + 2 % noise (fp32), smooth modes in P, learning rates small enough to keep the state finite."""
    g = torch.Generator(device=dev).manual_seed(0)
    e = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF, period_init=200.0, device=dev, path=path)
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


def run_shape(label, n, m, r, p, nF, path, dev, rounds, reps):
    e = make_engine(n, m, r, p, nF, path, dev)
    table = np.sort(np.random.default_rng(0).uniform(0.0, m, m)).astype(np.float32)
    graphs = {"grid": capture(e)}
    e.set_time_points(table)
    graphs["table"] = capture(e)
    for g in graphs.values():
        window_ms(g, 5)
    times = {name: [] for name in graphs}
    for _ in range(rounds):
        for name, g in graphs.items():  # alternated: drift of clocks and co-tenants hits both configurations alike
            times[name].append(window_ms(g, reps))
    med = {k: statistics.median(v) for k, v in times.items()}
    spread = {k: round(100.0 * (max(v) - min(v)) / med[k], 2) for k, v in times.items()}
    res = {"n": n, "m": m, "r": r, "polyorder": p, "nF": nF, "K": e.K, "path_used": e.path_used,
           "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
           "ms_per_step_windows": {k: [round(x, 4) for x in v] for k, v in times.items()},
           "table_over_grid": round(med["table"] / med["grid"], 4), "spread_pct": spread}
    kernels = {"table": kernel_breakdown(e)}
    e.set_time_points(None)
    kernels["grid"] = kernel_breakdown(e)
    res["kernels_ms"] = {k: {name: v for name, v in kb.items() if "build_w" in name or "update_kernel" in name} for k, kb in kernels.items()}
    del graphs, e
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    name, plimit, maxsm = smi("name,power.limit,clocks.max.sm")
    out = {"gpu": name, "power_limit_w": plimit, "max_sm_clock_mhz": maxsm, "rounds": a.rounds, "reps": a.reps, "storage": "fp32",
           "shapes": {}}
    for label in a.shapes.split(","):
        out["shapes"][label] = run_shape(label, *SHAPES[label], dev, a.rounds, a.reps)
        print(label, json.dumps(out["shapes"][label]["ms_per_step_median"]), out["shapes"][label]["table_over_grid"], flush=True)
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
