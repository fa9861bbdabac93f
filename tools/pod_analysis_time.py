"""Cost of the dense POD eigensolver (desmo_pod_eigh) and of DesmoEngine.pod_analysis(), in ONE process.

    python tools/pod_analysis_time.py [--reps 5] [--rounds 3] [--out FILE]             # timings
    python tools/pod_analysis_time.py --profile [--out FILE]                            # per-kernel split (torch.profiler), separate run

Timings (CUDA events after warm-up):
  - desmo_pod_eigh at m in {1000, 2000, 4096} and r in {4, 14, 32, 64} on the Gram of seeded data with sigma_i ~ (i+1)^-0.5;
    at r <= 14 the subspace solver desmo_pod_eig runs on the same Gram in the same rounds, the two alternating;
  - pod_analysis() end to end (Gram, eigensolve, projection; pod_timing) at 3 * 2^20 x 1000, r = 4, and at the channel-32modes shape
    262144 x 1000, r = 32; pod_from_snapshot() at the first for comparison.
The card's name and power limit are read in the same run.  One JSON object is printed (and written to --out)."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from profile_time import smi, timed  # noqa: E402

from desmo_b200 import DesmoEngine, _lib, ops  # noqa: E402,F401

MS, RS = (1000, 2000, 4096), (4, 14, 32, 64)


def gram(m, dev):
    g = torch.Generator(device=dev).manual_seed(m)
    X = torch.randn(m + 7, m, generator=g, device=dev, dtype=torch.float64) * (torch.arange(m, device=dev, dtype=torch.float64) + 1) ** -0.5
    return (X.T @ X).float().contiguous()


def eigh_call(Cm, r):
    m = Cm.shape[0]
    nbytes = C.c_size_t(0)
    _lib.check(_lib.load().desmo_pod_eigh_workspace_bytes(m, r, C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=Cm.device)
    S = torch.empty(m, dtype=torch.float64, device=Cm.device)
    V, sigma = torch.empty(r, m, device=Cm.device), torch.empty(r, device=Cm.device)
    return lambda: torch.ops.desmo_b200.pod_eigh(Cm, S, V, sigma, ws, m, r), ws


def eig_call(Cm, r):
    m = Cm.shape[0]
    ws = torch.zeros(2 * 8 * 16 * m + 1024, dtype=torch.uint8, device=Cm.device)
    V, sigma = torch.empty(r, m, device=Cm.device), torch.empty(r, device=Cm.device)
    return lambda: torch.ops.desmo_b200.pod_eig(Cm, V, sigma, ws, m, r), ws


def solver_times(dev, reps, rounds):
    out = {}
    for m in MS:
        Cm = gram(m, dev)
        calls = {}
        for r in RS:
            calls[f"eigh m={m} r={r}"] = eigh_call(Cm, r)
            if r <= 14:
                calls[f"eig m={m} r={r}"] = eig_call(Cm, r)
        for fn, _ in calls.values():
            fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in calls}
        names = list(calls)
        for rnd in range(rounds):
            for k in (names if rnd % 2 == 0 else names[::-1]):
                ms[k].append(round(timed(calls[k][0], reps), 3))
        for k, (_, ws) in calls.items():
            rep = {"ms": ms[k], "ms_best": min(ms[k])}
            if k.startswith("eigh"):
                rep["status"] = int(ws[:4].view(torch.int32).item())
                rep["residual_over_lambda1"] = float(ws[8:16].view(torch.float64).item())
            else:
                rep["sweeps"], rep["converged"] = ws[:8].view(torch.int32).tolist()
            out[k] = rep
        del Cm, calls
        torch.cuda.empty_cache()
    return out


def e2e(dev):
    out = {}
    for label, n, m, r in (("3x2^20 x 1000 r=4", 3 << 20, 1000, 4), ("channel-32modes 262144 x 1000 r=32", 262144, 1000, 32)):
        e = DesmoEngine(n, m, 2, r, omega_init=10.0, device=dev)
        g = torch.Generator(device=dev).manual_seed(1)
        e.U = torch.zeros(m, e.ld, device=dev)
        for t0 in range(0, m, 100):   # a few travelling modes plus 2 % noise
            t = torch.linspace(0, 1, m, device=dev)[t0:t0 + 100, None]
            x = torch.linspace(0, 1, n, device=dev)[None, :]
            blk = sum(torch.sin(6.2832 * (k + 1) * (x - 0.3 * t)) / (k + 1) for k in range(12))
            e.U[t0:t0 + 100, :n] = blk + 0.02 * torch.randn(blk.shape, generator=g, device=dev)
        runs = []
        for _ in range(3):
            e.pod_analysis()
            runs.append({k: round(v, 3) for k, v in e.pod_timing.items()})
        out[label] = {"pod_analysis": runs, "eigh_residual_over_lambda1": e.pod_eig_residual}
        if r <= 14:
            sub = []
            for _ in range(3):
                e.pod_from_snapshot()
                sub.append({k: round(v, 3) for k, v in e.pod_timing.items()})
            out[label]["pod_from_snapshot"] = sub
        del e
        torch.cuda.empty_cache()
    return out


def profile(dev):
    from torch.profiler import ProfilerActivity, profile as prof

    out = {}
    for m, r in ((1000, 4), (1000, 64), (4096, 64)):
        Cm = gram(m, dev)
        fn, _ = eigh_call(Cm, r)
        fn()
        torch.cuda.synchronize()
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            fn()
            torch.cuda.synchronize()
        split = {}
        for ev in p.key_averages():
            if ev.device_type == torch.autograd.DeviceType.CUDA and "eigh" in ev.key:
                split[ev.key] = round(ev.device_time_total / 1000.0, 3)
        out[f"m={m} r={r}"] = dict(sorted(split.items(), key=lambda kv: -kv[1]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pod_analysis_time.py needs a CUDA device")
    dev = torch.device("cuda:0")
    name, limit = smi("name,power.limit")
    res = {"gpu": name, "power_limit_w": limit}
    if a.profile:
        res["kernel_ms"] = profile(dev)
    else:
        res["solver"] = solver_times(dev, a.reps, a.rounds)
        res["end_to_end"] = e2e(dev)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
