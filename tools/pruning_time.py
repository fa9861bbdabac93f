"""Pruning profile (DesmoEngine.pruning_profile, full removal order) against greedy_removal (one residual_norm2() pass per step) and one
residual_profile() call, fp32 and bf16 storage of U alternated in ONE process, at the headline shape (3 * 2^20 x 1000, r = 4, p = 2,
K = 27) and the channel "32 modes" shape (262144 x 1000, r = 32, p = 2, K = 657).

    python tools/pruning_time.py [--rounds 2] [--reps 5] [--out FILE]

Per storage and shape: ms per pruning_profile() and residual_profile() call (CUDA events after warm-up, mean of --reps calls) and per
greedy_removal() sweep (host clock around the sweep, which ends in a device synchronise), the speed-up over the sweep, the ratio to
residual_profile(), the FFMA and U-read floors of the profile (2 (S + 1) n m FFMA at 128 FFMA / clock / SM and the card's maximum SM
clock; U's bytes at the HBM peak bench.py's load_peaks() returns), and the device time per kernel of one call from torch.profiler (a
separate pass).  The largest difference between the curve's relative errors and greedy_removal's is recorded as a parity check.  The
card's name, power limit and maximum SM clock are read in the same run.  One JSON object is printed (and written to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import load_peaks  # noqa: E402
from desmo_b200.sparsify import greedy_removal, pruning_profile, removal_order  # noqa: E402
from tools.profile_time import make_engines, smi, timed  # noqa: E402


def kernel_breakdown(e, order):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e.pruning_profile(order)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t and ev.count:
            name = ev.key
            for short in ("library_planes_kernel", "w_planes_kernel", "term_table_kernel", "prune_a_kernel", "prune_b_kernel",
                          "prune_snapshots_kernel", "gemm_planes_kernel", "build_w_kernel", "Memset"):
                if short in name:
                    name = short
            out[name] = {"ms": round(t / 1000.0, 4), "launches": ev.count}
    return out


def run_shape(label, n, m, r, p, dev, reps, rounds, hbm_gbs, clk_mhz, sms):
    eng = make_engines(n, m, r, p, dev)
    e0 = next(iter(eng.values()))
    order = removal_order(e0.term_norms(), e0.T, e0.r)
    S = len(order)
    models = {dt: types.SimpleNamespace(engine=e) for dt, e in eng.items()}
    x2 = {dt: float(e.pruning_profile([])["snapshot_norm2"].sum()) for dt, e in eng.items()}
    for e in eng.values():  # warm-up: first launches, the allocator's pool for the scratch
        for _ in range(2):
            e.pruning_profile(order)
            e.residual_profile()
        e.residual_norm2()
    torch.cuda.synchronize()
    res = {}
    for rnd in range(rounds):
        for dt in ((torch.float32, torch.bfloat16) if rnd % 2 == 0 else (torch.bfloat16, torch.float32)):
            key = str(dt).replace("torch.", "")
            out = res.setdefault(key, {"pruning_profile_ms": [], "residual_profile_ms": [], "greedy_removal_ms": []})
            e = eng[dt]
            out["pruning_profile_ms"].append(round(timed(lambda: e.pruning_profile(order), reps), 3))
            out["residual_profile_ms"].append(round(timed(e.residual_profile, reps), 3))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            greedy = greedy_removal(models[dt], x2[dt])
            torch.cuda.synchronize()
            out["greedy_removal_ms"].append(round((time.perf_counter() - t0) * 1e3, 1))
    for dt, e in eng.items():
        key = str(dt).replace("torch.", "")
        out = res[key]
        pp = pruning_profile(models[dt], order=order, snapshot_norm2=x2[dt])
        greedy = greedy_removal(models[dt], x2[dt])
        out["max_abs_relative_error_diff_vs_greedy"] = max(abs(a - g[1]) for a, g in zip(pp.relative_error, greedy))
        out["nonzero_terms_equal_greedy"] = pp.nonzero_terms == [g[2] for g in greedy]
        best = min(out["pruning_profile_ms"])
        out["speedup_vs_greedy_removal"] = round(min(out["greedy_removal_ms"]) / best, 1)
        out["ratio_to_residual_profile"] = round(best / min(out["residual_profile_ms"]), 3)
        ffma = 2.0 * (S + 1) * n * m
        out["ffma"] = ffma
        out["ffma_floor_ms"] = round(ffma / (sms * 128 * clk_mhz * 1e6) * 1e3, 3)
        ubytes = (2 if dt == torch.bfloat16 else 4) * n * m
        out["u_read_floor_ms"] = round(ubytes / hbm_gbs / 1e6, 3)
        out["kernels"] = kernel_breakdown(e, order)
    a, b = eng[torch.bfloat16].pruning_profile(order), eng[torch.float32].pruning_profile(order)
    parity = all(torch.equal(a[k], b[k]) for k in a)
    del eng, models
    torch.cuda.empty_cache()
    return {"shape": label, "n": n, "m": m, "r": r, "p": p, "steps": S, "bitwise_bf16_vs_fp32_of_uq": parity, "storages": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pruning_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    name, plim, clk = smi("name,power.limit,clocks.max.sm")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    hbm_gbs, _, _, peak_src = load_peaks()
    shapes = [run_shape("headline r4p2", 3 << 20, 1000, 4, 2, dev, a.reps, a.rounds, hbm_gbs, float(clk), sms),
              run_shape("channel-32modes", 262144, 1000, 32, 2, dev, a.reps, a.rounds, hbm_gbs, float(clk), sms)]
    rep = {"card": name, "power_limit_w": float(plim), "max_sm_clock_mhz": float(clk), "sms": sms, "hbm_peak_gbs": hbm_gbs,
           "hbm_peak_source": peak_src, "shapes": shapes}
    txt = json.dumps(rep, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
