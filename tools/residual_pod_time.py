"""Residual POD (DesmoEngine.residual_pod) against pod_analysis() and residual_profile(), fp32 and bf16 storage of U in ONE process, at
the headline shape (3 * 2^20 x 1000, r = 4, p = 2, K = 27) and the channel "32 modes" shape (262144 x 1000, r = 32, p = 2, K = 657),
for k = 8 and k = 32 residual modes.

    python tools/residual_pod_time.py [--rounds 5] [--out FILE]

Per storage, shape and k: the split of one call into the Gram pass (build_w + desmo_residual_gram), the eigensolve (desmo_pod_eigh) and
the modes pass (desmo_residual_modes) by CUDA events, median over --rounds; whole residual_pod(k), pod_analysis() and residual_profile()
calls by a host clock around each call ending in a device synchronise, alternated round by round, median; the scratch bytes; the Gram
GEMM's tensor-core floor (3 products of 2 mp^2 n / 2 flop over the upper tiles, (T + 1) / 2T of the square, at the bf16 dense peak
bench.py's load_peaks() returns) and U's read floor.  P is restored after each pod_analysis() call, so every residual_pod() call sees
the same model.  The card's name, power limit and maximum SM clock are read in the same run.  One JSON object is printed (and written
to --out)."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import load_peaks  # noqa: E402
from desmo_b200._lib import check  # noqa: E402
from tools.profile_time import make_engines, smi  # noqa: E402


def split_ms(e, k):
    """Event-timed Gram pass, eigensolve and modes pass of one residual POD (the engine's sequence, without its host reads)."""
    f32 = dict(dtype=torch.float32, device=e.device)
    scratch = e._residual_pod_scratch()
    Cm, tr = torch.empty(e.m, e.m, **f32), torch.empty(1, dtype=torch.float64, device=e.device)
    V, sigma, modes = torch.zeros(k, e.m, **f32), torch.zeros(k, **f32), torch.zeros(k, e.ld, **f32)
    S = torch.zeros(e.m, dtype=torch.float64, device=e.device)
    nb = C.c_size_t(0)
    check(e.lib.desmo_pod_eigh_workspace_bytes(e.m, k, C.byref(nb)))
    ws = torch.empty(nb.value, dtype=torch.uint8, device=e.device)
    st = torch.cuda.current_stream().cuda_stream
    args = (C.byref(e.shape), e.U.data_ptr(), e._u_dtype(), e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(), e.W.data_ptr())
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    torch.cuda.synchronize()
    ev[0].record()
    e.build_w(False)
    check(e.lib.desmo_residual_gram(*args, Cm.data_ptr(), tr.data_ptr(), scratch.data_ptr(), scratch.numel(), st))
    ev[1].record()
    check(e.lib.desmo_pod_eigh(e.m, k, Cm.data_ptr(), S.data_ptr(), V.data_ptr(), sigma.data_ptr(), ws.data_ptr(), ws.numel(), st))
    ev[2].record()
    check(e.lib.desmo_residual_modes(*args, k, V.data_ptr(), sigma.data_ptr(), modes.data_ptr(), scratch.data_ptr(), scratch.numel(), st))
    ev[3].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), scratch.numel()


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def run_shape(label, n, m, r, p, dev, rounds, hbm_gbs, bf16_tflops):
    eng = make_engines(n, m, r, p, dev)
    res = {}
    for dt, e in eng.items():
        P0 = e.P.clone()

        def pod(e=e, P0=P0):
            e.pod_analysis()
            e.P.copy_(P0)

        for _ in range(2):  # warm-up: first launches, allocator pools
            pod()
            e.residual_profile()
            for k in (8, 32):
                e.residual_pod(k)
                split_ms(e, k)
        key = str(dt).replace("torch.", "")
        out = res.setdefault(key, {})
        times = {"pod_analysis_ms": [], "residual_profile_ms": []}
        sp = {}
        for rnd in range(rounds):
            for k in ((8, 32) if rnd % 2 == 0 else (32, 8)):
                times.setdefault(f"residual_pod_k{k}_ms", []).append(host_ms(lambda k=k: e.residual_pod(k)))
                sp.setdefault(k, []).append(split_ms(e, k))
            times["pod_analysis_ms"].append(host_ms(pod))
            times["residual_profile_ms"].append(host_ms(e.residual_profile))
        for name, v in times.items():
            out[name] = round(statistics.median(v), 3)
        for k, v in sp.items():
            out[f"k{k}_split_ms"] = {"gram": round(statistics.median(x[0] for x in v), 3), "eigh": round(statistics.median(x[1] for x in v), 3),
                                     "modes": round(statistics.median(x[2] for x in v), 3)}
            out[f"k{k}_ratio_to_pod_analysis"] = round(out[f"residual_pod_k{k}_ms"] / out["pod_analysis_ms"], 3)
        out["scratch_bytes"] = sp[8][0][3]
        mp = (m + 127) // 128 * 128
        T = mp // 128
        flop = 3 * 2.0 * mp * mp * n * (T + 1) / (2 * T)
        out["gram_gemm_flop"] = flop
        out["gram_tensor_floor_ms"] = round(flop / (bf16_tflops * 1e12) * 1e3, 3)
        out["u_read_floor_ms"] = round((2 if dt == torch.bfloat16 else 4) * n * m / hbm_gbs / 1e6, 3)
    a, b = eng[torch.bfloat16].residual_pod(8), eng[torch.float32].residual_pod(8)
    parity = all(torch.equal(a[k], b[k]) for k in ("singular_values", "sigma", "temporal_modes", "spatial_modes", "gram"))
    del eng
    torch.cuda.empty_cache()
    return {"shape": label, "n": n, "m": m, "r": r, "p": p, "bitwise_bf16_vs_fp32_of_uq": parity, "storages": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("residual_pod_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    name, plim, clk = smi("name,power.limit,clocks.max.sm")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    peaks = load_peaks()
    hbm_gbs, bf16_tflops = peaks[0], peaks[1]
    shapes = [run_shape("headline r4p2", 3 << 20, 1000, 4, 2, dev, a.rounds, hbm_gbs, bf16_tflops),
              run_shape("channel-32modes", 262144, 1000, 32, 2, dev, a.rounds, hbm_gbs, bf16_tflops)]
    rep = {"card": name, "power_limit_w": float(plim), "max_sm_clock_mhz": float(clk), "sms": sms, "hbm_peak_gbs": hbm_gbs,
           "bf16_peak_tflops": bf16_tflops, "peak_source": peaks[3], "shapes": shapes}
    txt = json.dumps(rep, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
