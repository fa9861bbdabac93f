"""fp32 vs bf16 storage of the snapshot matrix U at a headline shape, in ONE process with the two storages alternated.

    python tools/bf16_time.py [--n 3145728] [--m 1000] [--steps 20] [--sustained 300] [--out FILE]

Reports, per storage: step time over graph-replayed DesmoTrainer steps, the per-launch series of the dominant kernel
(desmo_fused_kernel_ms_series, eager steps), a sustained region of back-to-back graph replays with SM clock / board power sampled by
read-only nvidia-smi queries, the POD Gram time, the algorithmic bytes of a step (U + phi/P/dphi + W/E: 4nm or 2nm, + 12nr + 8Km), their
share of the device-to-device copy bandwidth measured in the same run, and the largest n one GPU holds (from buffer sizes, not
allocated).  Also the bitwise parity of one step between bf16 storage and fp32 storage of U_q.float().  One JSON object is printed
(and written to --out); the card name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

os.environ.setdefault("DESMO_KERNEL_EVENTS", "1")
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from desmo_b200 import DesmoEngine, DesmoTrainer  # noqa: E402


def smi(fields):
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, timeout=20)
    return [v.strip() for v in out.stdout.strip().split(",")]


class Sampler(threading.Thread):
    def __init__(self):
        super().__init__(daemon=True)
        self.samples, self.stop = [], threading.Event()

    def run(self):
        while not self.stop.is_set():
            try:
                c, p = smi("clocks.sm,power.draw")
                self.samples.append((float(c), float(p)))
            except Exception:  # noqa: BLE001  (a missed sample is not a measurement error)
                pass
            time.sleep(0.1)


def hbm_copy_gbs(nbytes=8 << 30, reps=10):
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del a, b
    return 2 * nbytes / ms / 1e6  # read + write


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3 << 20)
    ap.add_argument("--m", type=int, default=1000)
    ap.add_argument("--r", type=int, default=4)
    ap.add_argument("--p", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--sustained", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    name, plim, maxclk = smi("name,power.limit,clocks.max.sm")
    n, m, r = a.n, a.m, a.r
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.linspace(0, 1, n, device=dev)
    P = torch.stack([torch.sin(3.1416 * (k + 1) * x + 0.3 * k) for k in range(r)]) * (2.0 / n) ** 0.5
    eng = {}
    for dt in (torch.bfloat16, torch.float32):
        e = DesmoEngine(n, m, a.p, r, omega_init=10.0, device=dev, snapshot_dtype=dt)
        e.P[:, :n] = P
        e.rows[:, :m] = 1.0
        eng[dt] = e
    K, Kp = eng[torch.float32].K, eng[torch.float32].Kp
    # snapshot: built once in fp32 on the device in slices of time; bf16 engine converts it, fp32 engine gets U_q.float()
    for t0 in range(0, m, 100):
        t = torch.linspace(0, 1, m, device=dev)[t0:t0 + 100]
        Us = sum(torch.cos(6.2832 * (k + 1) * t + k)[:, None] * torch.sin(3.1416 * (k + 1) * x + 0.3 * k)[None, :] / (k + 1) for k in range(5))
        Us = Us + 0.02 * torch.randn(Us.shape, device=dev, generator=g)
        eb = eng[torch.bfloat16]
        eb.U = eb.U if eb.U is not None else torch.zeros(m, eb.ld, dtype=torch.bfloat16, device=dev)
        ef = eng[torch.float32]
        ef.U = ef.U if ef.U is not None else torch.zeros(m, ef.ld, dtype=torch.float32, device=dev)
        src = Us.contiguous()
        eb.lib.desmo_snapshot_to_bf16(C.byref(eb.shape), src.data_ptr(), src.stride(0), t0, src.shape[0], eb.U.data_ptr(), None,
                                      torch.cuda.current_stream().cuda_stream)
        ef.U[t0:t0 + src.shape[0], :n] = src.bfloat16().float()
        del Us, src
    torch.cuda.synchronize()
    # bitwise parity of one step
    for e in eng.values():
        e.build_w(False)
        e.fused_residual_grad()
    torch.cuda.synchronize()
    ea, eb_ = eng[torch.bfloat16], eng[torch.float32]
    parity = bool(torch.equal(ea.red, eb_.red) and torch.equal(ea.dphi, eb_.dphi))
    peak = hbm_copy_gbs()
    trainers = {dt: DesmoTrainer(e, lrs=(1e-2, 1e-3, 1e-2, 1e-2), beta=1e-3, l1_lambda=1e-4, use_cuda_graph=True) for dt, e in eng.items()}
    lib = ea.lib
    res = {str(dt).replace("torch.", ""): {"step_ms": [], "kernel_ms_series": [], "sustained_step_ms": [], "sustained_clock_mhz": [],
                                           "sustained_power_w": [], "gram_ms": []} for dt in eng}
    for dt, tr in trainers.items():  # warm-up: graph capture and first launches
        for _ in range(5):
            tr.step()
    torch.cuda.synchronize()
    for rnd in range(a.rounds):
        for dt in ((torch.float32, torch.bfloat16) if rnd % 2 == 0 else (torch.bfloat16, torch.float32)):
            e, tr, out = eng[dt], trainers[dt], res[str(dt).replace("torch.", "")]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.steps):
                tr.step()
            e1.record()
            torch.cuda.synchronize()
            out["step_ms"].append(e0.elapsed_time(e1) / a.steps)
            # per-launch kernel series over eager steps
            mean, cnt = C.c_float(0), C.c_int32(0)
            lib.desmo_fused_kernel_ms_mean(C.byref(mean), C.byref(cnt), 1)
            for _ in range(a.steps):
                e.train_step()
            buf = (C.c_float * 64)()
            lib.desmo_fused_kernel_ms_series(buf, 64, C.byref(cnt))
            out["kernel_ms_series"].append([round(float(buf[i]), 4) for i in range(cnt.value)])
            # sustained region
            smp = Sampler()
            smp.start()
            e0.record()
            for _ in range(a.sustained):
                tr.step()
            e1.record()
            torch.cuda.synchronize()
            smp.stop.set()
            smp.join()
            out["sustained_step_ms"].append(e0.elapsed_time(e1) / a.sustained)
            tail = smp.samples[len(smp.samples) // 2:] or smp.samples
            out["sustained_clock_mhz"].append(sum(s[0] for s in tail) / max(1, len(tail)))
            out["sustained_power_w"].append(sum(s[1] for s in tail) / max(1, len(tail)))
            e.pod_from_snapshot()
            out["gram_ms"].append(e.pod_timing["gram_ms"])
    alg = {"float32": 4 * n * m + 12 * n * r + 8 * K * m, "bfloat16": 2 * n * m + 12 * n * r + 8 * K * m}
    gib = torch.cuda.get_device_properties(dev).total_memory
    for key, out in res.items():
        e = eng[torch.bfloat16 if key == "bfloat16" else torch.float32]
        kern = sorted(v for s in out["kernel_ms_series"] for v in s)
        kmed = kern[len(kern) // 2] if kern else float("nan")
        out["kernel_ms_median"] = kmed
        out["algorithmic_bytes"] = alg[key]
        out["algorithmic_gbs_at_median_kernel"] = alg[key] / kmed / 1e6
        out["share_of_measured_copy_bw"] = alg[key] / kmed / 1e6 / peak
        # largest n per GPU: U + 5 [r][ld] fp32 parameter / moment / gradient rows + the workspace's per-point part
        ws = []
        for nn in (1 << 20, 2 << 20):
            from desmo_b200._lib import make_shape
            s = make_shape(nn, m, r, a.p)
            b = C.c_size_t(0)
            e.lib.desmo_workspace_bytes(C.byref(s), C.byref(b))
            ws.append(b.value)
        per_point = (2 if key == "bfloat16" else 4) * m + 5 * 4 * r + (ws[1] - ws[0]) / (1 << 20)
        fixed = ws[0] - (ws[1] - ws[0]) + 4 * (3 * K * e.mld + Kp * e.mld)
        out["max_n_per_gpu"] = int((0.95 * gib - fixed) / per_point)
    rep = {"card": name, "power_limit_w": float(plim), "max_sm_clock_mhz": float(maxclk), "n": n, "m": m, "K": K,
           "measured_copy_gbs": peak, "bitwise_parity_one_step": parity, "storages": res}
    txt = json.dumps(rep, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
