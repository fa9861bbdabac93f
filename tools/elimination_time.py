"""Backward elimination (sparsify.backward_elimination) against the norm order's sparsify.pruning_profile() and greedy_removal(), fp32
and bf16 storage of U in ONE process, at the headline shape (3 * 2^20 x 1000, r = 4, p = 2, K = 27) and the channel "32 modes" shape
(262144 x 1000, r = 32, p = 2, K = 657).

    python tools/elimination_time.py [--rounds 3] [--out FILE]

Per storage and shape: whole backward_elimination() and pruning_profile() calls by a host clock around each call ending in a device
synchronise, alternated round by round, median over --rounds; the split of one call into the pass (build_w + desmo_elimination_pass),
the greedy (desmo_elimination_greedy, one launch per step) and the exact profile of the chosen order (DesmoEngine.pruning_profile) by
CUDA events, median; greedy_removal() once; the scratch bytes.  The card's name, power limit and maximum SM clock are read in the same
run.  One JSON object is printed (and written to --out)."""
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

from desmo_b200 import sparsify  # noqa: E402
from desmo_b200._lib import check  # noqa: E402
from tools.profile_time import make_engines, smi  # noqa: E402


class _Model:
    def __init__(self, e):
        self.engine = e


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def split_ms(e):
    """Event-timed pass, greedy and exact profile of one backward elimination (the engine's sequence, without its host reads)."""
    f64 = dict(dtype=torch.float64, device=e.device)
    scratch = e._elimination_scratch()
    A, F, r2 = torch.empty(e.K, e.K, **f64), torch.empty(e.K, e.mld, **f64), torch.empty(1, **f64)
    order, pred = torch.empty(e.K, dtype=torch.int32, device=e.device), torch.empty(e.K + 1, **f64)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    st = torch.cuda.current_stream().cuda_stream
    ev[0].record()
    e.build_w(False)
    check(e.lib.desmo_elimination_pass(C.byref(e.shape), e.U.data_ptr(), e._u_dtype(), e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(),
                                       e.W.data_ptr(), A.data_ptr(), F.data_ptr(), r2.data_ptr(), scratch.data_ptr(), scratch.numel(), st))
    ev[1].record()
    check(e.lib.desmo_elimination_greedy(C.byref(e.shape), A.data_ptr(), F.data_ptr(), r2.data_ptr(), e.W.data_ptr(), e.K, order.data_ptr(),
                                         pred.data_ptr(), scratch.data_ptr(), scratch.numel(), st))
    ev[2].record()
    e.pruning_profile(order.cpu().tolist())
    ev[3].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), scratch.numel()


def run_shape(label, n, m, r, p, dev, rounds):
    eng = make_engines(n, m, r, p, dev)
    res = {}
    for dt, e in eng.items():
        model = _Model(e)
        for _ in range(2):  # warm-up: first launches, allocator pools
            sparsify.backward_elimination(model)
            sparsify.pruning_profile(model)
            split_ms(e)
        key = str(dt).replace("torch.", "")
        out = res.setdefault(key, {})
        times = {"backward_elimination_ms": [], "pruning_profile_ms": []}
        sp = []
        for rnd in range(rounds):
            calls = [("backward_elimination_ms", lambda: sparsify.backward_elimination(model)),
                     ("pruning_profile_ms", lambda: sparsify.pruning_profile(model))]
            for name, fn in (calls if rnd % 2 == 0 else calls[::-1]):
                times[name].append(host_ms(fn))
            sp.append(split_ms(e))
        for name, v in times.items():
            out[name] = round(statistics.median(v), 3)
        out["ratio_to_pruning_profile"] = round(out["backward_elimination_ms"] / out["pruning_profile_ms"], 3)
        out["split_ms"] = {"pass": round(statistics.median(x[0] for x in sp), 3), "greedy": round(statistics.median(x[1] for x in sp), 3),
                           "exact_profile": round(statistics.median(x[2] for x in sp), 3)}
        out["greedy_us_per_step"] = round(1e3 * out["split_ms"]["greedy"] / e.K, 2)
        out["scratch_bytes"] = sp[0][3]
        snorm = float(sparsify.pruning_profile(model).snapshot_norm2.sum())
        out["greedy_removal_ms"] = round(host_ms(lambda: sparsify.greedy_removal(model, snorm)), 1)
        be, pp = sparsify.backward_elimination(model), sparsify.pruning_profile(model)
        out["relative_error_by_error_order"] = [round(v, 6) for v in be.relative_error[::max(1, e.K // 8)]]
        out["relative_error_by_norm_order"] = [round(v, 6) for v in pp.relative_error[::max(1, e.K // 8)]]
    a, b = eng[torch.bfloat16].backward_elimination(), eng[torch.float32].backward_elimination()
    parity = all(torch.equal(a[k], b[k]) for k in ("order", "predicted_residual2", "gram"))
    del eng
    torch.cuda.empty_cache()
    return {"shape": label, "n": n, "m": m, "r": r, "p": p, "bitwise_bf16_vs_fp32_of_uq": parity, "storages": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("elimination_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    name, plim, clk = smi("name,power.limit,clocks.max.sm")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    shapes = [run_shape("headline r4p2", 3 << 20, 1000, 4, 2, dev, a.rounds),
              run_shape("channel-32modes", 262144, 1000, 32, 2, dev, a.rounds)]
    rep = {"card": name, "power_limit_w": float(plim), "max_sm_clock_mhz": float(clk), "sms": sms, "shapes": shapes}
    txt = json.dumps(rep, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
