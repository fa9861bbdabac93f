"""Evaluation at chosen instants against the whole-matrix residual profile, in ONE process, at the headline shape (r = 4, p = 2) and the
channel "32 modes" shape (r = 32, p = 2, K = 657).

    python tools/eval_at_time.py [--n 3145728] [--m 1000] [--reps 20] [--rounds 3] [--out FILE]

Per shape (CUDA events after warm-up, ms per call and per snapshot):
  - reconstruct_at(index=...) for m' = 1, 16 and 128 (it does not read U, so fp32 storage only);
  - residual_profile_at on a held-out block of m' = 200 snapshots (every 5th index), fp32 and bf16 storage; the block is on the
    device in the storage's dtype, and for bf16 storage also in fp32 (which adds the chunked conversion);
  - residual_profile() on the resident m x n training matrix of the same engine.
The engines and data are tools/profile_time.py's.  The card's name and power limit are read in the same run.  One JSON object is
printed (and written to --out)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from profile_time import make_engines, smi, timed  # noqa: E402

HELD_OUT = 200


def run_shape(label, n, m, r, p, dev, reps, rounds):
    eng = make_engines(n, m, r, p, dev)
    ef, eb = eng[torch.float32], eng[torch.bfloat16]
    idx = list(range(0, m, m // HELD_OUT))[:HELD_OUT]
    block32 = ef.U[idx, :n].clone()  # stands in for held-out data: only the cost is measured here
    block16 = eb.U[idx, :n].clone()
    calls = {}
    for mp in (1, 16, 128):
        k = list(range(0, m, max(1, m // mp)))[:mp]
        calls[f"reconstruct_at m'={mp}"] = (mp, lambda k=k: ef.reconstruct_at(index=k))
    calls["residual_profile_at m'=200 float32"] = (HELD_OUT, lambda: ef.residual_profile_at(block32, index=idx))
    calls["residual_profile_at m'=200 bfloat16"] = (HELD_OUT, lambda: eb.residual_profile_at(block16, index=idx))
    calls["residual_profile_at m'=200 bfloat16 (fp32 block)"] = (HELD_OUT, lambda: eb.residual_profile_at(block32, index=idx))
    calls[f"residual_profile m={m} float32"] = (m, ef.residual_profile)
    calls[f"residual_profile m={m} bfloat16"] = (m, eb.residual_profile)
    for _, fn in calls.values():  # warm-up: first launches and the allocator's pool for every size
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    ms = {key: [] for key in calls}
    names = list(calls)
    for rnd in range(rounds):
        for key in (names if rnd % 2 == 0 else names[::-1]):
            ms[key].append(round(timed(calls[key][1], reps), 4))
    out = {}
    for key, (count, _) in calls.items():
        best = min(ms[key])
        out[key] = {"snapshots": count, "ms": ms[key], "ms_best": best, "ms_per_snapshot": round(best / count, 5)}
    for dt in ("float32", "bfloat16"):
        full = out[f"residual_profile m={m} {dt}"]["ms_best"]
        held = out[f"residual_profile_at m'=200 {dt}"]["ms_best"]
        out[f"residual_profile_at m'=200 {dt}"]["share_of_full_profile"] = round(held / full, 4)
        out[f"residual_profile_at m'=200 {dt}"]["m_prime_over_m"] = round(HELD_OUT / m, 4)
    del eng, ef, eb, block32, block16, calls
    torch.cuda.empty_cache()
    return {"shape": label, "n": n, "m": m, "r": r, "p": p, "calls": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=3 << 20)
    ap.add_argument("--m", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_at_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    name, plim = smi("name,power.limit")
    shapes = [run_shape("headline r4p2", a.n, a.m, 4, 2, dev, a.reps, a.rounds),
              run_shape("channel-32modes", a.n, a.m, 32, 2, dev, max(3, a.reps // 4), a.rounds)]
    rep = {"card": name, "power_limit_w": float(plim), "shapes": shapes}
    txt = json.dumps(rep, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()
