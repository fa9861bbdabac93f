"""Worker of tests/test_pod_analysis.py::test_sharded_pod_analysis_matches_unsharded (one process per GPU under torchrun): pod_analysis()
of a point-sharded engine (slab Grams, one all-reduce, replicated solve) against that of the whole mesh on one GPU."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desmo_b200 import DesmoEngine  # noqa: E402
from desmo_b200.dist import shard_bounds  # noqa: E402
from oracle import desmo_oracle as orc  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n, m, r = 4096, 240, 32
    X = orc.synthetic_snapshots("channel", n, m, 0)
    snap = torch.as_tensor(np.ascontiguousarray(X.T), dtype=torch.float32)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, 2, r, 10.0, device=dev, n_global=n, process_group=dist.group.WORLD)
    e.set_snapshot(snap[:, lo:hi].contiguous())
    sigma = e.pod_analysis()
    full = DesmoEngine(n, m, 2, r, 10.0, device=dev)
    full.set_snapshot(snap)
    full.pod_analysis()
    torch.cuda.synchronize()
    Vs = [torch.zeros_like(e.pod_V) for _ in range(world)]
    ss = [torch.zeros_like(sigma) for _ in range(world)]
    dist.all_gather(Vs, e.pod_V)
    dist.all_gather(ss, sigma)
    slabs = [None] * world
    dist.all_gather_object(slabs, (lo, hi, e.P[:, :hi - lo].double().cpu()))
    if rank == 0:
        slabs.sort(key=lambda s: s[0])
        P = torch.cat([s[2] for s in slabs], dim=1)
        Pf = full.P[:, :n].double().cpu()
        live = (full.pod_singular_values[:r] > 0).numpy()
        Pn, Fn = P / P.norm(dim=1, keepdim=True).clamp_min(1e-300), Pf / Pf.norm(dim=1, keepdim=True).clamp_min(1e-300)
        sin = [float(torch.sqrt(torch.clamp(1 - (Pn[i] @ Fn[i]) ** 2, min=0.0))) for i in np.flatnonzero(live)]
        out = {
            "V_identical_across_ranks": all(torch.equal(Vs[0], v) for v in Vs),
            "sigma_identical_across_ranks": all(torch.equal(ss[0], s) for s in ss),
            "mode_sin_vs_unsharded": max(sin[:8]) if sin else 0.0,
        }
        print("POD_ANALYSIS_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
