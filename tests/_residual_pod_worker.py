"""Worker of tests/test_residual_pod.py::test_sharded_residual_pod_matches_unsharded (one process per GPU under torchrun): the residual
POD of a point-sharded engine against the residual POD of the whole mesh on one GPU."""
import copy
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desmo_b200 import DesmoEngine  # noqa: E402
from desmo_b200.dist import shard_bounds  # noqa: E402
from tests.helpers import load_engine, make_case  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n, m, r, p = 60000, 300, 8, 3  # K = 189: chunks of 24 960 points, so every rank and the whole mesh run several, the last one short
    _, modes, snap, prm = make_case("cylinder", n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, omega_init=10.0, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    sharded = e.residual_pod(4)
    full = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev)
    load_engine(full, prm, modes, snap)
    whole = full.residual_pod(4)
    torch.cuda.synchronize()
    grams = [torch.zeros_like(sharded["gram"]) for _ in range(world)]
    dist.all_gather(grams, sharded["gram"].contiguous())
    slabs = [None] * world
    dist.all_gather_object(slabs, (lo, hi, sharded["spatial_modes"].cpu()))
    if rank == 0:
        slabs.sort(key=lambda s: s[0])
        psi = torch.cat([s[2] for s in slabs], dim=1)
        ref = whole["spatial_modes"].cpu()
        sg = torch.sign((psi * ref).sum(1, keepdim=True))
        tr = whole["residual_norm2"]
        out = {
            "gram_rel_vs_unsharded": float((sharded["gram"] - whole["gram"]).abs().max() / whole["gram"].abs().max()),
            "sv2_err_over_trace": float((sharded["singular_values"] ** 2 - whole["singular_values"] ** 2).abs().max() / tr),
            "identical_across_ranks": all(torch.equal(grams[0], g) for g in grams),
            "slab_rel_vs_unsharded": float((psi - sg * ref).norm() / ref.norm()),
        }
        print("RPOD_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
