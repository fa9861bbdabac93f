"""Worker of tests/test_pruning_profile.py::test_sharded_profile_matches_unsharded (one process per GPU under torchrun): the pruning
profile of a point-sharded engine against the profile of the whole mesh on one GPU."""
import copy
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desmo_b200 import DesmoEngine  # noqa: E402
from desmo_b200.dist import shard_bounds  # noqa: E402
from desmo_b200.sparsify import removal_order  # noqa: E402
from tests.helpers import load_engine, make_case  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n, m, r, p = 5000, 300, 8, 3
    _, modes, snap, prm = make_case("cylinder", n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    full = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev)
    load_engine(full, prm, modes, snap)
    order = removal_order(full.term_norms(), full.T, full.r)
    whole = full.pruning_profile(order)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, omega_init=10.0, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    sharded = e.pruning_profile(order)
    torch.cuda.synchronize()
    res = sharded["snapshot_residual2"].contiguous()
    gathered = [torch.zeros_like(res) for _ in range(world)]
    dist.all_gather(gathered, res)
    if rank == 0:
        ref = whole["snapshot_residual2"]
        rn = (sharded["snapshot_norm2"] - whole["snapshot_norm2"]).abs() / whole["snapshot_norm2"]
        out = {
            "rel_vs_unsharded": max(float(((res - ref).abs() / ref.clamp_min(1e-300)).max()), float(rn.max())),
            "identical_across_ranks": all(torch.equal(gathered[0], g) for g in gathered),
        }
        print("PRUNING_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
