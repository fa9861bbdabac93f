"""Worker of tests/test_residual_profile.py::test_sharded_profile_matches_unsharded (one process per GPU under torchrun): the residual
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
from tests.helpers import load_engine, make_case  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n, m, r, p = 5000, 300, 8, 3
    _, modes, snap, prm = make_case("cylinder", n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, omega_init=10.0, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    sharded = e.residual_profile()
    full = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev)
    load_engine(full, prm, modes, snap)
    whole = full.residual_profile()
    torch.cuda.synchronize()
    snaps = [torch.zeros_like(sharded["snapshot_residual2"]) for _ in range(world)]
    dist.all_gather(snaps, sharded["snapshot_residual2"].contiguous())
    slabs = [None] * world
    dist.all_gather_object(slabs, (lo, hi, sharded["point_residual2"].cpu(), sharded["point_norm2"].cpu()))
    if rank == 0:
        slabs.sort(key=lambda s: s[0])
        pr = torch.cat([s[2] for s in slabs])
        pn = torch.cat([s[3] for s in slabs])
        ref = whole["snapshot_residual2"]
        out = {
            "snapshot_rel_vs_unsharded": float(((sharded["snapshot_residual2"] - ref).abs() / ref).max()),
            "snapshot_identical_across_ranks": all(torch.equal(snaps[0], s) for s in snaps),
            "point_slabs_bit_identical": bool(torch.equal(pr, whole["point_residual2"].cpu()) and torch.equal(pn, whole["point_norm2"].cpu())),
        }
        print("PROFILE_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
