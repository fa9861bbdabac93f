"""Worker of tests/test_eval_at_time.py::test_sharded_held_out_profile_matches_unsharded (one process per GPU under torchrun): the
held-out residual profile and reconstruct_at of a point-sharded Fourier engine against those of the whole mesh on one GPU."""
import copy
import json
import os
import sys

import numpy as np
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
    n, m, r, p, nF = 5000, 300, 8, 3, 3
    X, modes, snap, prm = make_case("cylinder", n, m, r, p, nF=nF, omega_init=10.0, perturb_rel=0.3)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, omega_init=10.0, nF=nF, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    t = e.time_points(np.arange(m, m + 150))
    block = torch.from_numpy(np.ascontiguousarray(snap[::2][:150] * 1.1))  # a held-out block of 150 snapshots
    sharded = e.residual_profile_at(block[:, lo:hi].contiguous(), times=t)
    rec = e.reconstruct_at(times=t)
    full = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF, device=dev)
    load_engine(full, prm, modes, snap)
    whole = full.residual_profile_at(block, times=t)
    rec_full = full.reconstruct_at(times=t)
    torch.cuda.synchronize()
    snaps = [torch.zeros_like(sharded["snapshot_residual2"]) for _ in range(world)]
    dist.all_gather(snaps, sharded["snapshot_residual2"].contiguous())
    slabs = [None] * world
    dist.all_gather_object(slabs, (lo, hi, sharded["point_residual2"].cpu(), sharded["point_norm2"].cpu(), rec.cpu()))
    if rank == 0:
        slabs.sort(key=lambda s: s[0])
        pr = torch.cat([s[2] for s in slabs])
        pn = torch.cat([s[3] for s in slabs])
        rc = torch.cat([s[4] for s in slabs], dim=1)
        ref = whole["snapshot_residual2"]
        out = {
            "snapshot_rel_vs_unsharded": float(((sharded["snapshot_residual2"] - ref).abs() / ref).max()),
            "snapshot_identical_across_ranks": all(torch.equal(snaps[0], s) for s in snaps),
            "point_slabs_bit_identical": bool(torch.equal(pr, whole["point_residual2"].cpu()) and torch.equal(pn, whole["point_norm2"].cpu())),
            "recon_slabs_bit_identical": bool(torch.equal(rc, rec_full.cpu())),
        }
        print("EVAL_AT_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
