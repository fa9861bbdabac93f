"""Worker of tests/test_backward_elimination.py::test_sharded_order_matches_unsharded (one process per GPU under torchrun): the
backward elimination of a point-sharded engine against the one of the whole mesh on one GPU."""
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
    n, m, r, p = 60000, 300, 8, 3  # K = 189: several chunks of points per rank and for the whole mesh, the last one short
    _, modes, snap, prm = make_case("cylinder", n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, omega_init=10.0, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    sharded = e.backward_elimination()
    full = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev)
    load_engine(full, prm, modes, snap)
    whole = full.backward_elimination()
    torch.cuda.synchronize()
    orders = [None] * world
    dist.all_gather_object(orders, sharded["order"].tolist())
    if rank == 0:
        a, b = sharded["order"].tolist(), whole["order"].tolist()
        prefix = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), len(a))
        pw = whole["predicted_residual2"]
        out = {
            "identical_across_ranks": all(o == orders[0] for o in orders),
            "gram_rel_vs_unsharded": float((sharded["gram"] - whole["gram"]).abs().max() / whole["gram"].abs().max()),
            "same_prefix_as_unsharded": prefix,
            "pred_rel_vs_unsharded": float((sharded["predicted_residual2"][:prefix + 1] - pw[:prefix + 1]).abs().max() / pw[0]),
        }
        print("ELIM_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
