"""Worker of tests/test_active_terms.py::test_sharded_masked_step_matches_unsharded (one process per GPU under torchrun): masked
point-sharded steps against the same steps of the whole mesh on one GPU, and the check that diverging masks raise."""
import copy
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from desmo_b200 import DesmoEngine  # noqa: E402
from desmo_b200._lib import DesmoError  # noqa: E402
from desmo_b200.dist import shard_bounds  # noqa: E402
from tests.helpers import engine_params, load_engine, make_case  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n, m, r, p = 5000, 300, 8, 3
    _, modes, snap, prm = make_case("cylinder", n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    mask = torch.from_numpy(np.random.default_rng(7).random(prm.K) < 0.3)
    mask[0] = True
    full = DesmoEngine(n, m, p, r, omega_init=10.0, device=dev)
    load_engine(full, prm, modes, snap)
    full.set_active_terms(mask)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, omega_init=10.0, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    mismatch = False
    try:
        e.set_active_terms(mask if rank == 0 else ~mask | (torch.arange(prm.K) == 0))
    except DesmoError:
        mismatch = True
    e.set_active_terms(mask)
    for _ in range(5):
        full.train_step()
        e.train_step()
    torch.cuda.synchronize()
    mine, whole = engine_params(e), engine_params(full)
    worst = 0.0
    for k in ("gates", "omega", "zall"):
        a, b = torch.from_numpy(mine[k]).double(), torch.from_numpy(whole[k]).double()
        worst = max(worst, float((a - b).norm() / b.norm().clamp_min(1e-300)))
    phi_ref = torch.from_numpy(whole["phi"][:, lo:hi]).double()
    worst = max(worst, float((torch.from_numpy(mine["phi"]).double() - phi_ref).norm() / phi_ref.norm()))
    rep = torch.cat([e.gates, e.gates_m, e.gates_u, e.omega, e.omega_m, e.omega_u, e.rows.reshape(-1), e.rows_m.reshape(-1)])
    gathered = [torch.zeros_like(rep) for _ in range(world)]
    dist.all_gather(gathered, rep)
    if rank == 0:
        out = {"rel_vs_unsharded": worst, "identical_across_ranks": all(torch.equal(gathered[0], g) for g in gathered),
               "mismatch_raised": mismatch}
        print("ACTIVE_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
