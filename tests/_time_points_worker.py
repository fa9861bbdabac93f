"""Worker of tests/test_time_points.py::test_sharded_steps_share_the_table (one process per GPU under torchrun): point-sharded steps of a
Fourier model at a shared time table against the same steps of the whole mesh on one GPU, and the check that diverging tables raise."""
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
    n, m, r, p, nF = 5000, 300, 4, 3, 3
    _, modes, snap, prm = make_case("cylinder", n, m, r, p, nF, period_init=60.0, omega_init=2.0, perturb_rel=0.2)
    t = np.sort(np.random.default_rng(9).uniform(0.0, m, m)).astype(np.float32)
    full = DesmoEngine(n, m, p, r, nF=nF, device=dev, t_points=t)
    load_engine(full, prm, modes, snap)
    lo, hi = shard_bounds(n, world, rank)
    e = DesmoEngine(hi - lo, m, p, r, nF=nF, device=dev, n_global=n, process_group=dist.group.WORLD)
    q = copy.copy(prm)
    q.phi, q.n = prm.phi[:, lo:hi], hi - lo
    load_engine(e, q, modes[lo:hi], snap[:, lo:hi])
    mismatch = False
    try:
        e.set_time_points(t if rank == 0 else t[::-1].copy())
    except DesmoError:
        mismatch = True
    e.set_time_points(t)
    for _ in range(5):
        full.train_step()
        e.train_step()
    torch.cuda.synchronize()
    mine, whole = engine_params(e), engine_params(full)
    worst = 0.0
    for k in ("gates", "omega", "coefs", "periods"):
        a, b = torch.from_numpy(mine[k]).double(), torch.from_numpy(whole[k]).double()
        worst = max(worst, float((a - b).norm() / b.norm().clamp_min(1e-300)))
    phi_ref = torch.from_numpy(whole["phi"][:, lo:hi]).double()
    worst = max(worst, float((torch.from_numpy(mine["phi"]).double() - phi_ref).norm() / phi_ref.norm()))
    rep = torch.cat([e.gates, e.gates_m, e.omega, e.coefs.reshape(-1), e.coefs_m.reshape(-1), e.periods, e.periods_u, e._times])
    gathered = [torch.zeros_like(rep) for _ in range(world)]
    dist.all_gather(gathered, rep)
    if rank == 0:
        out = {"rel_vs_unsharded": worst, "identical_across_ranks": all(torch.equal(gathered[0], g) for g in gathered),
               "mismatch_raised": mismatch}
        print("TIMES_RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
