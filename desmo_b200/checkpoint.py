"""Checkpoints of point-sharded runs (SURVEY.md 8 f3): a multi-GPU run writes ONE file in the reference's key layout and resumes at any
world size.

The reference saves ``model.state_dict()`` only (CYL:781-786,802-805).  A sharded run holds ``phi_list[i]`` (and its Adamax moments, and
the POD modes) as per-rank slabs of mesh points; everything else is replicated.  ``gather_trainer_state`` assembles the full vectors on
rank 0 (``torch.distributed.gather`` of padded slabs), so that ``checkpoint["model"]`` is exactly the reference's ``state_dict`` for the
whole mesh -- loadable by the reference scripts -- and ``scatter_trainer_state`` cuts the slab of (rank, world) out of it again,
for any world size.  The active-term mask (``active_terms``, DesmoEngine.set_active_terms) is replicated and passes through as it is.
Works on any tensor device (the gloo tests run it on CPU tensors with a stand-in engine).
"""
from __future__ import annotations

from typing import Optional

import torch

from .dist import shard_bounds

_SLAB_KEYS = ("phi", "phi_m", "phi_u", "P")  # [r][ld] buffers whose first n columns are this rank's mesh points


def _dist_info(group=None):
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def _gather_rows(local: torch.Tensor, n_global: int, group=None) -> Optional[torch.Tensor]:
    """[r][n_local] slabs of every rank -> [r][n_global] on rank 0 (None elsewhere); slabs follow shard_bounds."""
    import torch.distributed as dist

    rank, world = _dist_info(group)
    if world == 1:
        return local.clone()
    width = max(shard_bounds(n_global, world, q)[1] - shard_bounds(n_global, world, q)[0] for q in range(world))
    pad = torch.zeros(local.shape[0], width, dtype=local.dtype, device=local.device)
    pad[:, :local.shape[1]] = local
    bufs = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, bufs, dst=0, group=group)
    if rank != 0:
        return None
    out = torch.empty(local.shape[0], n_global, dtype=local.dtype, device=local.device)
    for q in range(world):
        lo, hi = shard_bounds(n_global, world, q)
        out[:, lo:hi] = bufs[q][:, :hi - lo]
    return out


def gather_trainer_state(trainer, group=None) -> Optional[dict]:
    """The full-mesh checkpoint dictionary on rank 0 (None on the other ranks): reference-layout ``model`` state_dict, Adamax moments,
    step counter, scheduler, POD modes -- the same keys as ``DesmoTrainer.state_dict()`` of an unsharded run."""
    e = trainer.engine
    rank, world = _dist_info(group)
    lo, hi = shard_bounds(e.n_global, world, rank)
    if hi - lo != e.n:
        raise ValueError(f"rank {rank}: engine owns {e.n} points but shard_bounds gives {hi - lo}: slabs must follow desmo_b200.dist.shard_bounds")
    full = {k: _gather_rows(getattr(e, k)[:, :e.n].detach(), e.n_global, group) for k in _SLAB_KEYS}
    if rank != 0:
        return None
    sd = trainer.state_dict()  # local view: replicated entries are already global
    model = dict(sd["model"]) if sd["model"] is not None else {}
    for i in range(e.r):
        model[f"phi_list.{i}"] = full["phi"][i].clone()
    sd["model"] = {k: model[k] for k in (sd["model"].keys() if sd["model"] is not None else model.keys())}
    sd["optimizer"]["phi_m"], sd["optimizer"]["phi_u"] = full["phi_m"], full["phi_u"]
    sd["pod_modes"] = full["P"]
    sd["shape"] = dict(sd["shape"], n=e.n_global, n_global=e.n_global, saved_world_size=world)
    return sd


def save_checkpoint(trainer, path: str, group=None) -> None:
    """Collective: every rank calls it, rank 0 writes the single file."""
    sd = gather_trainer_state(trainer, group)
    if sd is not None:
        torch.save(sd, path)
    if _dist_info(group)[1] > 1:
        import torch.distributed as dist

        dist.barrier(group)


def scatter_trainer_state(sd: dict, rank: int, world: int) -> dict:
    """Cuts the slab of (rank, world) out of a full-mesh checkpoint: the dictionary ``DesmoTrainer.load_state_dict`` of that rank takes."""
    n_global = int(sd["shape"]["n_global"])
    if int(sd["shape"]["n"]) != n_global:
        raise ValueError("not a full-mesh checkpoint (save it with desmo_b200.checkpoint.save_checkpoint)")
    lo, hi = shard_bounds(n_global, world, rank)
    out = dict(sd)
    r = int(sd["shape"]["r"])
    if sd.get("model") is not None:
        out["model"] = {k: (v[lo:hi].clone() if k.startswith("phi_list.") else v) for k, v in sd["model"].items()}
    out["optimizer"] = dict(sd["optimizer"])
    for k in ("phi_m", "phi_u"):
        out["optimizer"][k] = sd["optimizer"][k][:, lo:hi]
    out["pod_modes"] = sd["pod_modes"][:, lo:hi]
    out["shape"] = dict(sd["shape"], n=hi - lo, n_global=n_global)
    assert len([k for k in (out["model"] or {}) if k.startswith("phi_list.")]) in (0, r)
    return out


def load_checkpoint(trainer, path_or_dict, group=None, map_location=None) -> None:
    """Every rank loads the single file and keeps its own slab; the world size may differ from the run that saved it."""
    sd = path_or_dict if isinstance(path_or_dict, dict) else torch.load(path_or_dict, map_location=map_location or "cpu", weights_only=False)
    rank, world = _dist_info(group)
    trainer.load_state_dict(scatter_trainer_state(sd, rank, world))
