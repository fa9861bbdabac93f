"""Post-hoc sparsification (CYL:624-692,1184-1270; TURB:1166-1245): term norms -> threshold sweep -> active mask."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np
import torch

from ._lib import DesmoError


def threshold_sweep(model, snapshot_norm2: float, thresholds=None) -> List[Tuple[float, float, int, torch.Tensor]]:
    """For every threshold: zero the gates whose term norm is below it (CYL:1228-1238), evaluate
    ||X - recon^T|| / ||X|| (CYL:1257) and count the surviving non-zero gates (CYL:1260-1265).
    Returns [(threshold, relative_error, n_active, mask)], restoring the gates afterwards."""
    e = model.engine
    if hasattr(model, "sync_parameters"):
        model.sync_parameters()
    if thresholds is None:
        thresholds = [10.0 ** (-4 + 0.5 * i) for i in range(14)]  # 10^-4 .. 10^2.5, half-decade steps (CYL:1213)
    norms = e.term_norms()  # the reference's semantics (raw phi_list; Fourier column quirk), see DesmoEngine.term_norms
    saved = e.gates.clone()
    out = []
    for thr in thresholds:
        e.gates.copy_(saved)
        mask = (norms >= thr) & (saved != 0)
        e.gates.mul_(mask.to(e.gates.dtype))
        err = (e.residual_norm2() / snapshot_norm2) ** 0.5
        out.append((float(thr), float(err), int(mask.sum().item()), mask.clone()))
    e.gates.copy_(saved)
    return out


def removal_order(norms: torch.Tensor, T: int, r: int) -> List[int]:
    """Packed K indices in the order the reference's sweep removes them: the list is built as the polynomial terms, then
    (sin_i, cos_i, tanh_i) per mode (TURB:1173-1181), and sorted by norm with a stable sort (TURB:1183)."""
    vals = norms.tolist()
    listed = list(range(T)) + [T + b * r + i for i in range(r) for b in range(3)]
    return sorted(listed, key=lambda k: vals[k])


def greedy_removal(model, snapshot_norm2: float) -> List[Tuple[int, float, int]]:
    """TURB:1166-1245: for step = 0..K zero the gates of the ``step`` smallest-norm terms, evaluate ||X - recon^T|| / ||X||
    (TURB:1227) and count the non-zero gates left (TURB:1229-1234).  One gradient-free fused pass per step on the resident
    snapshot instead of a DataLoader round trip + host numpy.  Returns [(step, relative_error, nonzero_terms)], gates restored."""
    e = model.engine
    if hasattr(model, "sync_parameters"):
        model.sync_parameters()
    order = removal_order(e.term_norms(), e.T, e.r)
    saved = e.gates.clone()
    out = []
    for step in range(e.K + 1):
        if step:
            e.gates[order[step - 1]] = 0.0
        out.append((step, float((e.residual_norm2() / snapshot_norm2) ** 0.5), int((e.gates != 0).sum().item())))
    e.gates.copy_(saved)
    return out


def threshold_steps(norms, gates, order, threshold: float) -> int:
    """How many leading terms of ``order`` a threshold removes.  threshold_sweep keeps a term iff norm >= threshold and its gate is
    non-zero; the removed terms are a prefix of the norm-ascending removal_order (a zero gate has norm 0 and comes first).  Raises
    DesmoError when the removed set is not a prefix of ``order``."""
    norms = np.asarray(norms.detach().cpu().numpy() if torch.is_tensor(norms) else norms, dtype=np.float64)
    gates = np.asarray(gates.detach().cpu().numpy() if torch.is_tensor(gates) else gates)
    removed = ~((norms >= threshold) & (gates != 0))
    s = int(removed.sum())
    if sorted(int(k) for k in order[:s]) != np.flatnonzero(removed).tolist():
        raise DesmoError(f"threshold {threshold} removes terms that are not the first {s} of this order")
    return s


@dataclass
class PruningProfile:
    """One pass over U for a whole pruning sequence.  Step s removes order[:s]; s = 0 .. len(order)."""
    order: List[int]
    snapshot_residual2: torch.Tensor  # (S+1, m) fp64: sum_x r_s(x, t)^2
    snapshot_norm2: torch.Tensor      # (m,) fp64: sum_x U(x, t)^2
    relative_error: List[float]       # ||X - recon_s|| / ||X|| per step (TURB:1227)
    nonzero_terms: List[int]          # non-zero gates left per step (TURB:1229-1234)
    term_norms: torch.Tensor          # (K,) fp64, the norms threshold_sweep compares with a threshold
    gates: torch.Tensor               # (K,) the gates the profile was taken with

    def steps_for_threshold(self, threshold: float) -> int:
        """The step whose removed terms are exactly those threshold_sweep removes at ``threshold``.  Raises DesmoError when no step
        of this order removes exactly that set, as for most thresholds on backward_elimination()'s order (a threshold removes a
        prefix of the norm order)."""
        return threshold_steps(self.term_norms, self.gates, self.order, threshold)

    def active_mask(self, step: int) -> torch.Tensor:
        """threshold_sweep's mask after ``step`` removals: gate non-zero and not among order[:step]."""
        mask = self.gates != 0
        mask[list(self.order[:step])] = False
        return mask

    def threshold_sweep(self, thresholds) -> List[Tuple[float, float, int, torch.Tensor]]:
        """threshold_sweep()'s [(threshold, relative_error, n_active, mask)], read off this profile."""
        out = []
        for thr in thresholds:
            s = self.steps_for_threshold(float(thr))
            out.append((float(thr), self.relative_error[s], self.nonzero_terms[s], self.active_mask(s)))
        return out


def pruning_profile(model, order=None, snapshot_norm2: Optional[float] = None) -> PruningProfile:
    """Every step of a term-pruning sequence scored in one pass over U (DesmoEngine.pruning_profile): per-snapshot residuals, the
    relative error ||X - recon_s|| / ||X|| and the non-zero gate count after removing order[:s], for s = 0 .. len(order).  The default
    order is removal_order(term_norms()), so the result is greedy_removal's curve, and threshold_sweep's points are read off it with
    steps_for_threshold.  ``snapshot_norm2`` is ||X||^2 (as greedy_removal takes it); by default the sum of the stored U's squares.
    The gates are not touched."""
    e = model.engine
    if hasattr(model, "sync_parameters"):
        model.sync_parameters()
    norms = e.term_norms()
    if order is None:
        order = removal_order(norms, e.T, e.r)
    order = [int(k) for k in (order.tolist() if torch.is_tensor(order) else order)]
    prof = e.pruning_profile(order)
    total = float(prof["snapshot_norm2"].sum()) if snapshot_norm2 is None else float(snapshot_norm2)
    rel = (prof["snapshot_residual2"].sum(1) / total).sqrt().tolist()
    gates = e.gates.clone()
    nz_host = (gates != 0).cpu().numpy()
    nonzero = [int(nz_host.sum())]
    for k in order:
        nonzero.append(nonzero[-1] - int(nz_host[k]))
    return PruningProfile(order, prof["snapshot_residual2"], prof["snapshot_norm2"], rel, nonzero, norms, gates)


def backward_elimination(model, steps: Optional[int] = None, snapshot_norm2: Optional[float] = None) -> PruningProfile:
    """Backward elimination by error at fixed coefficients: greedy_removal's experiment (no refit, one term per step) with the term
    whose removal raises ||X - recon|| least taken at each step instead of the smallest-norm one.  The order comes from the device
    greedy (DesmoEngine.backward_elimination: one pass over U, then A = G^T G and F = G^T R alone); the errors, per-snapshot
    residuals and non-zero counts come from pruning_profile(model, order), so they are exact and on the same axes as the norm order's
    pruning_profile(model).  active_mask(step) feeds set_active_terms for a refit; steps_for_threshold raises for this order (see
    there).  ``steps`` defaults to K; ``snapshot_norm2`` as in pruning_profile.  The gates, rows, step counter and any active set are
    left as they are."""
    e = model.engine
    if hasattr(model, "sync_parameters"):
        model.sync_parameters()
    order = e.backward_elimination(steps)["order"].tolist()
    return pruning_profile(model, order, snapshot_norm2)


def _stored_norm2(e) -> float:
    """||U||_F^2 of the stored snapshot matrix in fp64 (summed over the ranks when point-sharded), a few snapshots at a time."""
    if e.U is None:
        raise DesmoError("no snapshot matrix set (call set_snapshot)")
    tot = torch.zeros((), dtype=torch.float64, device=e.device)
    for t0 in range(0, e.m, 64):
        tot += e.U[t0:t0 + 64, :e.n].double().pow(2).sum()
    if e.n_global != e.n and torch.distributed.is_initialized():
        torch.distributed.all_reduce(tot, group=e.pg)
    return float(tot)


def sequential_thresholding(trainer, threshold: float, rounds: int, epochs: int,
                            snapshot_norm2: Optional[float] = None) -> List[Tuple[int, float]]:
    """Prune, then refit (sequentially thresholded sparse regression) on the engine's resident snapshot.  Each round takes
    threshold_sweep's mask at ``threshold`` (term norm >= threshold and gate non-zero), intersects it with the current active set,
    trains on the result (set_active_terms) for ``epochs`` steps of ``trainer`` and records (n_active, ||X - recon|| / ||X||) after
    the refit.  ``snapshot_norm2`` is ||X||^2; by default the sum of the stored U's squares.  The active set stays in place."""
    model, e = trainer.model, trainer.engine
    total = _stored_norm2(e) if snapshot_norm2 is None else float(snapshot_norm2)
    out = []
    for _ in range(int(rounds)):
        if hasattr(model, "sync_parameters"):
            model.sync_parameters()
        mask = ((e.term_norms() >= threshold) & (e.gates != 0)).cpu()
        if e.active_terms is not None:
            mask &= e.active_terms
        e.set_active_terms(mask)
        for _ in range(int(epochs)):
            trainer.step()
        out.append((int(mask.sum()), float((e.residual_norm2() / total) ** 0.5)))
    return out
