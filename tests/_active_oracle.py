"""The reference model on an active set of library terms, built on oracle/desmo_oracle.py: the gates multiplied by a fixed 0/1 buffer
(bool (K,)), and the pruned parameters -- a term's gate, temporal row (Fourier: coefficients and period) and, for a trig term
T + b r + i, omega[3i + b] -- left out of the optimizer.  What tests/test_active_terms*.py compare the engine with."""
from typing import Dict, Optional

import numpy as np

from oracle import desmo_oracle as orc


def frozen_masks(p: orc.DesmoParams, active: np.ndarray) -> Dict[str, np.ndarray]:
    """Trainable entries (True) of the per-term parameters under the active set."""
    active = np.asarray(active, dtype=bool)
    T, r = p.T, p.r
    q = np.arange(3 * r)
    out = {"gates": active.copy(), "omega": active[T + (q % 3) * r + q // 3]}
    for k in ("zall", "coefs", "periods"):
        v = getattr(p, k)
        if v is not None:
            out[k] = np.broadcast_to(active.reshape((-1,) + (1,) * (v.ndim - 1)), v.shape).copy()
    return out


def loss_and_grads(p: orc.DesmoParams, pod_modes: np.ndarray, snapshot: np.ndarray, beta: float, l1_lambda: float,
                   want_grads: bool = True, active: Optional[np.ndarray] = None) -> orc.StepOutput:
    """orc.loss_and_grads of the model with the gates multiplied by ``active``; the gradients of the frozen entries are exactly zero.
    active=None is orc.loss_and_grads itself."""
    if active is None:
        return orc.loss_and_grads(p, pod_modes, snapshot, beta, l1_lambda, want_grads)
    q = p.copy()
    q.gates = (p.gates * np.asarray(active, dtype=bool)).astype(p.gates.dtype)
    out = orc.loss_and_grads(q, pod_modes, snapshot, beta, l1_lambda, want_grads)
    for k, fm in frozen_masks(p, active).items():
        if k in out.grads:
            out.grads[k] = np.where(fm, out.grads[k], 0).astype(out.grads[k].dtype)
    return out


def adamax_step(opt: orc.Adamax, params: orc.DesmoParams, grads: Dict[str, np.ndarray], active: Optional[np.ndarray] = None) -> None:
    """opt.step with the frozen entries and their Adamax state left as they are (the same operations as orc.Adamax.step on the rest)."""
    if active is None:
        opt.step(params, grads)
        return
    fms = frozen_masks(params, active)
    opt.t += 1
    bc = 1.0 - opt.b1 ** opt.t
    for lr, names in zip(opt.lrs, opt.groups):
        for k in names:
            prm = getattr(params, k)
            dt = prm.dtype.type
            g = grads[k].astype(prm.dtype)
            m_, u_ = opt.exp_avg[k], opt.exp_inf[k]
            fm = fms.get(k, np.ones(prm.shape, bool))
            nm = m_ + dt(1.0 - opt.b1) * (g - m_)
            nu = np.maximum(u_ * dt(opt.b2), np.abs(g) + dt(opt.eps))
            m_[fm], u_[fm] = nm[fm], nu[fm]
            prm[fm] += dt(-(lr / bc)) * m_[fm] / u_[fm]


def train(p: orc.DesmoParams, pod_modes: np.ndarray, snapshot: np.ndarray, steps: int, beta: float, l1_lambda: float,
          patience: int = 1000, sched_every: int = 10, lrs=orc.REFERENCE_LRS, active: Optional[np.ndarray] = None,
          opt: Optional[orc.Adamax] = None, sch: Optional[orc.ReduceLROnPlateau] = None):
    """orc.train's loop on the active set; ``opt`` / ``sch`` continue an earlier run's optimizer and scheduler (the scheduler's epoch
    count restarts at 0, as orc.train's does).  Returns (loss history, opt, sch)."""
    opt = orc.Adamax(p, lrs) if opt is None else opt
    sch = orc.ReduceLROnPlateau(opt, patience) if sch is None else sch
    hist = []
    for ep in range(steps):
        o = loss_and_grads(p, pod_modes, snapshot, beta, l1_lambda, active=active)
        adamax_step(opt, p, o.grads, active)
        hist.append((o.mse, o.ortho, o.l1, o.total))
        if ep % sched_every == 0:
            sch.step(o.total)
    return np.array(hist), opt, sch
