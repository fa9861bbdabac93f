"""The reference model at caller-given times, built on oracle/desmo_oracle.py: the Fourier scripts evaluate every series at the module
global ``t_points`` (FCYL:485, torch.linspace(0, m, m) as shipped); here that global is a table the caller passes.  Every function
runs the unchanged oracle with its t_points(m) replaced by the table for the duration of the call, so at the grid
(orc.t_points(m)) the results are the oracle's own bits, and elsewhere they are the same formulas at other times.
What tests/test_time_points*.py compare the engine with."""
import contextlib
import threading
from typing import Optional

import numpy as np

from oracle import desmo_oracle as orc
from tests import _active_oracle as ao

_LOCK = threading.Lock()


@contextlib.contextmanager
def at_times(t_points: Optional[np.ndarray]):
    """Inside the block, the oracle evaluates column t of a Fourier model at t_points[t] (None: the grid, nothing replaced).  The table
    is the model's fp32 time coordinate; an fp64 oracle run widens it exactly."""
    if t_points is None:
        yield
        return
    table = np.asarray(t_points, dtype=np.float32).reshape(-1)

    def t_of(m: int, dtype=np.float32) -> np.ndarray:
        if m != table.size:
            raise ValueError(f"the time table has {table.size} entries, the model {m} snapshots")
        return table.astype(dtype)

    with _LOCK:
        saved = orc.t_points
        orc.t_points = t_of
        try:
            yield
        finally:
            orc.t_points = saved


def fourier_rows(p: orc.DesmoParams, t_points: Optional[np.ndarray]) -> np.ndarray:
    """(K, m) series of every term at the table's times."""
    with at_times(t_points):
        return orc.temporal_rows(p)


def loss_and_grads(p: orc.DesmoParams, pod_modes: np.ndarray, snapshot: np.ndarray, beta: float, l1_lambda: float,
                   t_points: Optional[np.ndarray], want_grads: bool = True, active: Optional[np.ndarray] = None) -> orc.StepOutput:
    """Loss and gradients (coefficients and periods included) with the snapshot rows at the table's times, optionally on an active set."""
    with at_times(t_points):
        return ao.loss_and_grads(p, pod_modes, snapshot, beta, l1_lambda, want_grads, active)


def term_norms(p: orc.DesmoParams, t_points: Optional[np.ndarray], pod_modes: Optional[np.ndarray] = None,
               physical: bool = False) -> np.ndarray:
    """orc.term_norms (poly_norm / nonlinear_norm, the Fourier scripts' column quirk included) with the series at the table's times."""
    with at_times(t_points):
        return orc.term_norms(p, pod_modes, physical)


def train(p: orc.DesmoParams, pod_modes: np.ndarray, snapshot: np.ndarray, steps: int, beta: float, l1_lambda: float,
          t_points: Optional[np.ndarray], patience: int = 1000, sched_every: int = 10, lrs=orc.REFERENCE_LRS,
          active: Optional[np.ndarray] = None):
    """The reference loop (Adamax, ReduceLROnPlateau) at the table's times; returns (loss history, opt, sch)."""
    with at_times(t_points):
        return ao.train(p, pod_modes, snapshot, steps, beta, l1_lambda, patience, sched_every, lrs, active)


def finite_difference(p: orc.DesmoParams, pod_modes: np.ndarray, snapshot: np.ndarray, t_points: np.ndarray, key: str, index,
                      h: float) -> float:
    """Central fp64 difference of the MSE w.r.t. one entry of ``key`` ('coefs' or 'periods'): the independent check of the analytic
    coefficient and period gradients at times off the grid."""
    q = p.copy()
    for k in ("phi", "gates", "omega", "coefs", "periods"):
        setattr(q, k, getattr(q, k).astype(np.float64))
    snap = snapshot.astype(np.float64)
    vals = []
    for sgn in (1.0, -1.0):
        r = q.copy()
        getattr(r, key)[index] += sgn * h
        vals.append(loss_and_grads(r, pod_modes.astype(np.float64), snap, 0.0, 0.0, t_points, want_grads=False).mse)
    return (vals[0] - vals[1]) / (2.0 * h)
