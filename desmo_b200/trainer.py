"""Training loop of the reference (CYL:592-618,699-786) around the fused step.

Adamax itself runs on the device (desmo_adamax_update).  ReduceLROnPlateau stays on the host exactly as the reference
configures it (mode='min', factor=0.1, min_lr=1e-6, threshold=1e-4 rel; stepped every ``sched_every`` epochs on the total
loss -- 10 for CYL/FCYL (CYL:776-778), 1 for TURB/ANEU/FANEU), but the losses are fetched with ONE small D2H copy only
on the epochs where the reference prints / steps the scheduler, not with an ``.item()`` sync per step (CYL:769).
"""
from __future__ import annotations

import ctypes
import math
from typing import List, NamedTuple, Optional, Sequence

import numpy as np
import torch

from .engine import REFERENCE_LRS, DesmoEngine


class PlateauScheduler:
    """torch.optim.lr_scheduler.ReduceLROnPlateau semantics for the engine's 4-5 learning rates."""

    def __init__(self, lrs: Sequence[float], patience: int, factor: float = 0.1, min_lr: float = 1e-6, threshold: float = 1e-4,
                 eps: float = 1e-8):
        self.lrs = [float(v) for v in lrs]
        self.patience, self.factor, self.min_lr, self.threshold, self.eps = patience, factor, min_lr, threshold, eps
        self.best, self.num_bad = math.inf, 0

    def step(self, metric: float) -> bool:
        if metric < self.best * (1.0 - self.threshold):
            self.best, self.num_bad = metric, 0
        else:
            self.num_bad += 1
        changed = False
        if self.num_bad > self.patience:
            for i, old in enumerate(self.lrs):
                new = max(old * self.factor, self.min_lr)
                if old - new > self.eps:
                    self.lrs[i] = new
                    changed = True
            self.num_bad = 0
        return changed


class Validation(NamedTuple):
    """A held-out validation entry of ``DesmoTrainer.history`` (fit(validation=...)): after ``epoch`` epochs, the relative error
    sqrt(residual2 / norm2) of the held-out block, with residual2 = sum r^2 and norm2 = sum u^2 over the block (residual_profile_at)."""
    epoch: int
    rel_error: float
    residual2: float
    norm2: float


class _PlateauState(ctypes.Structure):  # desmo_plateau (include/desmo_b200.h)
    _fields_ = [("best", ctypes.c_double), ("lrs", ctypes.c_double * 5), ("threshold", ctypes.c_double), ("factor", ctypes.c_double),
                ("min_lr", ctypes.c_double), ("eps", ctypes.c_double), ("num_bad", ctypes.c_int32), ("patience", ctypes.c_int32),
                ("every", ctypes.c_int32), ("n_groups", ctypes.c_int32), ("reductions", ctypes.c_int32), ("pad", ctypes.c_int32)]


class DesmoTrainer:
    """The loop of CYL:699-786.  ``device_scheduler=True`` runs ReduceLROnPlateau inside the captured step (desmo_plateau_step) instead
    of on the host: identical learning-rate trajectory, but no device->host round trip per scheduler epoch -- ``step()`` then returns
    the losses only every ``log_every`` epochs (0: never; read ``engine.losses`` or call ``sync_scheduler()`` when needed)."""

    def __init__(self, model, lrs: Sequence[float] = REFERENCE_LRS, beta: float = 1e-3, l1_lambda: float = 1e-4,
                 patience: int = 1000, sched_every: int = 10, use_cuda_graph: bool = True, device_scheduler: bool = False,
                 log_every: int = 0):
        self.model = model
        self.engine: DesmoEngine = model.engine if hasattr(model, "engine") else model
        n_groups = 5 if self.engine.nF else 4
        self.beta, self.l1_lambda = float(beta), float(l1_lambda)
        self.scheduler = PlateauScheduler(list(lrs)[:n_groups], patience)
        self.sched_every = sched_every
        self.epoch = 0
        self.history: List[tuple] = []
        self.engine.set_hyper(self.scheduler.lrs, self.beta, self.l1_lambda)
        self.use_cuda_graph = use_cuda_graph
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._graph_active = None  # the engine's active-term table the graph was captured with
        self._graph_times = None   # ... and its time table (None: the grid)
        self.device_scheduler, self.log_every = bool(device_scheduler), int(log_every)
        self._plateau_dev: Optional[torch.Tensor] = None
        if self.device_scheduler:
            self._push_scheduler()

    # ---- device-side scheduler state <-> the host mirror (self.scheduler) ----
    def _push_scheduler(self) -> None:
        sc = self.scheduler
        st = _PlateauState()
        st.best, st.threshold, st.factor, st.min_lr, st.eps = sc.best, sc.threshold, sc.factor, sc.min_lr, sc.eps
        for i in range(5):
            st.lrs[i] = sc.lrs[i] if i < len(sc.lrs) else 0.0
        st.num_bad, st.patience, st.every, st.n_groups, st.reductions = sc.num_bad, sc.patience, self.sched_every, len(sc.lrs), 0
        raw = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8)
        if self._plateau_dev is None:
            self._plateau_dev = torch.zeros(ctypes.sizeof(_PlateauState), dtype=torch.uint8, device=self.engine.device)
        self._plateau_dev.copy_(raw)
        self.engine.plateau_state = self._plateau_dev

    def sync_scheduler(self) -> PlateauScheduler:
        """Device scheduler: reads its state back into ``self.scheduler`` (one D2H copy).  No-op for the host scheduler."""
        if self.device_scheduler and self._plateau_dev is not None:
            st = _PlateauState.from_buffer_copy(bytes(self._plateau_dev.cpu().numpy().tobytes()))
            sc = self.scheduler
            sc.best, sc.num_bad = st.best, st.num_bad
            sc.lrs = [st.lrs[i] for i in range(len(sc.lrs))]
            self.engine.hyper_host[:len(sc.lrs)] = [float(v) for v in sc.lrs]
        return self.scheduler

    def _launch(self) -> None:
        if not self.use_cuda_graph:
            self.engine.train_step()
            return
        if self._graph is not None and (self._graph_active is not self.engine._active or
                                        self._graph_times is not getattr(self.engine, "_times", None)):
            self._graph = None  # set_active_terms / set_time_points(None <-> table) changed the launches: capture again
        if self._graph is None:
            # warm up once outside capture (function attributes, NCCL communicators), then capture the step
            e = self.engine
            snap = {k: getattr(e, k).clone() for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m",
                                                      "rows_u", "omega", "omega_m", "omega_u", "step_dev")}
            if e.nF:
                snap.update({k: getattr(e, k).clone() for k in ("coefs", "coefs_m", "coefs_u", "periods", "periods_m", "periods_u")})
            side = torch.cuda.Stream(device=e.device)
            side.wait_stream(torch.cuda.current_stream(e.device))
            with torch.cuda.stream(side):
                e.train_step()
            torch.cuda.current_stream(e.device).wait_stream(side)
            torch.cuda.synchronize(e.device)
            for k, v in snap.items():
                getattr(e, k).copy_(v)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                e.train_step()
            self._graph, self._graph_active, self._graph_times = g, e._active, getattr(e, "_times", None)
            for k, v in snap.items():  # capture does not execute, but keep state exact regardless
                getattr(e, k).copy_(v)
        self._graph.replay()

    def step(self, snapshot: Optional[torch.Tensor] = None) -> Optional[tuple]:
        """One epoch (CYL:706-778).  Returns (mse, ortho, l1, total) on scheduler epochs, else None (no host sync)."""
        if snapshot is not None:
            self.engine.set_snapshot(snapshot)
        if self.epoch % 256 == 0 and hasattr(self.model, "sync_parameters"):
            # user code may have rebound param.data (the reference's sweep does, CYL:1219-1226).  The check walks every Parameter
            # (~2 us each, 1400 of them at r = 32), so the hot loop pays it on the first epoch and every 256th only; forward(),
            # mse_loss() and the sparsify sweeps check on every call.
            self.model.sync_parameters()
        self._launch()
        out = None
        if self.device_scheduler:
            if self.log_every and self.epoch % self.log_every == 0:
                out = tuple(float(v) for v in self.engine.losses.tolist())
                self.history.append((self.epoch, *out))
            self.epoch += 1
            return out
        if self.epoch % self.sched_every == 0:
            vals = tuple(float(v) for v in self.engine.losses.tolist())  # the only D2H sync
            self.history.append((self.epoch, *vals))
            if self.scheduler.step(vals[3]):
                self.engine.set_hyper(self.scheduler.lrs, self.beta, self.l1_lambda)
            out = vals
        self.epoch += 1
        return out

    # ---- checkpoint / resume (SURVEY.md section 8f-3).  The reference saves only model.state_dict() (CYL:781-786,802-805): no
    # optimizer / scheduler state and no POD modes, so its checkpoints cannot resume a run.  `model.state_dict()` stays the
    # reference-compatible artefact; this adds everything else needed for an exact continuation.
    def state_dict(self) -> dict:
        e = self.engine
        opt = {k: getattr(e, k).detach().clone() for k in ("phi_m", "phi_u", "gates_m", "gates_u", "rows_m", "rows_u", "omega_m", "omega_u",
                                                           "coefs_m", "coefs_u", "periods_m", "periods_u") if getattr(e, k) is not None}
        self.sync_scheduler()
        return {"model": {k: v.detach().clone() for k, v in self.model.state_dict().items()} if hasattr(self.model, "state_dict") else None,
                "optimizer": opt, "step": int(e.step_dev.item()), "pod_modes": e.P[:, :e.n].detach().clone(),
                "scheduler": {"lrs": list(self.scheduler.lrs), "best": self.scheduler.best, "num_bad": self.scheduler.num_bad,
                              "patience": self.scheduler.patience},
                "epoch": self.epoch, "beta": self.beta, "l1_lambda": self.l1_lambda, "sched_every": self.sched_every,
                "active_terms": None if e.active_terms is None else e.active_terms.clone(),
                "t_points": None if getattr(e, "t_points", None) is None else torch.from_numpy(e.t_points.copy()),
                "shape": {"n": e.n, "m": e.m, "r": e.r, "polyorder": e.polyorder, "nF": e.nF, "n_global": e.n_global}}

    def load_state_dict(self, sd: dict) -> None:
        e = self.engine
        shp = sd["shape"]
        if (shp["n"], shp["m"], shp["r"], shp["polyorder"], shp["nF"], shp.get("n_global", shp["n"])) != \
                (e.n, e.m, e.r, e.polyorder, e.nF, e.n_global):
            raise ValueError(f"checkpoint shape {shp} does not match the engine (n={e.n}, m={e.m}, r={e.r}, p={e.polyorder}, "
                             f"nF={e.nF}, n_global={e.n_global}); re-shard with desmo_b200.checkpoint first")
        if sd.get("model") is not None and hasattr(self.model, "load_state_dict"):
            self.model.load_state_dict(sd["model"], strict=True)
        for k, v in sd["optimizer"].items():
            dst = getattr(e, k)
            if k in ("phi_m", "phi_u") and v.shape[-1] != dst.shape[-1]:  # unpadded [r][n] (gathered / re-sharded checkpoints)
                dst.zero_()
                dst[:, :e.n].copy_(v)
            else:
                dst.copy_(v)
        e.step_dev.fill_(int(sd["step"]))
        e.P.zero_()
        e.P[:, :e.n].copy_(sd["pod_modes"])
        sc = sd["scheduler"]
        self.scheduler.lrs, self.scheduler.best, self.scheduler.num_bad = list(sc["lrs"]), sc["best"], sc["num_bad"]
        self.scheduler.patience = int(sc.get("patience", self.scheduler.patience))  # the LR schedule continues as it was configured
        self.sched_every = int(sd.get("sched_every", self.sched_every))
        self.epoch, self.beta, self.l1_lambda = int(sd["epoch"]), float(sd["beta"]), float(sd["l1_lambda"])
        e.set_hyper(self.scheduler.lrs, self.beta, self.l1_lambda)
        e.set_active_terms(sd.get("active_terms"))  # checkpoints without the key train every term
        t_points = sd.get("t_points")  # checkpoints without the key train on the grid
        if t_points is not None or getattr(e, "t_points", None) is not None:
            e.set_time_points(t_points)
        if self.device_scheduler:
            self._push_scheduler()

    def validate(self, snapshots: torch.Tensor, instants) -> Validation:
        """The held-out relative error of the current parameters on ``snapshots`` (m', n) at ``instants``: integer snapshot indices
        (index=, the model's own times t_points[k] when it has a table) or float times (times=, Fourier models).  One
        residual_profile_at pass; nothing the model owns is written."""
        raw = instants.detach().cpu().numpy() if torch.is_tensor(instants) else np.asarray(instants)
        kw = {"index": raw} if np.issubdtype(raw.dtype, np.integer) else {"times": raw}
        prof = self.engine.residual_profile_at(snapshots, **kw)
        r2, u2 = float(prof["snapshot_residual2"].sum()), float(prof["snapshot_norm2"].sum())
        return Validation(self.epoch, math.sqrt(r2 / u2) if u2 > 0 else math.inf, r2, u2)

    def fit(self, snapshot: torch.Tensor, epochs: int, log_every: int = 0, validation=None, val_every: int = 1):
        """``epochs`` steps on ``snapshot``.  ``validation=(snapshots, times_or_index)``: a held-out block (m', n) and its instants (see
        validate()); every ``val_every`` epochs a Validation entry (held-out relative error sqrt(sum r^2 / sum u^2)) is appended to
        ``history`` after the loss entries of that epoch.  Validation is measurement only: it does not change the training."""
        if validation is not None:
            if int(val_every) < 1:
                raise ValueError(f"val_every must be >= 1, got {val_every}")
            val_snap, val_at = validation
        self.engine.set_snapshot(snapshot)
        for _ in range(epochs):
            vals = self.step()
            if log_every and vals is not None and (self.epoch - 1) % log_every == 0:
                print(f"Epoch [{self.epoch}/{epochs}], Rec Loss: {vals[0]:.12f}, Spatial ortho loss: {vals[1]:.8f}, "
                      f"L1 loss: {vals[2]:.4f} ", flush=True)  # CYL:777
            if validation is not None and self.epoch % int(val_every) == 0:
                self.history.append(self.validate(val_snap, val_at))
        return self.history
