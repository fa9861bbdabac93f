"""Drop-in ``DESMO`` / ``DESMOFourier`` modules (reference: CYL:500-576, FCYL:512-589) backed by the CUDA engine.

Same class names, constructor arguments, parameter names / shapes / registration order (so the reference's optimizer-group
construction CYL:592-612, L1 loop CYL:725-731, threshold code CYL:1219-1238 and ``state_dict`` / ``load_state_dict`` work
unchanged, and the shipped ``.pt`` files load with ``strict=True``).  Every ``nn.Parameter`` is a VIEW into the engine's
packed device buffers, so kernel-side updates are visible through the module and vice versa.

The reference reads ``POD_modes`` / ``device`` / ``t_points`` / ``period_init`` from module globals; here they are explicit
keyword arguments (``pod_modes=...``, ``DESMOFourier(..., t_points=...)``; ``t_points=None`` is the scripts' torch.linspace(0, m, m)).  ``forward(X)`` keeps the reference signature and returns the same 3-tuple; ``recon`` is
materialised and carries a ``grad_fn`` whose backward runs the fused kernels on the upstream gradient (``desmo_recon_backward``),
so the reference loop ``recon, lat, _ = model(snapshot); loss = criterion(recon, snapshot); total.backward(); optimizer.step()``
(CYL:711-768) runs unmodified.  The fast paths are ``DesmoTrainer.step()`` (fully fused, no m x n tensor besides the snapshot)
and ``model.mse_loss(snapshot)`` (autograd-visible loss whose backward is the fused pass).

The reference's post-hoc sweep rebinds ``param.data = clone`` (CYL:1219-1226), which detaches a Parameter from the packed
buffer it aliased; every entry point that launches kernels first calls ``sync_parameters()``, which copies such a Parameter's
values back into the packed storage and re-aliases it, so that code runs unmodified too.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import nn

from . import _lib
from .engine import DesmoEngine


class _FusedMSE(torch.autograd.Function):
    """mse = MSELoss(recon, snapshot) (CYL:722) with the fused pass as its backward."""

    @staticmethod
    def forward(ctx, engine: DesmoEngine, names, *params):
        g = engine.gradients(beta=0.0, l1_lambda=0.0)  # pure d mse / d params
        ctx.engine, ctx.names, ctx.grads = engine, names, g
        return engine.losses[0].clone()

    @staticmethod
    def backward(ctx, grad_out):
        eng, g = ctx.engine, ctx.grads
        res = []
        for kind, idx in ctx.names:
            res.append(_slice_grad(eng, g, kind, idx) * grad_out)
        return (None, None, *res)


class _FusedRecon(torch.autograd.Function):
    """recon = forward()[0] (CYL:572-576), differentiable: backward(dL/drecon) = desmo_recon_backward + desmo_assemble_grads."""

    @staticmethod
    def forward(ctx, engine: DesmoEngine, names, *params):
        ctx.engine, ctx.names = engine, names
        return engine.reconstruct()

    @staticmethod
    def backward(ctx, grad_recon):
        eng = ctx.engine
        g = eng.recon_backward(grad_recon)
        return (None, None, *[_slice_grad(eng, g, kind, idx) for kind, idx in ctx.names])


def _slice_grad(eng: DesmoEngine, g: dict, kind: str, idx) -> torch.Tensor:
    T, r = eng.T, eng.r
    rows_key = "coefs" if eng.nF else "rows"
    if kind == "c_coef":
        return g["gates"][:T]
    if kind == "phi":
        return g["phi"][idx]
    if kind == "z":
        return g[rows_key][idx]
    if kind in ("zsin", "zcos", "ztanh"):
        b = ("zsin", "zcos", "ztanh").index(kind)
        return g[rows_key][T + b * r + idx]
    if kind in ("sin_coef", "cos_coef", "tanh_coef"):
        b = ("sin_coef", "cos_coef", "tanh_coef").index(kind)
        return g["gates"][T + b * r + idx]
    if kind == "omega":
        return g["omega"][idx]
    if kind == "period":
        return g["periods"][idx:idx + 1]
    if kind == "trig_period":
        i, b = divmod(idx, 3)
        return g["periods"][T + b * r + i:T + b * r + i + 1]
    raise KeyError(kind)


class _DesmoBase(nn.Module):
    def _build(self, n, m, polyorder, r_DESMO, omega_init, nF, period_init, pod_modes, device, n_global, path, process_group,
               snapshot_dtype, t_points=None):
        self.engine = DesmoEngine(n, m, polyorder, r_DESMO, omega_init, nF, period_init, device=device, n_global=n_global,
                                  path=path, process_group=process_group, snapshot_dtype=snapshot_dtype, t_points=t_points)
        e = self.engine
        T, r = e.T, e.r
        print('Number of terms in polynomial library:', T)  # CYL:510
        P = lambda t: nn.Parameter(t)  # noqa: E731   (aliases the packed storage)
        rows = e.coefs if e.nF else e.rows[:, :e.m]
        self._order = []
        # registration order == reference's __init__ (CYL:506-530 / FCYL:518-544) -> identical state_dict key order
        self.phi_list = nn.ParameterList([P(e.phi[i, :e.n]) for i in range(r)])
        self.c_coef = P(e.gates[:T])
        self.z_list = nn.ParameterList([P(rows[j]) for j in range(T)])
        if e.nF:
            self.period_list = nn.ParameterList([P(e.periods[j:j + 1]) for j in range(T)])
            self.trig_period_list = nn.ParameterList(
                [P(e.periods[T + (q % 3) * r + q // 3:T + (q % 3) * r + q // 3 + 1]) for q in range(3 * r)])
        self.zsin_list = nn.ParameterList([P(rows[T + i]) for i in range(r)])
        self.zcos_list = nn.ParameterList([P(rows[T + r + i]) for i in range(r)])
        self.ztanh_list = nn.ParameterList([P(rows[T + 2 * r + i]) for i in range(r)])
        self.sin_coef_list = nn.ParameterList([P(e.gates[T + i]) for i in range(r)])
        self.cos_coef_list = nn.ParameterList([P(e.gates[T + r + i]) for i in range(r)])
        self.tanh_coef_list = nn.ParameterList([P(e.gates[T + 2 * r + i]) for i in range(r)])
        self.omega_list = nn.ParameterList([P(e.omega[i]) for i in range(3 * r)])
        if pod_modes is not None:
            e.set_pod_modes(pod_modes)

    # nn.Module re-orders nothing, but the reference registers phi_list BEFORE c_coef while state_dict lists c_coef first:
    # nn.Module.state_dict emits direct parameters (c_coef) before sub-module parameters (the ParameterLists).  Same here.

    def _named_for_autograd(self):
        e = self.engine
        names, params = [("c_coef", 0)], [self.c_coef]
        for kind, lst in (("phi", self.phi_list), ("z", self.z_list), ("zsin", self.zsin_list), ("zcos", self.zcos_list),
                          ("ztanh", self.ztanh_list), ("sin_coef", self.sin_coef_list), ("cos_coef", self.cos_coef_list),
                          ("tanh_coef", self.tanh_coef_list), ("omega", self.omega_list)):
            for i, p in enumerate(lst):
                names.append((kind, i))
                params.append(p)
        if e.nF:
            for i, p in enumerate(self.period_list):
                names.append(("period", i))
                params.append(p)
            for i, p in enumerate(self.trig_period_list):
                names.append(("trig_period", i))
                params.append(p)
        return names, params

    def _apply(self, fn, recurse=True):
        before = self.engine.phi.data_ptr()
        out = super()._apply(fn, recurse)
        if self.phi_list[0].data_ptr() != before:
            raise _lib.DesmoError("desmo_b200 parameters are views of packed CUDA buffers: construct the module with device=... "
                                  "instead of moving / casting it (no CPU fallback)")
        return out

    def _views(self):
        """(Parameter, view of the packed buffer it must alias) for every parameter, registration order."""
        e = self.engine
        T, r = e.T, e.r
        rows = e.coefs if e.nF else e.rows[:, :e.m]
        yield self.c_coef, e.gates[:T]
        for i in range(r):
            yield self.phi_list[i], e.phi[i, :e.n]
        for j in range(T):
            yield self.z_list[j], rows[j]
        if e.nF:
            for j in range(T):
                yield self.period_list[j], e.periods[j:j + 1]
            for q in range(3 * r):
                k = T + (q % 3) * r + q // 3
                yield self.trig_period_list[q], e.periods[k:k + 1]
        for b, (zl, cl) in enumerate(((self.zsin_list, self.sin_coef_list), (self.zcos_list, self.cos_coef_list),
                                      (self.ztanh_list, self.tanh_coef_list))):
            for i in range(r):
                yield zl[i], rows[T + b * r + i]
                yield cl[i], e.gates[T + b * r + i]
        for i in range(3 * r):
            yield self.omega_list[i], e.omega[i]

    def sync_parameters(self) -> int:
        """Re-establishes Parameter <-> packed-buffer aliasing after user code rebound ``param.data`` (the reference's threshold
        sweep does, CYL:1219-1226): the Parameter's current values are copied into the packed storage and the Parameter is
        pointed back at it.  Returns the number of parameters that had been detached.  Raises on a shape / device change."""
        fixed = 0
        for p, v in self._views():
            if p.data_ptr() == v.data_ptr() and p.shape == v.shape:
                continue
            if p.numel() != v.numel() or p.device != v.device or p.dtype != v.dtype:
                raise _lib.DesmoError(f"parameter rebound to an incompatible tensor: {tuple(p.shape)} {p.dtype} {p.device} "
                                      f"(expected {tuple(v.shape)} float32 on {v.device})")
            with torch.no_grad():
                v.copy_(p.data.reshape(v.shape))
            p.data = v
            fixed += 1
        return fixed

    # ---- reference surface -------------------------------------------------------------------------------------------
    def set_pod_modes(self, pod_modes) -> None:
        self.engine.set_pod_modes(pod_modes)

    def latent_spatial(self) -> torch.Tensor:
        """(n, r) = stack(phi_i * POD_i) with autograd through phi_list (CYL:538-545); cheap, used for the ortho term."""
        e = self.engine
        return torch.stack([p * e.P[i, :e.n] for i, p in enumerate(self.phi_list)], dim=1)

    def forward(self, X=None):
        """(recon (m, n), latent_spatial (n, r), z_values (T, m)) as CYL:576.  ``X`` is ignored, as in the reference.
        All three are differentiable like the reference's (recon through the fused backward kernels)."""
        e = self.engine
        self.sync_parameters()
        names, params = self._named_for_autograd()
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            recon = _FusedRecon.apply(e, names, *params)
        else:
            recon = e.reconstruct()
        lat = self.latent_spatial()
        if e.nF:
            zv = e.rows[:e.T, :e.m].clone()  # series as evaluated by the last build_w (FCYL:563)
        else:
            zv = torch.stack(list(self.z_list), dim=0)  # CYL:550
        return recon, lat, zv

    # ---- evaluation at chosen instants (DesmoEngine; exactly one of index= / times=, no autograd) ---------------------------
    def time_points(self, index):
        return self.engine.time_points(index)

    def temporal_rows_at(self, index=None, times=None) -> torch.Tensor:
        self.sync_parameters()
        return self.engine.temporal_rows_at(index=index, times=times)

    def reconstruct_at(self, index=None, times=None) -> torch.Tensor:
        self.sync_parameters()
        return self.engine.reconstruct_at(index=index, times=times)

    def residual_profile_at(self, snapshots: torch.Tensor, index=None, times=None) -> dict:
        self.sync_parameters()
        return self.engine.residual_profile_at(snapshots, index=index, times=times)

    def residual_pod(self, k: int = 8) -> dict:
        """POD of the residual recon - U of the current parameters: its singular spectrum and k leading modes (DesmoEngine.residual_pod)."""
        self.sync_parameters()
        return self.engine.residual_pod(k)

    def backward_elimination(self, steps=None) -> dict:
        """The removal order by error at fixed coefficients, chosen on the device (DesmoEngine.backward_elimination)."""
        self.sync_parameters()
        return self.engine.backward_elimination(steps)

    # ---- caller-given times (DesmoEngine.set_time_points) --------------------------------------------------------------------
    @property
    def t_points(self):
        """The fp32 (m,) host time table of the snapshot rows, or None for the grid torch.linspace(0, m, m)."""
        return self.engine.t_points

    def set_time_points(self, t_points) -> None:
        """Train and evaluate at ``t_points`` (m finite times, one per snapshot row; None: the grid); see DesmoEngine.set_time_points."""
        self.engine.set_time_points(t_points)

    # ---- training a pruned model (DesmoEngine.set_active_terms) ----------------------------------------------------------------
    def set_active_terms(self, mask) -> None:
        """Train on the terms of the bool (K,) ``mask`` only (None: every term); see DesmoEngine.set_active_terms.  The set applies to
        DesmoTrainer's fused step; a torch optimizer stepping this module's Parameters does not know it and would move frozen entries."""
        self.sync_parameters()
        self.engine.set_active_terms(mask)

    def mse_loss(self, snapshot: Optional[torch.Tensor] = None) -> torch.Tensor:
        """criterion(model(snapshot)[0], snapshot) (CYL:711,722) without materialising recon; differentiable w.r.t. every
        parameter of the module (backward = the fused residual+grad kernel)."""
        self.sync_parameters()
        if snapshot is not None:
            self.engine.set_snapshot(snapshot)
        names, params = self._named_for_autograd()
        return _FusedMSE.apply(self.engine, names, *params)


class DESMO(_DesmoBase):
    """``snapshot_dtype=torch.bfloat16`` stores the snapshot matrix in bf16 (see DesmoEngine).  Free temporal rows have no time
    coordinate: ``t_points`` other than None raises DesmoError."""

    def __init__(self, n, m, polyorder, r_DESMO, omega_init=10000, *, pod_modes=None, device=None, n_global=None,
                 path=_lib.PATH_AUTO, process_group=None, snapshot_dtype=torch.float32, t_points=None):
        if t_points is not None:
            raise _lib.DesmoError("DESMO has free temporal rows and no time coordinate: t_points needs DESMOFourier")
        super().__init__()
        self._build(n, m, polyorder, r_DESMO, omega_init, None, 0.0, pod_modes, device, n_global, path, process_group, snapshot_dtype)


class DESMOFourier(_DesmoBase):
    """``snapshot_dtype=torch.bfloat16`` stores the snapshot matrix in bf16 (see DesmoEngine).  ``t_points``: the times of the m
    snapshot rows (tensor, array or sequence; the reference's module global t_points, FCYL:485), or None for its default
    torch.linspace(0, m, m).  See DesmoEngine.set_time_points."""

    def __init__(self, n, m, polyorder, r_DESMO, omega_init=10000, nF=10, *, period_init=60.0, pod_modes=None, device=None,
                 n_global=None, path=_lib.PATH_AUTO, process_group=None, snapshot_dtype=torch.float32, t_points=None):
        super().__init__()
        self._build(n, m, polyorder, r_DESMO, omega_init, nF, period_init, pod_modes, device, n_global, path, process_group,
                    snapshot_dtype, t_points)
