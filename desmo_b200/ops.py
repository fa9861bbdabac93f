"""torch custom ops over the C ABI: one ``torch.ops.desmo_b200.*`` op per hot-path entry point of include/desmo_b200.h.

  build_w, fused_residual_grad, recon_backward, adamax_update, assemble_grads, reconstruct, library_colnorm2, term_norms,
  pod_gram, pod_eig, pod_project, preprocess, snapshot_to_bf16, plateau_step, peer_begin_step, peer_allreduce

They take the packed device tensors of a DesmoEngine (layout: include/desmo_b200.h) plus the shape integers and launch the
sm_100a kernels on the current stream.  CUDA only: no CPU implementation is registered and every op checks its tensors, so a call
with CPU tensors fails loudly.  The ops that read the snapshot matrix U take it in fp32 or bf16 (dispatched on U.dtype); any other
dtype raises before a launch."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import check, make_shape


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.DesmoError("desmo_b200 ops are CUDA-only (sm_100a); no CPU fallback")


@torch.library.custom_op("desmo_b200::build_w", mutates_args=("rows", "W", "step", "workspace"))
def build_w(gates: torch.Tensor, rows: torch.Tensor, coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor], W: torch.Tensor,
            step: torch.Tensor, workspace: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    _require_cuda(gates, rows, W)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(gates.device):
        check(_lib.load().desmo_build_w(C.byref(s), _p(gates), _p(rows), _p(coefs), _p(periods), _p(W), _p(step), _p(workspace),
                                        _stream(gates)), "desmo_build_w")


@torch.library.custom_op("desmo_b200::fused_residual_grad", mutates_args=("dphi", "red", "workspace"))
def fused_residual_grad(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, dphi: torch.Tensor,
                        red: torch.Tensor, workspace: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int,
                        path: int) -> None:
    _require_cuda(U, P, phi, omega, W, dphi, red)
    ud = _lib.u_dtype_code(U.dtype)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_fused_residual_grad_ex(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), _p(dphi), _p(red),
                                                       _p(workspace), _stream(U)), "desmo_fused_residual_grad")


@torch.library.custom_op("desmo_b200::recon_backward", mutates_args=("dphi", "red", "workspace"))
def recon_backward(grad_recon: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor,
                   dphi: torch.Tensor, red: torch.Tensor, workspace: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int,
                   nF: int, path: int) -> None:
    _require_cuda(grad_recon, P, phi, omega, W, dphi, red)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(P.device):
        check(_lib.load().desmo_recon_backward(C.byref(s), _p(grad_recon), _p(P), _p(phi), _p(omega), _p(W), _p(dphi), _p(red),
                                               _p(workspace), _stream(P)), "desmo_recon_backward")


@torch.library.custom_op("desmo_b200::adamax_update",
                         mutates_args=("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "coefs", "coefs_m",
                                       "coefs_u", "periods", "periods_m", "periods_u", "omega", "omega_m", "omega_u", "losses", "workspace"))
def adamax_update(red: torch.Tensor, dphi: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, phi_m: torch.Tensor, phi_u: torch.Tensor,
                  gates: torch.Tensor, gates_m: torch.Tensor, gates_u: torch.Tensor, rows: torch.Tensor, rows_m: torch.Tensor,
                  rows_u: torch.Tensor, coefs: Optional[torch.Tensor], coefs_m: Optional[torch.Tensor], coefs_u: Optional[torch.Tensor],
                  periods: Optional[torch.Tensor], periods_m: Optional[torch.Tensor], periods_u: Optional[torch.Tensor],
                  omega: torch.Tensor, omega_m: torch.Tensor, omega_u: torch.Tensor, hyper: torch.Tensor, step: torch.Tensor,
                  losses: torch.Tensor, workspace: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int,
                  path: int) -> None:
    _require_cuda(red, dphi, P, phi, gates, rows, omega, hyper, step, losses)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_adamax_update(
            C.byref(s), _p(red), _p(dphi), _p(P), _p(phi), _p(phi_m), _p(phi_u), _p(gates), _p(gates_m), _p(gates_u), _p(rows), _p(rows_m),
            _p(rows_u), _p(coefs), _p(coefs_m), _p(coefs_u), _p(periods), _p(periods_m), _p(periods_u), _p(omega), _p(omega_m), _p(omega_u),
            _p(hyper), _p(step), _p(losses), _p(workspace), _stream(phi)), "desmo_adamax_update")


@torch.library.custom_op("desmo_b200::assemble_grads",
                         mutates_args=("dphi", "d_gates", "d_rows", "d_coefs", "d_periods", "d_omega", "losses", "workspace"))
def assemble_grads(red: torch.Tensor, dphi: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, gates: torch.Tensor, rows: torch.Tensor,
                   coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor], hyper: torch.Tensor, d_gates: torch.Tensor,
                   d_rows: Optional[torch.Tensor], d_coefs: Optional[torch.Tensor], d_periods: Optional[torch.Tensor], d_omega: torch.Tensor,
                   losses: torch.Tensor, workspace: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int,
                   path: int) -> None:
    _require_cuda(red, dphi, P, phi, gates, rows, hyper, d_gates, d_omega, losses)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_assemble_grads(
            C.byref(s), _p(red), _p(dphi), _p(P), _p(phi), _p(gates), _p(rows), _p(coefs), _p(periods), _p(hyper), _p(d_gates), _p(d_rows),
            _p(d_coefs), _p(d_periods), _p(d_omega), _p(losses), _p(workspace), _stream(phi)), "desmo_assemble_grads")


@torch.library.custom_op("desmo_b200::reconstruct", mutates_args=("out",))
def reconstruct(P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, out: torch.Tensor, n: int, n_global: int, m: int,
                r: int, polyorder: int, nF: int, path: int) -> None:
    _require_cuda(P, phi, omega, W, out)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(P.device):
        check(_lib.load().desmo_reconstruct(C.byref(s), _p(P), _p(phi), _p(omega), _p(W), _p(out), _stream(P)), "desmo_reconstruct")


@torch.library.custom_op("desmo_b200::library_colnorm2", mutates_args=("out",))
def library_colnorm2(P: Optional[torch.Tensor], phi: torch.Tensor, omega: torch.Tensor, out: torch.Tensor, n: int, n_global: int, m: int,
                     r: int, polyorder: int, nF: int, path: int) -> None:
    _require_cuda(P, phi, omega, out)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_library_colnorm2(C.byref(s), _p(P), _p(phi), _p(omega), _p(out), _stream(phi)), "desmo_library_colnorm2")


@torch.library.custom_op("desmo_b200::term_norms", mutates_args=("out",))
def term_norms(g2: torch.Tensor, gates: torch.Tensor, rows: torch.Tensor, fourier_quirk: int, out: torch.Tensor, n: int, n_global: int,
               m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    _require_cuda(g2, gates, rows, out)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(g2.device):
        check(_lib.load().desmo_term_norms(C.byref(s), _p(g2), _p(gates), _p(rows), fourier_quirk, _p(out), _stream(g2)), "desmo_term_norms")


@torch.library.custom_op("desmo_b200::pod_gram", mutates_args=("Cm", "workspace"))
def pod_gram(U: torch.Tensor, Cm: torch.Tensor, workspace: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int,
             path: int) -> None:
    _require_cuda(U, Cm, workspace)
    ud = _lib.u_dtype_code(U.dtype)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_pod_gram_ex(C.byref(s), _p(U), ud, _p(Cm), _p(workspace), _stream(U)), "desmo_pod_gram")


@torch.library.custom_op("desmo_b200::pod_eig", mutates_args=("V", "sigma", "workspace"))
def pod_eig(Cm: torch.Tensor, V: torch.Tensor, sigma: torch.Tensor, workspace: torch.Tensor, m: int, r: int) -> None:
    _require_cuda(Cm, V, sigma, workspace)
    with torch.cuda.device(Cm.device):
        check(_lib.load().desmo_pod_eig(m, r, _p(Cm), _p(V), _p(sigma), _p(workspace), workspace.numel() * workspace.element_size(),
                                        _stream(Cm)), "desmo_pod_eig")


@torch.library.custom_op("desmo_b200::pod_project", mutates_args=("P",))
def pod_project(U: torch.Tensor, V: torch.Tensor, sigma: torch.Tensor, P: torch.Tensor, n: int, n_global: int, m: int, r: int,
                polyorder: int, nF: int, path: int) -> None:
    _require_cuda(U, V, sigma, P)
    ud = _lib.u_dtype_code(U.dtype)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_pod_project_ex(C.byref(s), _p(U), ud, _p(V), _p(sigma), _p(P), _stream(U)), "desmo_pod_project")


@torch.library.custom_op("desmo_b200::preprocess", mutates_args=("U", "mean"))
def preprocess(V: torch.Tensor, U: torch.Tensor, mean: Optional[torch.Tensor], m_in: int, t_stride: int, d_in: int, d_use: int, flags: int,
               n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """U is written in its own dtype: fp32, or bf16 (the fp32 result rounded to nearest even once more)."""
    _require_cuda(V, U, mean)
    if V.dtype not in (torch.float32, torch.float64) or V.dim() != 2 or V.stride(1) != 1:
        raise ValueError("V must be a [m_in, n*d_in] fp32/fp64 tensor with unit inner stride")
    ud = _lib.u_dtype_code(U.dtype)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(V.device):
        check(_lib.load().desmo_preprocess_ex(C.byref(s), _p(V), 1 if V.dtype == torch.float64 else 0, V.stride(0), m_in, t_stride, d_in,
                                              d_use, flags, _p(U), ud, None, _p(mean), _stream(V)), "desmo_preprocess")


@torch.library.custom_op("desmo_b200::snapshot_to_bf16", mutates_args=("U", "qsums"))
def snapshot_to_bf16(src: torch.Tensor, U: torch.Tensor, qsums: Optional[torch.Tensor], t0: int, n: int, n_global: int, m: int, r: int,
                     polyorder: int, nF: int, path: int) -> None:
    """fp32 rows src [rows, >= n] -> bf16 U[t0 : t0 + rows, :] (round to nearest even, pad columns zeroed); qsums (fp64 [2], optional)
    += {sum (u - q)^2, sum u^2} (desmo_snapshot_to_bf16)."""
    _require_cuda(src, U, qsums)
    if src.dtype != torch.float32 or src.dim() != 2 or src.stride(1) != 1:
        raise ValueError("src must be a [rows, >= n] fp32 tensor with unit inner stride")
    if U.dtype != torch.bfloat16:
        raise _lib.DesmoError(f"snapshot_to_bf16 writes a bfloat16 U, got {U.dtype}")
    if qsums is not None and (qsums.dtype != torch.float64 or qsums.numel() < 2):
        raise ValueError("qsums must be a float64 tensor of 2 elements")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_snapshot_to_bf16(C.byref(s), _p(src), src.stride(0), t0, src.shape[0], _p(U), _p(qsums), _stream(U)),
              "desmo_snapshot_to_bf16")


@torch.library.custom_op("desmo_b200::plateau_step", mutates_args=("state", "hyper"))
def plateau_step(state: torch.Tensor, step: torch.Tensor, losses: torch.Tensor, hyper: torch.Tensor) -> None:
    """ReduceLROnPlateau.step(losses[3]) on the device (desmo_plateau_step); ``state`` is the desmo_plateau struct as bytes."""
    _require_cuda(state, step, losses, hyper)
    with torch.cuda.device(state.device):
        check(_lib.load().desmo_plateau_step(_p(state), _p(step), _p(losses), _p(hyper), _stream(state)), "desmo_plateau_step")


@torch.library.custom_op("desmo_b200::peer_begin_step", mutates_args=("peer_state",))
def peer_begin_step(peer_tables: torch.Tensor, peer_state: torch.Tensor, world: int, rank: int) -> None:
    """Waits (on the stream) until every peer has consumed this rank's previous ``red``.  peer_tables: int64 [2 * world] device tensor
    (addresses of every rank's red buffer, then of every rank's flag pad); peer_state: int32 [2]."""
    from .engine import _PeerDesc

    _require_cuda(peer_tables, peer_state)
    d = _PeerDesc(world, rank, peer_tables.data_ptr(), peer_tables.data_ptr() + 8 * world, peer_state.data_ptr())
    with torch.cuda.device(peer_tables.device):
        check(_lib.load().desmo_peer_begin_step(C.byref(d), _stream(peer_tables)), "desmo_peer_begin_step")


@torch.library.custom_op("desmo_b200::peer_allreduce", mutates_args=("red_sum", "peer_state"))
def peer_allreduce(peer_tables: torch.Tensor, peer_state: torch.Tensor, red_sum: torch.Tensor, world: int, rank: int) -> None:
    """One-shot rank-ordered sum of every rank's peer-mapped ``red`` into red_sum (desmo_peer_allreduce)."""
    from .engine import _PeerDesc

    _require_cuda(peer_tables, peer_state, red_sum)
    d = _PeerDesc(world, rank, peer_tables.data_ptr(), peer_tables.data_ptr() + 8 * world, peer_state.data_ptr())
    with torch.cuda.device(peer_tables.device):
        check(_lib.load().desmo_peer_allreduce(C.byref(d), red_sum.numel(), _p(red_sum), _stream(peer_tables)), "desmo_peer_allreduce")


def _shape_args(e):
    return (e.n, e.n_global, e.m, e.r, e.polyorder, e.nF, e.shape.path)


def engine_step_via_ops(e) -> None:
    """One train step of a DesmoEngine routed entirely through the registered ops."""
    sa = _shape_args(e)
    torch.ops.desmo_b200.build_w(e.gates, e.rows, e.coefs, e.periods, e.W, e.step_dev, e.workspace, *sa)
    torch.ops.desmo_b200.fused_residual_grad(e.U, e.P, e.phi, e.omega, e.W, e.dphi, e.red, e.workspace, *sa)
    e.all_reduce()
    torch.ops.desmo_b200.adamax_update(e.red, e.dphi, e.P, e.phi, e.phi_m, e.phi_u, e.gates, e.gates_m, e.gates_u, e.rows, e.rows_m,
                                       e.rows_u, e.coefs, e.coefs_m, e.coefs_u, e.periods, e.periods_m, e.periods_u, e.omega, e.omega_m,
                                       e.omega_u, e.hyper, e.step_dev, e.losses, e.workspace, *sa)


def engine_term_norms_via_ops(e, physical: bool = False) -> torch.Tensor:
    sa = _shape_args(e)
    g2 = torch.zeros(e.K, dtype=torch.float32, device=e.device)
    out = torch.zeros(e.K, dtype=torch.float64, device=e.device)
    scratch_step = e.step_dev.clone()  # build_w advances the counter it is given; the optimizer's own one must not move
    torch.ops.desmo_b200.build_w(e.gates, e.rows, e.coefs, e.periods, e.W, scratch_step, e.workspace, *sa)
    torch.ops.desmo_b200.library_colnorm2(e.P if physical else None, e.phi, e.omega, g2, *sa)
    torch.ops.desmo_b200.term_norms(g2, e.gates, e.rows, 1 if (e.nF and not physical) else 0, out, *sa)
    return out


def engine_pod_via_ops(e) -> torch.Tensor:
    """POD init of the resident snapshot (CYL:197-205) through the registered pod_gram / pod_eig / pod_project ops."""
    sa = _shape_args(e)
    f32 = dict(dtype=torch.float32, device=e.device)
    Cm = torch.zeros(e.m, e.m, **f32)
    V, sigma = torch.zeros(e.r, e.m, **f32), torch.zeros(e.r, **f32)
    ws = torch.zeros(2 * 8 * 16 * e.m + 1024, dtype=torch.uint8, device=e.device)
    torch.ops.desmo_b200.pod_gram(e.U, Cm, e.workspace, *sa)
    if e.n_global != e.n and torch.distributed.is_initialized():
        torch.distributed.all_reduce(Cm, group=e.pg)
    torch.ops.desmo_b200.pod_eig(Cm, V, sigma, ws, e.m, e.r)
    torch.ops.desmo_b200.pod_project(e.U, V, sigma, e.P, *sa)
    return sigma
