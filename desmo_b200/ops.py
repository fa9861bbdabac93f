"""torch custom ops over the C ABI: one ``torch.ops.desmo_b200.*`` op per hot-path entry point of include/desmo_b200.h.

  build_w, build_w_at, fused_residual_grad, recon_backward, adamax_update, assemble_grads, reconstruct, residual_profile, pruning_profile, library_colnorm2, term_norms,
  pod_gram, pod_eig, pod_eigh, pod_project, preprocess, snapshot_to_bf16, plateau_step, peer_begin_step, peer_allreduce,
  active_terms_prepare, build_w_active, fused_residual_grad_active, adamax_update_active, assemble_grads_active,
  residual_gram, residual_modes, elimination_pass, elimination_greedy,
  time_points_prepare, build_w_times, adamax_update_times, assemble_grads_times

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


@torch.library.custom_op("desmo_b200::build_w_at", mutates_args=("W_out", "rows_out"))
def build_w_at(gates: torch.Tensor, rows: torch.Tensor, coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor],
               index: Optional[torch.Tensor], times: Optional[torch.Tensor], W_out: torch.Tensor, rows_out: Optional[torch.Tensor], n: int,
               n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """W_out [Kp, mld_out] (and rows_out [K, mld_out]) = diag(gates) z(t_i) at the instants of exactly one of index (int32, training
    snapshot indices) or times (fp32, Fourier models), both HOST tensors (desmo_build_w_at); m_out = their length, mld_out =
    W_out.shape[1].  Nothing the model owns is written."""
    _require_cuda(gates, rows, W_out, rows_out)
    inst = index if times is None else times
    if inst is None or (index is not None and times is not None):
        raise _lib.DesmoError("build_w_at: pass exactly one of index / times")
    want = torch.int32 if times is None else torch.float32
    if inst.device.type != "cpu" or inst.dtype != want or inst.dim() != 1 or not inst.is_contiguous():
        raise _lib.DesmoError(f"build_w_at: {'index' if times is None else 'times'} must be a contiguous 1-D {want} host tensor")
    if W_out.dtype != torch.float32 or W_out.dim() != 2 or not W_out.is_contiguous() or \
            (rows_out is not None and (rows_out.dtype != torch.float32 or not rows_out.is_contiguous() or rows_out.shape[-1] != W_out.shape[1])):
        raise _lib.DesmoError("build_w_at: W_out [Kp, mld_out] and rows_out [K, mld_out] must be contiguous float32")
    lib = _lib.load()
    Kp, K = lib.desmo_padded_k(r, polyorder), lib.desmo_num_terms(r, polyorder) + 3 * r
    if W_out.shape[0] < Kp or (rows_out is not None and rows_out.numel() < K * W_out.shape[1]):
        raise _lib.DesmoError(f"build_w_at: W_out needs {Kp} rows and rows_out {K}")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(gates.device):
        check(lib.desmo_build_w_at(C.byref(s), _p(gates), _p(rows), _p(coefs), _p(periods), inst.numel(), W_out.shape[1],
                                           _p(index), _p(times), _p(W_out), _p(rows_out), _stream(gates)), "desmo_build_w_at")


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


@torch.library.custom_op("desmo_b200::residual_profile", mutates_args=("snap", "point"))
def residual_profile(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, snap: torch.Tensor,
                     point: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """snap (fp64 [2, m]) = {sum_x r^2, sum_x U^2}, point (fp32 [2, ld]) = {sum_t r^2, sum_t U^2}, r = G W - U (desmo_residual_profile)."""
    _require_cuda(U, P, phi, omega, W, snap, point)
    ud = _lib.u_dtype_code(U.dtype)
    if snap.dtype != torch.float64 or point.dtype != torch.float32:
        raise _lib.DesmoError("residual_profile: snap must be float64 and point float32")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    if snap.numel() < 2 * m or point.numel() < 2 * s.ld or not (snap.is_contiguous() and point.is_contiguous()):
        raise _lib.DesmoError(f"residual_profile: need contiguous snap [2, {m}] and point [2, {s.ld}]")
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_residual_profile(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), _p(snap), _p(point), _stream(U)),
              "desmo_residual_profile")


@torch.library.custom_op("desmo_b200::pruning_profile", mutates_args=("snap", "norm"))
def pruning_profile(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, order: torch.Tensor,
                    snap: torch.Tensor, norm: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """snap (fp64 [S+1, m]) = sum_x r_s^2 with the terms order[0 .. s) removed, norm (fp64 [m]) = sum_x U^2 (desmo_pruning_profile).
    ``order`` is a host int32 tensor of S distinct term indices."""
    _require_cuda(U, P, phi, omega, W, snap, norm)
    ud = _lib.u_dtype_code(U.dtype)
    if order.device.type != "cpu" or order.dtype != torch.int32 or order.dim() != 1 or not order.is_contiguous():
        raise _lib.DesmoError("pruning_profile: order must be a contiguous 1-D int32 tensor on the host")
    S = order.numel()
    if snap.dtype != torch.float64 or norm.dtype != torch.float64:
        raise _lib.DesmoError("pruning_profile: snap and norm must be float64")
    if snap.numel() < (S + 1) * m or norm.numel() < m or not (snap.is_contiguous() and norm.is_contiguous()):
        raise _lib.DesmoError(f"pruning_profile: need contiguous snap [{S + 1}, {m}] and norm [{m}]")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_pruning_profile(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), S, _p(order) if S else None,
                                                _p(snap), _p(norm), _stream(U)), "desmo_pruning_profile")


def _scratch_ok(scratch: torch.Tensor, who: str) -> None:
    if scratch.dtype != torch.uint8 or not scratch.is_contiguous():
        raise _lib.DesmoError(f"{who}: scratch must be a contiguous uint8 tensor (desmo_residual_gram_scratch_bytes)")


@torch.library.custom_op("desmo_b200::residual_gram", mutates_args=("C_out", "trace", "scratch"))
def residual_gram(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, C_out: torch.Tensor,
                  trace: torch.Tensor, scratch: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """C_out (fp32 [m, m]) = C_R = R R^T of r = G W - U, trace (fp64 [1]) its trace (desmo_residual_gram)."""
    _require_cuda(U, P, phi, omega, W, C_out, trace, scratch)
    ud = _lib.u_dtype_code(U.dtype)
    if C_out.dtype != torch.float32 or trace.dtype != torch.float64 or C_out.numel() < m * m or not C_out.is_contiguous():
        raise _lib.DesmoError(f"residual_gram: need contiguous float32 C_out [{m}, {m}] and float64 trace [1]")
    _scratch_ok(scratch, "residual_gram")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_residual_gram(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), _p(C_out), _p(trace), _p(scratch),
                                              scratch.numel(), _stream(U)), "desmo_residual_gram")


@torch.library.custom_op("desmo_b200::residual_modes", mutates_args=("modes", "scratch"))
def residual_modes(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, V: torch.Tensor,
                   sigma: torch.Tensor, modes: torch.Tensor, scratch: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int,
                   nF: int, path: int) -> None:
    """modes (fp32 [k, ld]) row i = R^T V[i] / sigma[i] (zero when sigma_i = 0), k = V.shape[0] (desmo_residual_modes)."""
    _require_cuda(U, P, phi, omega, W, V, sigma, modes, scratch)
    ud = _lib.u_dtype_code(U.dtype)
    k = V.shape[0]
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    if V.dtype != torch.float32 or sigma.dtype != torch.float32 or modes.dtype != torch.float32 or V.numel() != k * m or \
            sigma.numel() < k or modes.numel() < k * s.ld or not (V.is_contiguous() and modes.is_contiguous()):
        raise _lib.DesmoError(f"residual_modes: need contiguous float32 V [k, {m}], sigma [k] and modes [k, {s.ld}]")
    _scratch_ok(scratch, "residual_modes")
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_residual_modes(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), k, _p(V), _p(sigma), _p(modes),
                                               _p(scratch), scratch.numel(), _stream(U)), "desmo_residual_modes")


@torch.library.custom_op("desmo_b200::elimination_pass", mutates_args=("A", "F", "r2", "scratch"))
def elimination_pass(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, A: torch.Tensor,
                     F: torch.Tensor, r2: torch.Tensor, scratch: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int,
                     nF: int, path: int) -> None:
    """A (fp64 [K, K]) = G^T G, F (fp64 [K, mld]) = G^T R, r2 (fp64 [1]) = ||R||_F^2 of R = G W - U (desmo_elimination_pass)."""
    _require_cuda(U, P, phi, omega, W, A, F, r2, scratch)
    ud = _lib.u_dtype_code(U.dtype)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    K = _lib.load().desmo_num_terms(r, polyorder) + 3 * r
    if any(t.dtype != torch.float64 or not t.is_contiguous() for t in (A, F, r2)) or A.numel() < K * K or F.numel() < K * s.mld or \
            r2.numel() < 1:
        raise _lib.DesmoError(f"elimination_pass: need contiguous float64 A [{K}, {K}], F [{K}, {s.mld}] and r2 [1]")
    _scratch_ok(scratch, "elimination_pass")
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_elimination_pass(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), _p(A), _p(F), _p(r2),
                                                 _p(scratch), scratch.numel(), _stream(U)), "desmo_elimination_pass")


@torch.library.custom_op("desmo_b200::elimination_greedy", mutates_args=("F", "order", "predicted", "scratch"))
def elimination_greedy(A: torch.Tensor, F: torch.Tensor, r2: torch.Tensor, W: torch.Tensor, order: torch.Tensor, predicted: torch.Tensor,
                       scratch: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """order (int32 [S]) and predicted (fp64 [S+1]) of the greedy on A, F (consumed), r2 and W, S = predicted.numel() - 1
    (desmo_elimination_greedy)."""
    _require_cuda(A, F, r2, W, order, predicted, scratch)
    S = predicted.numel() - 1
    if order.dtype != torch.int32 or predicted.dtype != torch.float64 or order.numel() < S or S < 0 or \
            not (order.is_contiguous() and predicted.is_contiguous()):
        raise _lib.DesmoError("elimination_greedy: need contiguous int32 order [S] and float64 predicted [S + 1]")
    _scratch_ok(scratch, "elimination_greedy")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(A.device):
        check(_lib.load().desmo_elimination_greedy(C.byref(s), _p(A), _p(F), _p(r2), _p(W), S, _p(order), _p(predicted), _p(scratch),
                                                   scratch.numel(), _stream(A)), "desmo_elimination_greedy")


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


@torch.library.custom_op("desmo_b200::pod_eigh", mutates_args=("S", "V", "sigma", "workspace"))
def pod_eigh(Cm: torch.Tensor, S: torch.Tensor, V: torch.Tensor, sigma: torch.Tensor, workspace: torch.Tensor, m: int, r: int) -> None:
    """All m singular values S (fp64) and the top r eigenpairs (V, sigma) of the Gram Cm (desmo_pod_eigh); report in workspace[:16]."""
    _require_cuda(Cm, S, V, sigma, workspace)
    with torch.cuda.device(Cm.device):
        check(_lib.load().desmo_pod_eigh(m, r, _p(Cm), _p(S), _p(V), _p(sigma), _p(workspace), workspace.numel() * workspace.element_size(),
                                         _stream(Cm)), "desmo_pod_eigh")


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


@torch.library.custom_op("desmo_b200::active_terms_prepare", mutates_args=("table",))
def active_terms_prepare(indices: torch.Tensor, table: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int,
                         path: int) -> None:
    """The device table of an active set (desmo_active_terms_prepare): ``indices`` a contiguous 1-D int32 HOST tensor of strictly
    increasing packed term indices, ``table`` an int32 device tensor of desmo_active_terms_bytes / 4 elements."""
    _require_cuda(table)
    if indices.device.type != "cpu" or indices.dtype != torch.int32 or indices.dim() != 1 or not indices.is_contiguous():
        raise _lib.DesmoError("active_terms_prepare: indices must be a contiguous 1-D int32 tensor on the host")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    nbytes = C.c_size_t(0)
    check(_lib.load().desmo_active_terms_bytes(C.byref(s), indices.numel(), C.byref(nbytes)), "desmo_active_terms_bytes")
    if table.dtype != torch.int32 or not table.is_contiguous() or table.numel() * 4 < nbytes.value:
        raise _lib.DesmoError(f"active_terms_prepare: table must be a contiguous int32 tensor of at least {nbytes.value // 4} elements")
    with torch.cuda.device(table.device):
        check(_lib.load().desmo_active_terms_prepare(C.byref(s), _p(indices), indices.numel(), _p(table), _stream(table)),
              "desmo_active_terms_prepare")


@torch.library.custom_op("desmo_b200::build_w_active", mutates_args=("rows", "W", "step", "workspace"))
def build_w_active(gates: torch.Tensor, rows: torch.Tensor, coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor], W: torch.Tensor,
                   step: torch.Tensor, workspace: torch.Tensor, active: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int,
                   nF: int, path: int) -> None:
    """build_w on an active set (desmo_build_w_active): absent rows of W are zero, the L1 sum takes the active gates."""
    _require_cuda(gates, rows, W, active)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(gates.device):
        check(_lib.load().desmo_build_w_active(C.byref(s), _p(gates), _p(rows), _p(coefs), _p(periods), _p(W), _p(step), _p(workspace),
                                               _p(active), _stream(gates)), "desmo_build_w_active")


@torch.library.custom_op("desmo_b200::fused_residual_grad_active", mutates_args=("dphi", "red", "workspace"))
def fused_residual_grad_active(U: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, omega: torch.Tensor, W: torch.Tensor, dphi: torch.Tensor,
                               red: torch.Tensor, workspace: torch.Tensor, active: torch.Tensor, active_count: int, n: int, n_global: int,
                               m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """fused_residual_grad on an active set of ``active_count`` terms (desmo_fused_residual_grad_active)."""
    _require_cuda(U, P, phi, omega, W, dphi, red, active)
    ud = _lib.u_dtype_code(U.dtype)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(U.device):
        check(_lib.load().desmo_fused_residual_grad_active(C.byref(s), _p(U), ud, _p(P), _p(phi), _p(omega), _p(W), _p(dphi), _p(red),
                                                           _p(workspace), _p(active), active_count, _stream(U)),
              "desmo_fused_residual_grad_active")


@torch.library.custom_op("desmo_b200::adamax_update_active",
                         mutates_args=("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "coefs", "coefs_m",
                                       "coefs_u", "periods", "periods_m", "periods_u", "omega", "omega_m", "omega_u", "losses", "workspace"))
def adamax_update_active(red: torch.Tensor, dphi: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, phi_m: torch.Tensor, phi_u: torch.Tensor,
                         gates: torch.Tensor, gates_m: torch.Tensor, gates_u: torch.Tensor, rows: torch.Tensor, rows_m: torch.Tensor,
                         rows_u: torch.Tensor, coefs: Optional[torch.Tensor], coefs_m: Optional[torch.Tensor], coefs_u: Optional[torch.Tensor],
                         periods: Optional[torch.Tensor], periods_m: Optional[torch.Tensor], periods_u: Optional[torch.Tensor],
                         omega: torch.Tensor, omega_m: torch.Tensor, omega_u: torch.Tensor, hyper: torch.Tensor, step: torch.Tensor,
                         losses: torch.Tensor, workspace: torch.Tensor, active: torch.Tensor, n: int, n_global: int, m: int, r: int,
                         polyorder: int, nF: int, path: int) -> None:
    """adamax_update on an active set (desmo_adamax_update_active): absent terms' parameters and Adamax state are not written."""
    _require_cuda(red, dphi, P, phi, gates, rows, omega, hyper, step, losses, active)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_adamax_update_active(
            C.byref(s), _p(red), _p(dphi), _p(P), _p(phi), _p(phi_m), _p(phi_u), _p(gates), _p(gates_m), _p(gates_u), _p(rows), _p(rows_m),
            _p(rows_u), _p(coefs), _p(coefs_m), _p(coefs_u), _p(periods), _p(periods_m), _p(periods_u), _p(omega), _p(omega_m), _p(omega_u),
            _p(hyper), _p(step), _p(losses), _p(workspace), _p(active), _stream(phi)), "desmo_adamax_update_active")


@torch.library.custom_op("desmo_b200::assemble_grads_active",
                         mutates_args=("dphi", "d_gates", "d_rows", "d_coefs", "d_periods", "d_omega", "losses", "workspace"))
def assemble_grads_active(red: torch.Tensor, dphi: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, gates: torch.Tensor, rows: torch.Tensor,
                          coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor], hyper: torch.Tensor, d_gates: torch.Tensor,
                          d_rows: Optional[torch.Tensor], d_coefs: Optional[torch.Tensor], d_periods: Optional[torch.Tensor],
                          d_omega: torch.Tensor, losses: torch.Tensor, workspace: torch.Tensor, active: torch.Tensor, n: int, n_global: int,
                          m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """assemble_grads on an active set (desmo_assemble_grads_active): absent terms' gradients are exactly 0."""
    _require_cuda(red, dphi, P, phi, gates, rows, hyper, d_gates, d_omega, losses, active)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_assemble_grads_active(
            C.byref(s), _p(red), _p(dphi), _p(P), _p(phi), _p(gates), _p(rows), _p(coefs), _p(periods), _p(hyper), _p(d_gates), _p(d_rows),
            _p(d_coefs), _p(d_periods), _p(d_omega), _p(losses), _p(workspace), _p(active), _stream(phi)), "desmo_assemble_grads_active")


@torch.library.custom_op("desmo_b200::time_points_prepare", mutates_args=("table",))
def time_points_prepare(times: torch.Tensor, table: torch.Tensor, n: int, n_global: int, m: int, r: int, polyorder: int, nF: int,
                        path: int) -> None:
    """The device time table of a Fourier model (desmo_time_points_prepare): ``times`` a contiguous 1-D float32 HOST tensor of m finite
    values, ``table`` a float32 device tensor of m elements."""
    _require_cuda(table)
    if times.device.type != "cpu" or times.dtype != torch.float32 or times.dim() != 1 or not times.is_contiguous():
        raise _lib.DesmoError("time_points_prepare: times must be a contiguous 1-D float32 tensor on the host")
    if table.dtype != torch.float32 or not table.is_contiguous() or table.numel() < m:
        raise _lib.DesmoError(f"time_points_prepare: table must be a contiguous float32 tensor of at least {m} elements")
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(table.device):
        check(_lib.load().desmo_time_points_prepare(C.byref(s), _p(times), times.numel(), _p(table), _stream(table)),
              "desmo_time_points_prepare")


@torch.library.custom_op("desmo_b200::build_w_times", mutates_args=("rows", "W", "step", "workspace"))
def build_w_times(gates: torch.Tensor, rows: torch.Tensor, coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor], W: torch.Tensor,
                  step: torch.Tensor, workspace: torch.Tensor, active: Optional[torch.Tensor], t_points: Optional[torch.Tensor], n: int,
                  n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """build_w with an optional active set and an optional time table (desmo_build_w_times)."""
    _require_cuda(gates, rows, W)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(gates.device):
        check(_lib.load().desmo_build_w_times(C.byref(s), _p(gates), _p(rows), _p(coefs), _p(periods), _p(W), _p(step), _p(workspace),
                                              _p(active), _p(t_points), _stream(gates)), "desmo_build_w_times")


@torch.library.custom_op("desmo_b200::adamax_update_times",
                         mutates_args=("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "coefs", "coefs_m",
                                       "coefs_u", "periods", "periods_m", "periods_u", "omega", "omega_m", "omega_u", "losses", "workspace"))
def adamax_update_times(red: torch.Tensor, dphi: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, phi_m: torch.Tensor, phi_u: torch.Tensor,
                        gates: torch.Tensor, gates_m: torch.Tensor, gates_u: torch.Tensor, rows: torch.Tensor, rows_m: torch.Tensor,
                        rows_u: torch.Tensor, coefs: Optional[torch.Tensor], coefs_m: Optional[torch.Tensor], coefs_u: Optional[torch.Tensor],
                        periods: Optional[torch.Tensor], periods_m: Optional[torch.Tensor], periods_u: Optional[torch.Tensor],
                        omega: torch.Tensor, omega_m: torch.Tensor, omega_u: torch.Tensor, hyper: torch.Tensor, step: torch.Tensor,
                        losses: torch.Tensor, workspace: torch.Tensor, active: Optional[torch.Tensor], t_points: Optional[torch.Tensor],
                        n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """adamax_update with an optional active set and an optional time table (desmo_adamax_update_times)."""
    _require_cuda(red, dphi, P, phi, gates, rows, omega, hyper, step, losses)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_adamax_update_times(
            C.byref(s), _p(red), _p(dphi), _p(P), _p(phi), _p(phi_m), _p(phi_u), _p(gates), _p(gates_m), _p(gates_u), _p(rows), _p(rows_m),
            _p(rows_u), _p(coefs), _p(coefs_m), _p(coefs_u), _p(periods), _p(periods_m), _p(periods_u), _p(omega), _p(omega_m), _p(omega_u),
            _p(hyper), _p(step), _p(losses), _p(workspace), _p(active), _p(t_points), _stream(phi)), "desmo_adamax_update_times")


@torch.library.custom_op("desmo_b200::assemble_grads_times",
                         mutates_args=("dphi", "d_gates", "d_rows", "d_coefs", "d_periods", "d_omega", "losses", "workspace"))
def assemble_grads_times(red: torch.Tensor, dphi: torch.Tensor, P: torch.Tensor, phi: torch.Tensor, gates: torch.Tensor, rows: torch.Tensor,
                         coefs: Optional[torch.Tensor], periods: Optional[torch.Tensor], hyper: torch.Tensor, d_gates: torch.Tensor,
                         d_rows: Optional[torch.Tensor], d_coefs: Optional[torch.Tensor], d_periods: Optional[torch.Tensor],
                         d_omega: torch.Tensor, losses: torch.Tensor, workspace: torch.Tensor, active: Optional[torch.Tensor],
                         t_points: Optional[torch.Tensor], n: int, n_global: int, m: int, r: int, polyorder: int, nF: int, path: int) -> None:
    """assemble_grads with an optional active set and an optional time table (desmo_assemble_grads_times)."""
    _require_cuda(red, dphi, P, phi, gates, rows, hyper, d_gates, d_omega, losses)
    s = make_shape(n, m, r, polyorder, nF, n_global, path)
    with torch.cuda.device(phi.device):
        check(_lib.load().desmo_assemble_grads_times(
            C.byref(s), _p(red), _p(dphi), _p(P), _p(phi), _p(gates), _p(rows), _p(coefs), _p(periods), _p(hyper), _p(d_gates), _p(d_rows),
            _p(d_coefs), _p(d_periods), _p(d_omega), _p(losses), _p(workspace), _p(active), _p(t_points), _stream(phi)),
            "desmo_assemble_grads_times")


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


def _build_w_op(e, step, sa) -> None:
    """W of the engine's current parameters through the build_w op, or build_w_times at the engine's time table."""
    if e._times is not None:
        torch.ops.desmo_b200.build_w_times(e.gates, e.rows, e.coefs, e.periods, e.W, step, e.workspace, None, e._times, *sa)
    else:
        torch.ops.desmo_b200.build_w(e.gates, e.rows, e.coefs, e.periods, e.W, step, e.workspace, *sa)


def engine_step_via_ops(e) -> None:
    """One train step of a DesmoEngine routed entirely through the registered ops (on its active set and at its time table, if set)."""
    sa = _shape_args(e)
    opt = (e.red, e.dphi, e.P, e.phi, e.phi_m, e.phi_u, e.gates, e.gates_m, e.gates_u, e.rows, e.rows_m, e.rows_u, e.coefs, e.coefs_m,
           e.coefs_u, e.periods, e.periods_m, e.periods_u, e.omega, e.omega_m, e.omega_u, e.hyper, e.step_dev, e.losses, e.workspace)
    if e._times is not None:
        torch.ops.desmo_b200.build_w_times(e.gates, e.rows, e.coefs, e.periods, e.W, e.step_dev, e.workspace, e._active, e._times, *sa)
        if e._active is not None:
            torch.ops.desmo_b200.fused_residual_grad_active(e.U, e.P, e.phi, e.omega, e.W, e.dphi, e.red, e.workspace, e._active,
                                                            e._active_count, *sa)
        else:
            torch.ops.desmo_b200.fused_residual_grad(e.U, e.P, e.phi, e.omega, e.W, e.dphi, e.red, e.workspace, *sa)
        e.all_reduce()
        torch.ops.desmo_b200.adamax_update_times(*opt, e._active, e._times, *sa)
        return
    if e._active is not None:
        torch.ops.desmo_b200.build_w_active(e.gates, e.rows, e.coefs, e.periods, e.W, e.step_dev, e.workspace, e._active, *sa)
        torch.ops.desmo_b200.fused_residual_grad_active(e.U, e.P, e.phi, e.omega, e.W, e.dphi, e.red, e.workspace, e._active,
                                                        e._active_count, *sa)
        e.all_reduce()
        torch.ops.desmo_b200.adamax_update_active(*opt, e._active, *sa)
        return
    torch.ops.desmo_b200.build_w(e.gates, e.rows, e.coefs, e.periods, e.W, e.step_dev, e.workspace, *sa)
    torch.ops.desmo_b200.fused_residual_grad(e.U, e.P, e.phi, e.omega, e.W, e.dphi, e.red, e.workspace, *sa)
    e.all_reduce()
    torch.ops.desmo_b200.adamax_update(*opt, *sa)


def engine_term_norms_via_ops(e, physical: bool = False) -> torch.Tensor:
    sa = _shape_args(e)
    g2 = torch.zeros(e.K, dtype=torch.float32, device=e.device)
    out = torch.zeros(e.K, dtype=torch.float64, device=e.device)
    scratch_step = e.step_dev.clone()  # build_w advances the counter it is given; the optimizer's own one must not move
    _build_w_op(e, scratch_step, sa)
    torch.ops.desmo_b200.library_colnorm2(e.P if physical else None, e.phi, e.omega, g2, *sa)
    torch.ops.desmo_b200.term_norms(g2, e.gates, e.rows, 1 if (e.nF and not physical) else 0, out, *sa)
    return out


def engine_residual_profile_via_ops(e) -> dict:
    """DesmoEngine.residual_profile() through the registered build_w / residual_profile ops (the optimizer's step counter is not moved)."""
    sa = _shape_args(e)
    snap = torch.empty(2, e.m, dtype=torch.float64, device=e.device)
    point = torch.empty(2, e.ld, dtype=torch.float32, device=e.device)
    scratch_step = e.step_dev.clone()
    _build_w_op(e, scratch_step, sa)
    torch.ops.desmo_b200.residual_profile(e.U, e.P, e.phi, e.omega, e.W, snap, point, *sa)
    if e.n_global != e.n and torch.distributed.is_initialized():
        torch.distributed.all_reduce(snap, group=e.pg)
    return {"snapshot_residual2": snap[0], "snapshot_norm2": snap[1], "point_residual2": point[0, :e.n], "point_norm2": point[1, :e.n]}


def engine_pruning_profile_via_ops(e, order) -> dict:
    """DesmoEngine.pruning_profile() through the registered build_w / pruning_profile ops (the optimizer's step counter is not moved)."""
    from .engine import pruning_order

    sa = _shape_args(e)
    idx = torch.from_numpy(pruning_order(order, e.K))
    snap = torch.empty(idx.numel() + 1, e.m, dtype=torch.float64, device=e.device)
    norm = torch.empty(e.m, dtype=torch.float64, device=e.device)
    scratch_step = e.step_dev.clone()
    _build_w_op(e, scratch_step, sa)
    torch.ops.desmo_b200.pruning_profile(e.U, e.P, e.phi, e.omega, e.W, idx, snap, norm, *sa)
    if e.n_global != e.n and torch.distributed.is_initialized():
        torch.distributed.all_reduce(snap, group=e.pg)
        torch.distributed.all_reduce(norm, group=e.pg)
    return {"snapshot_residual2": snap, "snapshot_norm2": norm}


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


def engine_pod_analysis_via_ops(e) -> torch.Tensor:
    """DesmoEngine.pod_analysis() through the registered pod_gram / pod_eigh / pod_project ops: returns sigma, fills e.P (untouched when
    the solver's report is not OK)."""
    sa = _shape_args(e)
    f32 = dict(dtype=torch.float32, device=e.device)
    Cm = torch.zeros(e.m, e.m, **f32)
    V, sigma = torch.zeros(e.r, e.m, **f32), torch.zeros(e.r, **f32)
    S = torch.zeros(e.m, dtype=torch.float64, device=e.device)
    ws = e._eigh_workspace()
    torch.ops.desmo_b200.pod_gram(e.U, Cm, e.workspace, *sa)
    if e.n_global != e.n and torch.distributed.is_initialized():
        torch.distributed.all_reduce(Cm, group=e.pg)
    torch.ops.desmo_b200.pod_eigh(Cm, S, V, sigma, ws, e.m, e.r)
    status, residual = int(ws[:4].view(torch.int32).item()), float(ws[8:16].view(torch.float64).item())
    if status != 0 or not residual <= 2.0 ** -27:
        raise _lib.DesmoError(f"desmo_pod_eigh failed (status {status}, residual {residual:.2e} lambda_1); P is unchanged")
    torch.ops.desmo_b200.pod_project(e.U, V, sigma, e.P, *sa)
    return sigma


def engine_residual_pod_via_ops(e, k: int = 8) -> dict:
    """DesmoEngine.residual_pod(k) through the registered build_w / residual_gram / pod_eigh / residual_modes ops (the optimizer's step
    counter is not moved)."""
    sa = _shape_args(e)
    f32 = dict(dtype=torch.float32, device=e.device)
    scratch = e._residual_pod_scratch()
    Cm, tr = torch.empty(e.m, e.m, **f32), torch.empty(1, dtype=torch.float64, device=e.device)
    V, sigma, modes = torch.zeros(k, e.m, **f32), torch.zeros(k, **f32), torch.zeros(k, e.ld, **f32)
    S = torch.zeros(e.m, dtype=torch.float64, device=e.device)
    scratch_step = e.step_dev.clone()
    _build_w_op(e, scratch_step, sa)
    torch.ops.desmo_b200.residual_gram(e.U, e.P, e.phi, e.omega, e.W, Cm, tr, scratch, *sa)
    if e.n_global != e.n and torch.distributed.is_initialized():
        torch.distributed.all_reduce(Cm, group=e.pg)
        torch.distributed.all_reduce(tr, group=e.pg)
    if float(tr.item()) > 0.0:
        nbytes = C.c_size_t(0)
        check(_lib.load().desmo_pod_eigh_workspace_bytes(e.m, k, C.byref(nbytes)), "desmo_pod_eigh_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=e.device)
        torch.ops.desmo_b200.pod_eigh(Cm, S, V, sigma, ws, e.m, k)
        status, residual = int(ws[:4].view(torch.int32).item()), float(ws[8:16].view(torch.float64).item())
        if status != 0 or not residual <= 2.0 ** -27:
            raise _lib.DesmoError(f"residual_pod: desmo_pod_eigh failed (status {status}, residual {residual:.2e} lambda_1)")
        torch.ops.desmo_b200.residual_modes(e.U, e.P, e.phi, e.omega, e.W, V, sigma, modes, scratch, *sa)
    return {"singular_values": S.cpu(), "sigma": sigma, "temporal_modes": V, "spatial_modes": modes[:, :e.n], "residual_norm2": float(tr.item()),
            "gram": Cm}


def engine_backward_elimination_via_ops(e, steps=None) -> dict:
    """DesmoEngine.backward_elimination() through the registered build_w / elimination_pass / elimination_greedy ops (the optimizer's
    step counter is not moved)."""
    sa = _shape_args(e)
    S = e.K if steps is None else int(steps)
    f64 = dict(dtype=torch.float64, device=e.device)
    scratch = e._elimination_scratch()
    A, F, r2 = torch.empty(e.K, e.K, **f64), torch.empty(e.K, e.mld, **f64), torch.empty(1, **f64)
    order, pred = torch.empty(max(S, 1), dtype=torch.int32, device=e.device), torch.empty(S + 1, **f64)
    scratch_step = e.step_dev.clone()
    _build_w_op(e, scratch_step, sa)
    torch.ops.desmo_b200.elimination_pass(e.U, e.P, e.phi, e.omega, e.W, A, F, r2, scratch, *sa)
    if e.n_global != e.n and torch.distributed.is_initialized():
        for t in (A, F, r2):
            torch.distributed.all_reduce(t, group=e.pg)
    torch.ops.desmo_b200.elimination_greedy(A, F, r2, e.W, order, pred, scratch, *sa)
    return {"order": order[:S].cpu().long(), "predicted_residual2": pred, "gram": A}
