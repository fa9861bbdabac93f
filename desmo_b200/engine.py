"""Device-resident packed state of one DESMO model shard and the per-step launch sequence.

PyTorch is used for memory, streams, CUDA graphs and torch.distributed only; all arithmetic is in libdesmo_b200.so.
Layout: see include/desmo_b200.h.  One step = build_w -> fused_residual_grad -> [all_reduce(red)] -> adamax_update,
i.e. the body of the reference loop CYL:711-768 for one full batch.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import check, make_shape, round_up

REFERENCE_LRS = (1e-2, 1e-3, 1e-2, 1e3, 1e-2)  # gates, phi, z, omega, periods  (CYL:592-612, FCYL:628-631)
SNAPSHOT_CHUNK_BYTES = 256 << 20  # fp32 staging per chunk when set_snapshot converts into bf16 storage


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def time_points(index, m: int) -> np.ndarray:
    """The fp32 times at which a model with m snapshots evaluates training snapshot k = index[i]: t_point of csrc/library.cu, i.e.
    torch.linspace(0, m, m)[k] as ATen computes it (FCYL:485).  step = m / (m - 1); k < m / 2 gives step * k, otherwise
    m - step * (m - 1 - k).  k >= m continues the grid as step * k, so time_points(range(m, 2 * m), m) is the next window at the
    training spacing.  Every operation is one fp32 rounding, as on the device."""
    m = int(m)
    if m < 2:
        raise _lib.DesmoError(f"time_points needs m >= 2, got {m}")
    k = np.asarray(index, dtype=np.int64).reshape(-1)
    if k.size and int(k.min()) < 0:
        raise _lib.DesmoError("time_points: negative snapshot index")
    step = np.float32(m) / np.float32(m - 1)
    up = step * k.astype(np.float32)
    down = np.float32(m) - step * (m - 1 - k).astype(np.float32)
    return np.where((k < m // 2) | (k >= m), up, down).astype(np.float32)


def _instants(index, times, m: int, nF: int):
    """Host arrays for desmo_build_w_at: (int32 index or None, fp32 times or None).  Raises DesmoError before any launch."""
    if (index is None) == (times is None):
        raise _lib.DesmoError("pass exactly one of index= (training snapshot indices) or times= (Fourier model times)")
    if times is not None:
        if not nF:
            raise _lib.DesmoError("times= needs a Fourier model: DESMO's free temporal rows exist only at the m training snapshots")
        t = np.ascontiguousarray((times.detach().cpu().numpy() if torch.is_tensor(times) else np.asarray(times)), dtype=np.float32).reshape(-1)
        if t.size == 0:
            raise _lib.DesmoError("times= is empty")
        if not np.isfinite(t).all():
            raise _lib.DesmoError("times= must be finite")
        return None, t
    raw = index.detach().cpu().numpy() if torch.is_tensor(index) else np.asarray(index)
    if raw.size == 0:
        raise _lib.DesmoError("index= is empty")
    if not np.issubdtype(raw.dtype, np.integer):
        raise _lib.DesmoError(f"index= must hold integers, got {raw.dtype}")
    k = raw.astype(np.int64).reshape(-1)
    if int(k.min()) < 0 or int(k.max()) >= m:
        raise _lib.DesmoError(f"index= must lie in 0 .. {m - 1} (training snapshots; use times= to evaluate elsewhere)")
    return np.ascontiguousarray(k, dtype=np.int32), None


class _PeerDesc(C.Structure):  # desmo_peer (include/desmo_b200.h)
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("red_ptrs", C.c_void_p), ("flag_ptrs", C.c_void_p), ("state", C.c_void_p)]


class DesmoEngine:
    """``snapshot_dtype``: storage of the snapshot matrix U -- torch.float32 (default) or torch.bfloat16.  bf16 storage halves U's
    memory and HBM traffic; every kernel widens it exactly to fp32, so training on it is bit-identical to fp32 storage of
    U_q.float(), U_q = the snapshot rounded to bf16 (see snapshot_quantization_error).  fp16 is rejected: snapshots in physical units
    would need a per-tensor scale to stay clear of its overflow / subnormal range; bf16 has fp32's range."""

    def __init__(self, n: int, m: int, polyorder: int, r: int, omega_init: float = 10000.0, nF: Optional[int] = None,
                 period_init: float = 60.0, device: Optional[torch.device] = None, n_global: Optional[int] = None,
                 path: int = _lib.PATH_AUTO, process_group=None, snapshot_dtype: torch.dtype = torch.float32):
        if snapshot_dtype not in (torch.float32, torch.bfloat16):
            raise _lib.DesmoError(f"snapshot_dtype must be torch.float32 or torch.bfloat16, got {snapshot_dtype}")
        self.snapshot_dtype = snapshot_dtype
        self.lib = _lib.load()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
        if device is None or torch.device(device).type != "cuda":
            raise _lib.DesmoError("desmo_b200 needs a CUDA (sm_100a) device; there is no CPU fallback")
        self.device = torch.device(device)
        self.n, self.m, self.r, self.polyorder = int(n), int(m), int(r), int(polyorder)
        self.nF = int(nF) if nF else 0
        self.T = self.lib.desmo_num_terms(self.r, self.polyorder)
        if self.T < 0:
            raise _lib.DesmoError(f"unsupported library r={r} polyorder={polyorder} (K must be <= {_lib.MAX_K})")
        self.K = self.T + 3 * self.r
        self.Kp = self.lib.desmo_padded_k(self.r, self.polyorder)
        self.pg = process_group
        self.n_global = int(n_global) if n_global else self.n
        self.shape = make_shape(self.n, self.m, self.r, self.polyorder, self.nF, self.n_global, path)
        self.ld, self.mld = self.shape.ld, self.shape.mld
        self.path_used = int(self.lib.desmo_selected_path(C.byref(self.shape)))  # 1 FFMA, 2 fused tcgen05, 3 tcgen05 GEMM path
        if self.path_used < 0:
            raise _lib.DesmoError(self.lib.desmo_last_error().decode(errors="replace"))
        f32 = dict(dtype=torch.float32, device=self.device)
        z = lambda *s: torch.zeros(*s, **f32)  # noqa: E731
        self.U: Optional[torch.Tensor] = None
        self._qsums: Optional[torch.Tensor] = None  # fp64 [sum (u - q)^2, sum u^2] of the last bf16 conversion of U
        self.P = z(self.r, self.ld)
        self.phi, self.phi_m, self.phi_u, self.dphi = z(self.r, self.ld), z(self.r, self.ld), z(self.r, self.ld), z(self.r, self.ld)
        self.phi[:, :self.n] = 1.0
        self.gates, self.gates_m, self.gates_u = torch.ones(self.K, **f32), z(self.K), z(self.K)
        self.rows, self.rows_m, self.rows_u = z(self.K, self.mld), z(self.K, self.mld), z(self.K, self.mld)
        self.coefs = self.coefs_m = self.coefs_u = self.periods = self.periods_m = self.periods_u = None
        if self.nF:
            w = 2 * self.nF + 1
            self.coefs, self.coefs_m, self.coefs_u = torch.ones(self.K, w, **f32), z(self.K, w), z(self.K, w)
            self.periods, self.periods_m, self.periods_u = torch.full((self.K,), float(period_init), **f32), z(self.K), z(self.K)
        else:
            self.rows[:, :self.m] = 1.0
        self.omega, self.omega_m, self.omega_u = torch.full((3 * self.r,), float(omega_init), **f32), z(3 * self.r), z(3 * self.r)
        self.W = z(self.Kp, self.mld)
        cnt = int(self.lib.desmo_red_count(C.byref(self.shape)))
        self._red_pad = z((cnt + 3) // 4 * 4)   # the peer exchange moves float4s
        self.red = self._red_pad[:cnt]
        self.red_local: Optional[torch.Tensor] = None   # peer mode: this rank's contribution, in peer-mapped memory
        self._peer: Optional[_PeerDesc] = None
        self.peer_status = "off"
        self.plateau_state: Optional[torch.Tensor] = None   # desmo_plateau on the device (DesmoTrainer(device_scheduler=True))
        self.hyper = z(_lib.HYP_COUNT)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.losses = z(4)
        nbytes = C.c_size_t(0)
        with torch.cuda.device(self.device):
            check(self.lib.desmo_workspace_bytes(C.byref(self.shape), C.byref(nbytes)), "desmo_workspace_bytes")
        self.workspace = torch.zeros(nbytes.value, dtype=torch.uint8, device=self.device)
        self.launches_per_step = 0
        self._side: Optional[torch.cuda.Stream] = None
        self.set_hyper(REFERENCE_LRS, 1e-3, 1e-4)

    # ------------------------------------------------------------------ inputs
    def set_pod_modes(self, pod_modes) -> None:
        """POD_modes[:, :r] (n x >=r, numpy fp64 or tensor) -> fp32 mode-major, as CYL:538-541 casts them per forward."""
        pm = torch.as_tensor(np.asarray(pod_modes)[:, :self.r] if not torch.is_tensor(pod_modes) else pod_modes[:, :self.r])
        if pm.shape != (self.n, self.r):
            raise ValueError(f"POD modes must be ({self.n}, >={self.r}), got {tuple(pm.shape)}")
        self.P.zero_()
        self.P[:, :self.n] = pm.to(torch.float32).t().to(self.device)

    def set_snapshot(self, snapshot: torch.Tensor, non_blocking: bool = True) -> None:
        """The reference's (m, n) batch (CYL:708).  Host tensors are uploaded; any float dtype is cast to fp32.

        bf16 storage: bf16 input is stored as it is; fp32 / fp64 input is rounded to bf16 (nearest even) by desmo_snapshot_to_bf16
        in chunks of at most SNAPSHOT_CHUNK_BYTES of fp32, so the device never holds an fp32 copy of the whole matrix."""
        if tuple(snapshot.shape) != (self.m, self.n):
            raise ValueError(f"snapshot must be ({self.m}, {self.n}) like the reference batch, got {tuple(snapshot.shape)}")
        if self.U is None or self.U.dtype != self.snapshot_dtype:
            self.U = torch.zeros(self.m, self.ld, dtype=self.snapshot_dtype, device=self.device)
        if self.snapshot_dtype == torch.float32:
            self.U[:, :self.n].copy_(snapshot, non_blocking=non_blocking)
            return
        if snapshot.dtype == torch.bfloat16:
            self.U[:, :self.n].copy_(snapshot, non_blocking=non_blocking)
            self._qsums = None  # nothing was rounded
            return
        if snapshot.dtype not in (torch.float32, torch.float64):
            raise _lib.DesmoError(f"bf16 storage takes fp32, fp64 or bf16 snapshots, got {snapshot.dtype}")
        self._qsums = self._snapshot_to_bf16(snapshot, self.U, self.shape, non_blocking)

    def _snapshot_to_bf16(self, snapshot: torch.Tensor, U: torch.Tensor, shape, non_blocking: bool) -> torch.Tensor:
        """fp32 / fp64 snapshot (rows, n) -> bf16 U[0 .. rows)[ld] of `shape` by desmo_snapshot_to_bf16, in chunks of at most
        SNAPSHOT_CHUNK_BYTES of fp32.  Returns the fp64 quantisation sums [sum (u - q)^2, sum u^2]."""
        qsums = torch.zeros(2, dtype=torch.float64, device=self.device)
        rows = max(1, min(snapshot.shape[0], SNAPSHOT_CHUNK_BYTES // (4 * self.n)))
        with torch.cuda.device(self.device):
            for t0 in range(0, snapshot.shape[0], rows):
                part = snapshot[t0:t0 + rows]
                if part.dtype != torch.float32 and part.device.type == "cpu":
                    part = part.to(torch.float32)  # cast on the host: only fp32 crosses the bus
                src = part.to(self.device, torch.float32, non_blocking=non_blocking).contiguous()
                check(self.lib.desmo_snapshot_to_bf16(C.byref(shape), src.data_ptr(), src.stride(0), t0, src.shape[0],
                                                      U.data_ptr(), qsums.data_ptr(), self._stream()),
                      "desmo_snapshot_to_bf16")
                del part, src  # the next chunk reuses this block: at most one chunk is resident
        return qsums

    def snapshot_quantization_error(self) -> float:
        """||U - U_q||_F / ||U||_F of the bf16 snapshot storage (fp64; over all ranks when point-sharded): U the fp32 snapshot the
        fp32 path would train on, U_q what is stored.  0.0 for fp32 storage or a snapshot given in bf16."""
        if self.U is None:
            raise _lib.DesmoError("no snapshot matrix set")
        if self._qsums is None or self.U.dtype != torch.bfloat16:
            return 0.0
        q = self._qsums.clone()
        if self._sharded():
            torch.distributed.all_reduce(q, group=self.pg)
        e2, u2 = q.tolist()
        return (e2 / u2) ** 0.5 if u2 > 0 else 0.0

    def _u_dtype(self) -> int:
        if self.U is None:
            raise _lib.DesmoError("no snapshot matrix set (call set_snapshot)")
        return _lib.u_dtype_code(self.U.dtype)

    def set_hyper(self, lrs: Sequence[float], beta: float, l1_lambda: float) -> None:
        vals = list(lrs) + [REFERENCE_LRS[4]] * (5 - len(lrs)) + [beta, l1_lambda]
        self.hyper_host = [float(v) for v in vals]
        self.hyper.copy_(torch.tensor(self.hyper_host, dtype=torch.float32), non_blocking=False)

    def _refresh_hyper_host(self) -> None:
        """A device-side scheduler (desmo_plateau_step) lowers the learning rates in ``hyper`` without the host knowing: re-read them
        before code that saves / restores the hyper-parameters through the host mirror."""
        if self.plateau_state is not None:
            self.hyper_host = [float(v) for v in self.hyper.tolist()]

    def reset_optimizer(self) -> None:
        for t in (self.phi_m, self.phi_u, self.gates_m, self.gates_u, self.rows_m, self.rows_u, self.omega_m, self.omega_u,
                  self.coefs_m, self.coefs_u, self.periods_m, self.periods_u):
            if t is not None:
                t.zero_()
        self.step_dev.zero_()

    # ------------------------------------------------------------------ launches
    def uses_tensor_cores(self) -> bool:
        """True when desmo_fused_residual_grad dispatches to a tcgen05 implementation (fused kernel or GEMM path)."""
        return self.path_used in (_lib.PATH_TC, _lib.PATH_GEMM)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def build_w(self, advance_step: bool = True) -> None:
        check(self.lib.desmo_build_w(C.byref(self.shape), _ptr(self.gates), _ptr(self.rows), _ptr(self.coefs), _ptr(self.periods),
                                     _ptr(self.W), _ptr(self.step_dev) if advance_step else None, _ptr(self.workspace),
                                     self._stream()), "desmo_build_w")

    def fused_residual_grad(self, red: Optional[torch.Tensor] = None) -> None:
        ud = self._u_dtype()
        check(self.lib.desmo_fused_residual_grad_ex(C.byref(self.shape), _ptr(self.U), ud, _ptr(self.P), _ptr(self.phi), _ptr(self.omega),
                                                    _ptr(self.W), _ptr(self.dphi), _ptr(self.red if red is None else red),
                                                    _ptr(self.workspace), self._stream()),
              "desmo_fused_residual_grad")

    def enable_peer_allreduce(self, group=None) -> bool:
        """Point-sharded runs on one node: replaces the two NCCL all-reduces of the train step by the one-shot exchange over NVLink /
        NVSwitch peer memory (csrc/peer.cu: every rank reads all ranks' `red` directly and adds them in rank order).  Collective: every
        rank of the group must call it.  Returns False -- and the step keeps using NCCL -- when peer-mapped (symmetric) memory is not
        available; ``peer_status`` says why."""
        import torch.distributed as dist

        if not self._sharded():
            self.peer_status = "off (not sharded)"
            return False
        pg = group or self.pg or dist.group.WORLD
        world, rank = dist.get_world_size(pg), dist.get_rank(pg)
        ok = torch.ones(1, device=self.device)
        sym = hdl = None
        why = ""
        try:
            import torch.distributed._symmetric_memory as symm

            if world > 16:
                raise RuntimeError("more than DESMO_MAX_PEERS ranks")
            cnt4 = self._red_pad.numel()
            sym = symm.empty(cnt4 + 64, dtype=torch.float32, device=self.device)  # [red | 2 * world uint32 flags]
            sym.zero_()
            hdl = symm.rendezvous(sym, pg.group_name)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            if len(ptrs) != world or any(p == 0 for p in ptrs):
                raise RuntimeError("rendezvous returned no peer pointers")
        except Exception as ex:  # noqa: BLE001  (any failure of the optional transport keeps the NCCL path)
            ok.zero_()
            why = f"{type(ex).__name__}: {ex}"
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=pg)  # all ranks or none
        if float(ok.item()) < 1.0:
            self.peer_status = "off (symmetric memory unavailable" + (": " + why if why else " on a peer") + ")"
            return False
        cnt4 = self._red_pad.numel()
        self._peer_keep = (sym, hdl,
                           torch.tensor(ptrs + [p + 4 * cnt4 for p in ptrs], dtype=torch.int64, device=self.device),
                           torch.zeros(2, dtype=torch.int32, device=self.device))
        tbl, state = self._peer_keep[2], self._peer_keep[3]
        self.red_local = sym[:self.red.numel()]
        self._peer = _PeerDesc(world, rank, tbl.data_ptr(), tbl.data_ptr() + 8 * world, state.data_ptr())
        torch.cuda.synchronize(self.device)
        dist.barrier(group=pg)  # every pad is zeroed before anybody signals
        self.peer_status = f"on ({world} ranks, one-shot exchange over peer memory)"
        return True

    def all_reduce(self) -> None:
        if self.pg is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()
                                   and self.n_global != self.n):
            torch.distributed.all_reduce(self.red, group=self.pg)

    def adamax_update(self) -> None:
        check(self.lib.desmo_adamax_update(
            C.byref(self.shape), _ptr(self.red), _ptr(self.dphi), _ptr(self.P), _ptr(self.phi), _ptr(self.phi_m), _ptr(self.phi_u),
            _ptr(self.gates), _ptr(self.gates_m), _ptr(self.gates_u), _ptr(self.rows), _ptr(self.rows_m), _ptr(self.rows_u),
            _ptr(self.coefs), _ptr(self.coefs_m), _ptr(self.coefs_u), _ptr(self.periods), _ptr(self.periods_m), _ptr(self.periods_u),
            _ptr(self.omega), _ptr(self.omega_m), _ptr(self.omega_u), _ptr(self.hyper), _ptr(self.step_dev), _ptr(self.losses),
            _ptr(self.workspace), self._stream()), "desmo_adamax_update")

    def _sharded(self) -> bool:
        return self.pg is not None or (torch.distributed.is_available() and torch.distributed.is_initialized() and self.n_global != self.n)

    def train_step(self) -> None:
        """forward + losses + backward + optimizer.step of CYL:711-768; losses land in self.losses (device).

        Multi-GPU: the K x m block of `red` (E = G^T R) is final as soon as the dominant kernel has run, so its all-reduce is issued
        on a side stream and overlaps the chain-rule kernel; only the 1 + r^2 + 3r scalars are reduced afterwards."""
        with torch.cuda.device(self.device):
            self.build_w(True)
            if not self._sharded():
                self.fused_residual_grad()
            elif self._peer is not None:
                # one-shot exchange over NVLink peer memory: no NCCL call, no side stream
                st = self._stream()
                check(self.lib.desmo_peer_begin_step(C.byref(self._peer), st), "desmo_peer_begin_step")
                self.fused_residual_grad(self.red_local)
                check(self.lib.desmo_peer_allreduce(C.byref(self._peer), self._red_pad.numel(), _ptr(self._red_pad), st), "desmo_peer_allreduce")
            else:
                args = (C.byref(self.shape), _ptr(self.U), self._u_dtype(), _ptr(self.P), _ptr(self.phi), _ptr(self.omega), _ptr(self.W), _ptr(self.dphi),
                        _ptr(self.red), _ptr(self.workspace))
                main = torch.cuda.current_stream(self.device)
                if self._side is None:
                    self._side = torch.cuda.Stream(device=self.device)
                ecount = self.Kp * self.mld
                check(self.lib.desmo_fused_residual_grad_begin_ex(*args, main.cuda_stream), "desmo_fused_residual_grad_begin")
                self._side.wait_stream(main)
                with torch.cuda.stream(self._side):
                    torch.distributed.all_reduce(self.red[:ecount], group=self.pg)
                check(self.lib.desmo_fused_residual_grad_finish_ex(*args, main.cuda_stream), "desmo_fused_residual_grad_finish")
                torch.distributed.all_reduce(self.red[ecount:], group=self.pg)
                main.wait_stream(self._side)
            self.adamax_update()
            if self.plateau_state is not None:  # ReduceLROnPlateau.step(total_loss) of this epoch, on the device
                check(self.lib.desmo_plateau_step(_ptr(self.plateau_state), _ptr(self.step_dev), _ptr(self.losses), _ptr(self.hyper),
                                                  self._stream()), "desmo_plateau_step")

    def gradients(self, beta: Optional[float] = None, l1_lambda: Optional[float] = None) -> dict:
        """d total_loss / d every packed parameter (what total_loss.backward() leaves in .grad, CYL:766)."""
        self._refresh_hyper_host()
        saved = list(self.hyper_host)
        if beta is not None or l1_lambda is not None:
            self.set_hyper(saved[:5], saved[5] if beta is None else beta, saved[6] if l1_lambda is None else l1_lambda)
        f32 = dict(dtype=torch.float32, device=self.device)
        g = {"gates": torch.zeros(self.K, **f32), "omega": torch.zeros(3 * self.r, **f32), "phi": torch.zeros(self.r, self.ld, **f32)}
        if self.nF:
            g["coefs"], g["periods"] = torch.zeros_like(self.coefs), torch.zeros_like(self.periods)
        else:
            g["rows"] = torch.zeros(self.K, self.mld, **f32)
        with torch.cuda.device(self.device):
            self.build_w(False)
            self.fused_residual_grad()
            self.all_reduce()
            g["phi"].copy_(self.dphi)
            check(self.lib.desmo_assemble_grads(
                C.byref(self.shape), _ptr(self.red), _ptr(g["phi"]), _ptr(self.P), _ptr(self.phi), _ptr(self.gates), _ptr(self.rows),
                _ptr(self.coefs), _ptr(self.periods), _ptr(self.hyper), _ptr(g["gates"]), _ptr(g.get("rows")), _ptr(g.get("coefs")),
                _ptr(g.get("periods")), _ptr(g["omega"]), _ptr(self.losses), _ptr(self.workspace), self._stream()),
                "desmo_assemble_grads")
        if beta is not None or l1_lambda is not None:
            self.set_hyper(saved[:5], saved[5], saved[6])
        g["phi"] = g["phi"][:, :self.n]
        if "rows" in g:
            g["rows"] = g["rows"][:, :self.m]
        return g

    def recon_backward(self, grad_recon: torch.Tensor) -> dict:
        """d L / d every packed parameter for an upstream gradient dL/drecon of shape (m, n) (autograd backward of forward()'s
        recon, CYL:766): desmo_recon_backward (the fused G3 / G4 machinery with R supplied) + desmo_assemble_grads."""
        if tuple(grad_recon.shape) != (self.m, self.n):
            raise ValueError(f"grad_recon must be ({self.m}, {self.n}), got {tuple(grad_recon.shape)}")
        f32 = dict(dtype=torch.float32, device=self.device)
        gr = torch.zeros(self.m, self.ld, **f32)  # the layout of U: pitch ld, pad columns zero
        gr[:, :self.n].copy_(grad_recon)
        self._refresh_hyper_host()
        saved = list(self.hyper_host)
        self.set_hyper(saved[:5], 0.0, 0.0)  # no regulariser terms: pure chain rule of the upstream gradient
        g = {"gates": torch.zeros(self.K, **f32), "omega": torch.zeros(3 * self.r, **f32), "phi": torch.zeros(self.r, self.ld, **f32)}
        if self.nF:
            g["coefs"], g["periods"] = torch.zeros_like(self.coefs), torch.zeros_like(self.periods)
        else:
            g["rows"] = torch.zeros(self.K, self.mld, **f32)
        losses = torch.zeros(4, **f32)
        with torch.cuda.device(self.device):
            self.build_w(False)
            check(self.lib.desmo_recon_backward(C.byref(self.shape), _ptr(gr), _ptr(self.P), _ptr(self.phi), _ptr(self.omega),
                                                _ptr(self.W), _ptr(self.dphi), _ptr(self.red), _ptr(self.workspace), self._stream()),
                  "desmo_recon_backward")
            self.all_reduce()
            g["phi"].copy_(self.dphi)
            check(self.lib.desmo_assemble_grads(
                C.byref(self.shape), _ptr(self.red), _ptr(g["phi"]), _ptr(self.P), _ptr(self.phi), _ptr(self.gates), _ptr(self.rows),
                _ptr(self.coefs), _ptr(self.periods), _ptr(self.hyper), _ptr(g["gates"]), _ptr(g.get("rows")), _ptr(g.get("coefs")),
                _ptr(g.get("periods")), _ptr(g["omega"]), _ptr(losses), _ptr(self.workspace), self._stream()), "desmo_assemble_grads")
        self.set_hyper(saved[:5], saved[5], saved[6])
        g["phi"] = g["phi"][:, :self.n]
        if "rows" in g:
            g["rows"] = g["rows"][:, :self.m]
        return g

    def reconstruct(self) -> torch.Tensor:
        """recon (m, n) -- first element of forward()'s tuple (CYL:576)."""
        out = torch.empty(self.m, self.ld, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self.build_w(False)
            check(self.lib.desmo_reconstruct(C.byref(self.shape), _ptr(self.P), _ptr(self.phi), _ptr(self.omega), _ptr(self.W),
                                             _ptr(out), self._stream()), "desmo_reconstruct")
        return out[:, :self.n]

    def residual_profile(self) -> dict:
        """Where and when the model misfits: the marginals of r^2, r = recon - U (the training step's residual for the current
        parameters; U as stored), in one pass over U without materialising recon (desmo_residual_profile).  Nothing else is written.

          snapshot_residual2 (m,) fp64  sum_x r(x, t)^2      summed over ranks when point-sharded
          snapshot_norm2     (m,) fp64  sum_x U(x, t)^2      summed over ranks when point-sharded
          point_residual2    (n,) fp32  sum_t r(x, t)^2      this rank's points
          point_norm2        (n,) fp32  sum_t U(x, t)^2      this rank's points

        Relative error per snapshot (over the cardiac cycle / shedding period): e(t) = sqrt(snapshot_residual2 / snapshot_norm2).
        Misfit map over the mesh: point_residual2, or sqrt(point_residual2 / point_norm2) for the relative error of each point.
        The totals equal residual_norm2() up to the order of the sums.  Bit-identical from call to call."""
        ud = self._u_dtype()
        snap = torch.empty(2, self.m, dtype=torch.float64, device=self.device)
        point = torch.empty(2, self.ld, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self.build_w(False)
            check(self.lib.desmo_residual_profile(C.byref(self.shape), _ptr(self.U), ud, _ptr(self.P), _ptr(self.phi), _ptr(self.omega),
                                                  _ptr(self.W), _ptr(snap), _ptr(point), self._stream()), "desmo_residual_profile")
            if self.n_global != self.n and torch.distributed.is_initialized():
                torch.distributed.all_reduce(snap, group=self.pg)
        return {"snapshot_residual2": snap[0], "snapshot_norm2": snap[1], "point_residual2": point[0, :self.n],
                "point_norm2": point[1, :self.n]}

    # ------------------------------------------------------------------ evaluation at chosen instants
    # Each of these takes exactly one of index= (training snapshot indices, any order, repeats allowed) or times= (fp32 times in the
    # model's own time coordinate, Fourier models only, any finite value: between grid points, before 0, beyond the window).  They
    # write nothing the model owns: parameters, optimizer state, rows, W, red, dphi, losses, step_dev and U stay as they are.
    def time_points(self, index) -> np.ndarray:
        """fp32 times of the given snapshot indices (k >= m continues the grid): times=time_points(range(m, 2 * m)) is the next
        window at the training spacing, and times=time_points(index) gives the same bits as index=index."""
        return time_points(index, self.m)

    def _w_at(self, idx: Optional[np.ndarray], t: Optional[np.ndarray], mld_out: int, rows_out: Optional[torch.Tensor] = None):
        """W' [Kp][mld_out] at the instants _instants() validated (desmo_build_w_at); rows_out [K][mld_out] receives z(t_i)."""
        m_out = (idx if idx is not None else t).size
        W = torch.empty(self.Kp, mld_out, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.desmo_build_w_at(C.byref(self.shape), _ptr(self.gates), _ptr(self.rows), _ptr(self.coefs), _ptr(self.periods),
                                            m_out, mld_out, None if idx is None else idx.ctypes.data, None if t is None else t.ctypes.data,
                                            _ptr(W), _ptr(rows_out), self._stream()), "desmo_build_w_at")
        return W

    def _shape_at(self, m_out: int):
        """The engine's shape with m' snapshots (the spatial entry points need m >= 2: m' = 1 runs as two with a zero second column)."""
        return make_shape(self.n, max(m_out, 2), self.r, self.polyorder, self.nF, self.n_global, self.shape.path, ld=self.ld)

    def temporal_rows_at(self, index=None, times=None) -> torch.Tensor:
        """z(t) at the instants, (K, m') fp32: forward()'s z_values there, unscaled by the gates, all K terms in K order."""
        idx, t = _instants(index, times, self.m, self.nF)
        m_out = (idx if idx is not None else t).size
        rows = torch.empty(self.K, round_up(m_out, 16), dtype=torch.float32, device=self.device)
        self._w_at(idx, t, rows.shape[1], rows)
        return rows[:, :m_out]

    def reconstruct_at(self, index=None, times=None) -> torch.Tensor:
        """recon at the instants, (m', n) fp32, allocating only m' rows: desmo_build_w_at, then desmo_reconstruct on an m'-snapshot
        shape.  reconstruct_at(index=k) is bit for bit reconstruct()[k]."""
        idx, t = _instants(index, times, self.m, self.nF)
        m_out = (idx if idx is not None else t).size
        sh = self._shape_at(m_out)
        W = self._w_at(idx, t, sh.mld)
        out = torch.empty(sh.m, self.ld, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.desmo_reconstruct(C.byref(sh), _ptr(self.P), _ptr(self.phi), _ptr(self.omega), _ptr(W), _ptr(out), self._stream()),
                  "desmo_reconstruct")
        return out[:m_out, :self.n]

    def residual_profile_at(self, snapshots: torch.Tensor, index=None, times=None) -> dict:
        """residual_profile() for a held-out block: r = recon(t_i) - snapshots[i], snapshots (m', n) fp32, fp64 or bf16, on the host or
        the device.  The block is stored as U is (snapshot_dtype; fp32 / fp64 into bf16 by desmo_snapshot_to_bf16 in chunks of at
        most SNAPSHOT_CHUNK_BYTES) in a temporary [m'][ld] buffer.  Returns the four keys of residual_profile(): (m',) snapshot
        sums, summed over ranks when point-sharded, and this rank's (n,) point sums."""
        idx, t = _instants(index, times, self.m, self.nF)
        m_out = (idx if idx is not None else t).size
        if not torch.is_tensor(snapshots) or tuple(snapshots.shape) != (m_out, self.n):
            got = tuple(snapshots.shape) if torch.is_tensor(snapshots) else type(snapshots).__name__
            raise _lib.DesmoError(f"snapshots must be a ({m_out}, {self.n}) tensor, one row per instant, got {got}")
        if snapshots.dtype not in (torch.float32, torch.float64, torch.bfloat16):
            raise _lib.DesmoError(f"snapshots must be float32, float64 or bfloat16, got {snapshots.dtype}")
        sh = self._shape_at(m_out)
        W = self._w_at(idx, t, sh.mld)
        U = torch.zeros(sh.m, self.ld, dtype=self.snapshot_dtype, device=self.device)
        if self.snapshot_dtype == torch.float32 or snapshots.dtype == torch.bfloat16:
            U[:m_out, :self.n].copy_(snapshots)
        else:
            self._snapshot_to_bf16(snapshots, U, sh, False)
        snap = torch.empty(2, sh.m, dtype=torch.float64, device=self.device)
        point = torch.empty(2, self.ld, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.desmo_residual_profile(C.byref(sh), _ptr(U), _lib.u_dtype_code(U.dtype), _ptr(self.P), _ptr(self.phi),
                                                  _ptr(self.omega), _ptr(W), _ptr(snap), _ptr(point), self._stream()), "desmo_residual_profile")
            if self.n_global != self.n and torch.distributed.is_initialized():
                torch.distributed.all_reduce(snap, group=self.pg)
        return {"snapshot_residual2": snap[0, :m_out], "snapshot_norm2": snap[1, :m_out], "point_residual2": point[0, :self.n],
                "point_norm2": point[1, :self.n]}

    def term_norms(self, physical: bool = False) -> torch.Tensor:
        """Per-term norms of the post-hoc sweep, K order, fp64 (poly_norm / nonlinear_norm, CYL:624-692; FCYL:644-720).

        Default = the reference's semantics, which define the active mask: the scripts pass the RAW ``phi_list`` (CYL:1192-1194),
        so the library is evaluated on phi alone, and the Fourier scripts weight polynomial term i by all T series at time index
        i (FCYL:652,659).  ``physical=True`` returns ||gate_j G_j z_j^T||_F of the term as it enters forward() (phi * POD)."""
        g2 = torch.zeros(self.K, dtype=torch.float32, device=self.device)
        out = torch.zeros(self.K, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            self.build_w(False)  # refreshes rows for the Fourier variant
            check(self.lib.desmo_library_colnorm2(C.byref(self.shape), _ptr(self.P) if physical else None, _ptr(self.phi),
                                                  _ptr(self.omega), _ptr(g2), self._stream()), "desmo_library_colnorm2")
            if self.n_global != self.n and torch.distributed.is_initialized():
                torch.distributed.all_reduce(g2, group=self.pg)
            check(self.lib.desmo_term_norms(C.byref(self.shape), _ptr(g2), _ptr(self.gates), _ptr(self.rows),
                                            1 if (self.nF and not physical) else 0, _ptr(out), self._stream()), "desmo_term_norms")
        return out

    def residual_norm2(self) -> float:
        """||G W - U||_F^2 over all ranks with the current gates (evaluation pass, no update)."""
        with torch.cuda.device(self.device):
            self.build_w(False)
            self.fused_residual_grad()
            self.all_reduce()
        return float(self.red[self.Kp * self.mld].item())

    # ------------------------------------------------------------------ POD (method of snapshots)
    def preprocess_snapshot(self, raw: torch.Tensor, d_in: int = 1, d_use: Optional[int] = None, magnitude: bool = True,
                            subtract_mean: bool = True, scale_sqrt_m: bool = False, t_stride: int = 1) -> torch.Tensor:
        """Reader output -> resident snapshot U on the device (desmo_preprocess): magnitude of the first ``d_use`` of ``d_in``
        velocity components (CYL:88-133), temporal-mean removal (CYL:136-149), optional 1/sqrt(m) (ANEU:143) and every
        ``t_stride``-th snapshot (TURB:189).  ``raw`` is X.T as read: [m_in, n*d_in], fp32 or fp64, on this device.
        bf16 storage receives the fp32 result rounded once more (and the quantisation error is recorded).
        Returns the fp64 temporal mean [n] (the reference's X_mean)."""
        d_use = d_in if d_use is None else d_use
        if raw.device != self.device or raw.dtype not in (torch.float32, torch.float64) or raw.dim() != 2 or raw.stride(1) != 1:
            raise ValueError("raw must be a [m_in, n*d_in] fp32/fp64 tensor on the engine's device with unit inner stride")
        if raw.shape[1] != self.n * d_in:
            raise ValueError(f"raw has {raw.shape[1]} columns, expected n*d_in = {self.n * d_in}")
        if self.U is None or self.U.dtype != self.snapshot_dtype:
            self.U = torch.empty(self.m, self.ld, dtype=self.snapshot_dtype, device=self.device)
        mean = torch.empty(self.n, dtype=torch.float64, device=self.device)
        flags = (_lib.PRE_MAGNITUDE if magnitude else 0) | (_lib.PRE_SUBTRACT_MEAN if subtract_mean else 0) | \
                (_lib.PRE_SCALE_SQRT_M if scale_sqrt_m else 0)
        bf16 = self.snapshot_dtype == torch.bfloat16
        self._qsums = torch.zeros(2, dtype=torch.float64, device=self.device) if bf16 else None
        _lib.check(self.lib.desmo_preprocess_ex(C.byref(self.shape), raw.data_ptr(), 1 if raw.dtype == torch.float64 else 0, raw.stride(0),
                                                raw.shape[0], t_stride, d_in, d_use, flags, self.U.data_ptr(), self._u_dtype(),
                                                _ptr(self._qsums), mean.data_ptr(), self._stream()), "desmo_preprocess")
        return mean

    def pod_from_snapshot(self) -> torch.Tensor:
        """Replaces POD_analysis (CYL:197-205) for the resident snapshot matrix: returns singular values (r,), fills self.P.

        r <= 14 (the on-device eigensolver's limit; a larger r raises before P is touched).  A mode whose eigenvalue is at the rounding
        level of the fp32 Gram (lambda_i <= 2^-23 trace) comes back as sigma_i = 0 with a zero row of P.  Raises DesmoError when the
        eigensolver does not converge (P then holds the projection of the unconverged modes)."""
        ud = self._u_dtype()
        f32 = dict(dtype=torch.float32, device=self.device)
        V, sigma = torch.zeros(self.r, self.m, **f32), torch.zeros(self.r, **f32)
        ws = torch.zeros(2 * 8 * 16 * self.m + 1024, dtype=torch.uint8, device=self.device)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.device(self.device):
            Cm, trace = self._pod_gram(ev[0], ev[1])
            check(self.lib.desmo_pod_eig(self.m, self.r, _ptr(Cm), _ptr(V), _ptr(sigma), _ptr(ws), ws.numel(), self._stream()), "desmo_pod_eig")
            ev[2].record()
            check(self.lib.desmo_pod_project_ex(C.byref(self.shape), _ptr(self.U), ud, _ptr(V), _ptr(sigma), _ptr(self.P), self._stream()),
                  "desmo_pod_project")
            ev[3].record()
        torch.cuda.synchronize(self.device)
        self.pod_timing = {"gram_ms": ev[0].elapsed_time(ev[1]), "eig_ms": ev[1].elapsed_time(ev[2]), "project_ms": ev[2].elapsed_time(ev[3])}
        self.pod_V, self.pod_gram = V, Cm
        # the eigensolver's report at the head of its workspace (desmo_pod_eig): sweeps, converged flag, worst residual / lambda_1
        iterations, converged = ws[:8].view(torch.int32).tolist()
        self.pod_eig_iterations, self.pod_eig_residual = iterations, float(ws[16:24].view(torch.float64).item())
        if not converged:
            raise _lib.DesmoError(f"desmo_pod_eig did not converge in {iterations} sweeps (residual {self.pod_eig_residual:.2e} lambda_1)")
        # POD_analysis' diagnostics (CYL:200-211) without forming X_approx: energy_content = S^2 / sum(S^2) of the r leading modes, its
        # running sum, and err_POD = ||X - X_r|| / ||X|| = sqrt(1 - sum_{i<r} sigma_i^2 / ||X||_F^2) (Eckart-Young)
        s2 = sigma.double() ** 2
        self.pod_energy = (s2 / trace).cpu()
        self.pod_cumulative_energy = torch.cumsum(self.pod_energy, 0)
        self.pod_error = float(torch.sqrt(torch.clamp(1.0 - s2.sum() / trace, min=0.0)))
        return sigma

    def _pod_gram(self, ev_start: torch.cuda.Event, ev_gram: torch.cuda.Event):
        """C = U U^T of the resident snapshot, all-reduced over the ranks when point-sharded, and its fp64 trace (= ||X||_F^2).  The
        events bracket the Gram kernel (the all-reduce comes after ev_gram).  Call inside torch.cuda.device(self.device)."""
        Cm = torch.zeros(self.m, self.m, dtype=torch.float32, device=self.device)
        ev_start.record()
        check(self.lib.desmo_pod_gram_ex(C.byref(self.shape), _ptr(self.U), self._u_dtype(), _ptr(Cm), _ptr(self.workspace), self._stream()),
              "desmo_pod_gram")
        ev_gram.record()
        if self.n_global != self.n and torch.distributed.is_initialized():
            torch.distributed.all_reduce(Cm, group=self.pg)
        return Cm, Cm.diagonal().sum(dtype=torch.float64)

    def _eigh_workspace(self) -> torch.Tensor:
        nbytes = C.c_size_t(0)
        check(self.lib.desmo_pod_eigh_workspace_bytes(self.m, self.r, C.byref(nbytes)), "desmo_pod_eigh_workspace_bytes")
        return torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)

    def pod_analysis(self) -> torch.Tensor:
        """POD_analysis (CYL:197-211) of the resident snapshot matrix for any r <= 64: returns the singular values sigma (r,) and
        fills self.P with the r leading modes.

        The Gram C = U U^T (all-reduced when point-sharded) goes through the dense fp64 eigensolver (desmo_pod_eigh), which also
        returns the whole spectrum: self.pod_singular_values holds all m singular values (fp64, host, descending), POD_analysis'
        S for the energy plot and the choice of r.  Sets the attributes pod_from_snapshot sets (pod_V = the temporal coefficients
        V^T[:r], pod_gram, pod_energy, pod_cumulative_energy, pod_error, pod_timing).  A mode at the rounding level of the fp32 Gram
        (lambda_i <= 2^-23 trace) comes back as sigma_i = 0 with a zero row of P.  Raises DesmoError, with P untouched, when the
        solver reports a non-finite result or a residual ||C v_i - lambda_i v_i|| above 2^-27 lambda_1."""
        f32 = dict(dtype=torch.float32, device=self.device)
        V, sigma = torch.zeros(self.r, self.m, **f32), torch.zeros(self.r, **f32)
        S = torch.zeros(self.m, dtype=torch.float64, device=self.device)
        ws = self._eigh_workspace()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        with torch.cuda.device(self.device):
            Cm, trace = self._pod_gram(ev[0], ev[1])
            check(self.lib.desmo_pod_eigh(self.m, self.r, _ptr(Cm), _ptr(S), _ptr(V), _ptr(sigma), _ptr(ws), ws.numel(), self._stream()),
                  "desmo_pod_eigh")
            ev[2].record()
            status = int(ws[:4].view(torch.int32).item())
            residual = float(ws[8:16].view(torch.float64).item())
            self.pod_eig_residual = residual
            if status != 0 or not residual <= 2.0 ** -27:
                raise _lib.DesmoError(f"desmo_pod_eigh failed (status {status}, residual {residual:.2e} lambda_1); P is unchanged")
            check(self.lib.desmo_pod_project_ex(C.byref(self.shape), _ptr(self.U), self._u_dtype(), _ptr(V), _ptr(sigma), _ptr(self.P),
                                                self._stream()), "desmo_pod_project")
            ev[3].record()
        torch.cuda.synchronize(self.device)
        self.pod_timing = {"gram_ms": ev[0].elapsed_time(ev[1]), "eig_ms": ev[1].elapsed_time(ev[2]), "project_ms": ev[2].elapsed_time(ev[3])}
        self.pod_V, self.pod_gram = V, Cm
        self.pod_singular_values = S.cpu()
        s2 = sigma.double() ** 2
        self.pod_energy = (s2 / trace).cpu()
        self.pod_cumulative_energy = torch.cumsum(self.pod_energy, 0)
        self.pod_error = float(torch.sqrt(torch.clamp(1.0 - s2.sum() / trace, min=0.0)))
        return sigma
