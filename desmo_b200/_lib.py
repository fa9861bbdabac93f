"""ctypes binding of libdesmo_b200.so (include/desmo_b200.h).  No fallback: a missing library or a failing call raises."""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, List

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DESMO_B200_LIB") or os.path.join(HERE, "libdesmo_b200.so")  # override: kernel experiments (tools/variant.sh)
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "desmo_b200.h")

PATH_AUTO, PATH_FP32, PATH_TC, PATH_GEMM = 0, 1, 2, 3
PATH_NAMES = {1: "fp32 ffma", 2: "fused tcgen05 (bf16-split)", 3: "tcgen05 GEMM path (bf16-split)"}
HYP_LR_GATES, HYP_LR_PHI, HYP_LR_Z, HYP_LR_OMEGA, HYP_LR_PERIOD, HYP_BETA, HYP_L1_LAMBDA, HYP_COUNT = range(8)
MAX_R, MAX_P, MAX_K = 64, 7, 4096
PRE_MAGNITUDE, PRE_SUBTRACT_MEAN, PRE_SCALE_SQRT_M = 1, 2, 4
DTYPE_F32, DTYPE_F64, DTYPE_BF16 = 0, 1, 2


class DesmoError(RuntimeError):
    pass


class Shape(C.Structure):
    _fields_ = [("n", C.c_int64), ("ld", C.c_int64), ("n_global", C.c_int64), ("m", C.c_int32), ("mld", C.c_int32),
                ("r", C.c_int32), ("polyorder", C.c_int32), ("nF", C.c_int32), ("path", C.c_int32)]


_vp, _i32, _i64, _f = C.c_void_p, C.c_int32, C.c_int64, C.c_float
_SP = C.POINTER(Shape)

# name -> (restype, argtypes); must list every function declared in include/desmo_b200.h (tests check this)
SIGNATURES: Dict[str, tuple] = {
    "desmo_last_error": (C.c_char_p, []),
    "desmo_version": (C.c_char_p, []),
    "desmo_num_terms": (_i32, [_i32, _i32]),
    "desmo_padded_k": (_i32, [_i32, _i32]),
    "desmo_red_count": (_i64, [_SP]),
    "desmo_selected_path": (_i32, [_SP]),
    "desmo_workspace_bytes": (C.c_int, [_SP, C.POINTER(C.c_size_t)]),
    "desmo_build_w": (C.c_int, [_SP] + [_vp] * 8),
    "desmo_build_w_at": (C.c_int, [_SP] + [_vp] * 4 + [_i32, _i32] + [_vp] * 5),
    "desmo_fused_residual_grad": (C.c_int, [_SP] + [_vp] * 9),
    "desmo_recon_backward": (C.c_int, [_SP] + [_vp] * 9),
    "desmo_fused_residual_grad_begin": (C.c_int, [_SP] + [_vp] * 9),
    "desmo_fused_residual_grad_finish": (C.c_int, [_SP] + [_vp] * 9),
    "desmo_fused_residual_grad_ex": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8),
    "desmo_fused_residual_grad_begin_ex": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8),
    "desmo_fused_residual_grad_finish_ex": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8),
    "desmo_adamax_update": (C.c_int, [_SP] + [_vp] * 26),
    "desmo_assemble_grads": (C.c_int, [_SP] + [_vp] * 17),
    "desmo_active_terms_bytes": (C.c_int, [_SP, _i32, C.POINTER(C.c_size_t)]),
    "desmo_active_terms_prepare": (C.c_int, [_SP, _vp, _i32, _vp, _vp]),
    "desmo_build_w_active": (C.c_int, [_SP] + [_vp] * 9),
    "desmo_fused_residual_grad_active": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8 + [_i32, _vp]),
    "desmo_fused_residual_grad_begin_active": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8 + [_i32, _vp]),
    "desmo_fused_residual_grad_finish_active": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8 + [_i32, _vp]),
    "desmo_adamax_update_active": (C.c_int, [_SP] + [_vp] * 27),
    "desmo_assemble_grads_active": (C.c_int, [_SP] + [_vp] * 18),
    "desmo_time_points_prepare": (C.c_int, [_SP, _vp, _i32, _vp, _vp]),
    "desmo_build_w_times": (C.c_int, [_SP] + [_vp] * 10),
    "desmo_adamax_update_times": (C.c_int, [_SP] + [_vp] * 28),
    "desmo_assemble_grads_times": (C.c_int, [_SP] + [_vp] * 19),
    "desmo_reconstruct": (C.c_int, [_SP] + [_vp] * 6),
    "desmo_library_colnorm2": (C.c_int, [_SP] + [_vp] * 5),
    "desmo_residual_profile": (C.c_int, [_SP, _vp, _i32] + [_vp] * 7),
    "desmo_pruning_profile": (C.c_int, [_SP, _vp, _i32] + [_vp] * 4 + [_i32] + [_vp] * 4),
    "desmo_pruning_profile_scratch_bytes": (C.c_int, [_SP, _i32, _i32, C.POINTER(C.c_size_t)]),
    "desmo_residual_gram_scratch_bytes": (C.c_int, [_SP, _i32, C.POINTER(C.c_size_t)]),
    "desmo_residual_gram": (C.c_int, [_SP, _vp, _i32] + [_vp] * 7 + [C.c_size_t, _vp]),
    "desmo_residual_modes": (C.c_int, [_SP, _vp, _i32] + [_vp] * 4 + [_i32] + [_vp] * 4 + [C.c_size_t, _vp]),
    "desmo_elimination_scratch_bytes": (C.c_int, [_SP, _i32, C.POINTER(C.c_size_t)]),
    "desmo_elimination_pass": (C.c_int, [_SP, _vp, _i32] + [_vp] * 8 + [C.c_size_t, _vp]),
    "desmo_elimination_greedy": (C.c_int, [_SP] + [_vp] * 4 + [_i32] + [_vp] * 3 + [C.c_size_t, _vp]),
    "desmo_term_norms": (C.c_int, [_SP, _vp, _vp, _vp, _i32, _vp, _vp]),
    "desmo_selftest_tables": (C.c_int, []),
    "desmo_selftest_chain_sweep": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "desmo_last_fused_kernel_ms": (C.c_int, [C.POINTER(C.c_float)]),
    "desmo_fused_kernel_ms_mean": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int32), C.c_int32]),
    "desmo_graph_fused_kernel_ms": (C.c_int, [C.POINTER(C.c_float)]),
    "desmo_fused_kernel_ms_series": (C.c_int, [C.POINTER(C.c_float), C.c_int32, C.POINTER(C.c_int32)]),
    "desmo_debug_timers": (C.c_int, [_SP, _vp, _vp, _i32]),
    "desmo_pod_gram": (C.c_int, [_SP] + [_vp] * 4),
    "desmo_pod_eig": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "desmo_pod_project": (C.c_int, [_SP] + [_vp] * 5),
    "desmo_pod_gram_ex": (C.c_int, [_SP, _vp, _i32, _vp, _vp, _vp]),
    "desmo_pod_project_ex": (C.c_int, [_SP, _vp, _i32, _vp, _vp, _vp, _vp]),
    "desmo_pod_eigh_workspace_bytes": (C.c_int, [_i32, _i32, C.POINTER(C.c_size_t)]),
    "desmo_pod_eigh": (C.c_int, [_i32, _i32] + [_vp] * 5 + [C.c_size_t, _vp]),
    "desmo_preprocess": (C.c_int, [_SP, _vp, _i32, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "desmo_preprocess_ex": (C.c_int, [_SP, _vp, _i32, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp, _vp, _vp]),
    "desmo_snapshot_to_bf16": (C.c_int, [_SP, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "desmo_plateau_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "desmo_peer_begin_step": (C.c_int, [_vp, _vp]),
    "desmo_peer_allreduce": (C.c_int, [_vp, _i64, _vp, _vp]),
    "desmo_session_create": (C.c_int, [_i64, _i32, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "desmo_session_create_sharded": (C.c_int, [_i64, _i64, _i32, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "desmo_session_set_allreduce": (C.c_int, [_vp, _vp, _vp]),
    "desmo_session_destroy": (C.c_int, [_vp]),
    "desmo_session_set_pod_host": (C.c_int, [_vp, _vp]),
    "desmo_session_set_params_host": (C.c_int, [_vp] * 6),
    "desmo_session_set_hyper": (C.c_int, [_vp, _vp, _f, _f]),
    "desmo_session_upload_snapshot_host": (C.c_int, [_vp, _vp]),
    "desmo_session_step_host": (C.c_int, [_vp, _vp, _vp]),
    "desmo_session_get_params_host": (C.c_int, [_vp] * 6),
    "desmo_train_host": (C.c_int, [_i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _i32, _vp, _i32]),
}

_lib = None


def declared_symbols() -> List[str]:
    """Function names declared in include/desmo_b200.h."""
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(desmo_[a-z0-9_]+)\s*\(", src)))


def load(build_if_missing: bool = True):
    """Loads the shared library; builds it in-tree with nvcc when absent.  Raises DesmoError if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if "DESMO_B200_LIB" not in os.environ:
        # in-tree library: (re)build when it is missing or older than the sources (build() compares a source digest and returns
        # at once on a match), so that edited kernels are never tested against a stale binary
        from . import build as _build

        try:
            _build.build()
        except _build.NvccMissing as e:  # no compiler here: an existing library is used as it is (a failed compile still raises)
            if not os.path.exists(LIB_PATH):
                raise DesmoError(f"{LIB_PATH} is missing and cannot be built ({e}); there is no CPU fallback") from e
    elif not os.path.exists(LIB_PATH):
        raise DesmoError(f"DESMO_B200_LIB={LIB_PATH} does not exist")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise DesmoError(f"cannot load {LIB_PATH}: {e} (no CPU fallback)") from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, _vp, _i64, _vp, _vp)  # desmo_allreduce_fn


def torch_allreduce_hook(group=None):
    """A desmo_allreduce_fn that sums the session's `red` buffer with torch.distributed (NCCL) on the session's own stream.
    Keep the returned object alive as long as the session uses it."""
    import torch
    import torch.distributed as dist

    class _Dev:  # exposes the raw device pointer to torch without a copy
        def __init__(self, ptr, count):
            self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None}

    cache = {}

    def hook(ptr, count, stream, user):
        try:
            key = (ptr, count)
            if key not in cache:
                cache[key] = torch.as_tensor(_Dev(ptr, count), device=torch.device("cuda", torch.cuda.current_device()))
            with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
                dist.all_reduce(cache[key], group=group)
            return 0
        except Exception as ex:  # a Python exception must not unwind through the C caller
            import sys
            print(f"desmo_b200 all-reduce hook failed: {ex}", file=sys.stderr)
            return 1

    return ALLREDUCE_FN(hook)


def u_dtype_code(dtype) -> int:
    """DESMO_DTYPE_* of a snapshot matrix's torch dtype: fp32 or bf16 storage; anything else raises before a launch."""
    import torch

    if dtype == torch.float32:
        return DTYPE_F32
    if dtype == torch.bfloat16:
        return DTYPE_BF16
    raise DesmoError(f"the snapshot matrix U must be float32 or bfloat16, got {dtype}")


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().desmo_last_error().decode(errors="replace")
        raise DesmoError(f"{what or 'desmo_b200'} failed (code {rc}): {msg}")


def round_up(v: int, a: int) -> int:
    return (v + a - 1) // a * a


def make_shape(n: int, m: int, r: int, polyorder: int, nF: int = 0, n_global: int | None = None, path: int = PATH_AUTO,
               ld: int | None = None, mld: int | None = None) -> Shape:
    return Shape(n=n, ld=ld or round_up(n, 256), n_global=n_global or n, m=m, mld=mld or round_up(m, 16), r=r,
                 polyorder=polyorder, nF=nF or 0, path=path)
