"""CPU-side checks of the bf16 snapshot storage boundary: the C ABI's new entry points are bound, the dtype codes match the header,
and dtypes other than fp32 / bf16 are refused before anything is launched."""
import re

import pytest

from desmo_b200 import _lib

torch = pytest.importorskip("torch")

NEW_SYMBOLS = ("desmo_fused_residual_grad_ex", "desmo_fused_residual_grad_begin_ex", "desmo_fused_residual_grad_finish_ex",
               "desmo_pod_gram_ex", "desmo_pod_project_ex", "desmo_preprocess_ex", "desmo_snapshot_to_bf16")


def test_signatures_cover_the_bf16_entry_points():
    declared = set(_lib.declared_symbols())
    for name in NEW_SYMBOLS:
        assert name in declared and name in _lib.SIGNATURES, name
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name), name
    # (shape, U, u_dtype, ...): the dtype is a 32-bit integer right after the snapshot pointer
    for name in NEW_SYMBOLS[:5]:
        assert _lib.SIGNATURES[name][1][2] is _lib._i32, name


def test_dtype_codes_match_the_header():
    src = open(_lib.HEADER_PATH).read()
    codes = {k: int(v) for k, v in re.findall(r"#define DESMO_DTYPE_(\w+) (\d+)", src)}
    assert codes == {"F32": _lib.DTYPE_F32, "F64": _lib.DTYPE_F64, "BF16": _lib.DTYPE_BF16}


def test_snapshot_dtype_is_fp32_or_bf16_only():
    assert _lib.u_dtype_code(torch.float32) == _lib.DTYPE_F32
    assert _lib.u_dtype_code(torch.bfloat16) == _lib.DTYPE_BF16
    for dt in (torch.float16, torch.float64, torch.int16):
        with pytest.raises(_lib.DesmoError):
            _lib.u_dtype_code(dt)
    from desmo_b200 import DesmoEngine

    with pytest.raises(_lib.DesmoError, match="snapshot_dtype"):
        DesmoEngine(300, 40, 2, 2, snapshot_dtype=torch.float16)
