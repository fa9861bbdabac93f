"""CPU-side checks of the dense POD eigensolver's C ABI: the workspace size formula and the argument errors, which are returned
before anything touches a device."""
import ctypes as C

import pytest

from desmo_b200 import _lib


def _ws_bytes(m, r):
    """head (256 bytes) + fp64 [A: m^2 | d, e, e^2, tau: 4m | p: 2m | lambda: m | Z, Y: 2rm | residuals: r | LU factors: 5rm]"""
    return 256 + 8 * (m * m + 7 * m + r * (7 * m + 1))


@pytest.mark.parametrize("m,r", [(1, 1), (2, 2), (17, 16), (1000, 4), (1000, 64), (4096, 32), (8192, 64)])
def test_workspace_bytes_formula(m, r):
    nbytes = C.c_size_t(0)
    assert _lib.load().desmo_pod_eigh_workspace_bytes(m, r, C.byref(nbytes)) == 0
    assert nbytes.value == _ws_bytes(m, r)


@pytest.mark.parametrize("m,r,code", [(100, 0, 1), (100, 65, 2), (10, 11, 1), (8193, 4, 2), (0, 1, 1), (100, -1, 1)])
def test_argument_errors_without_a_device(m, r, code):
    lib = _lib.load()
    nbytes = C.c_size_t(0)
    assert lib.desmo_pod_eigh_workspace_bytes(m, r, C.byref(nbytes)) == code
    dummy = C.c_void_p(16)   # never dereferenced: the arguments are rejected first
    assert lib.desmo_pod_eigh(m, r, dummy, dummy, dummy, dummy, dummy, 1 << 40, None) == code
    assert lib.desmo_last_error()


def test_workspace_too_small_without_a_device():
    lib = _lib.load()
    dummy = C.c_void_p(16)
    need = _ws_bytes(1000, 32)
    assert lib.desmo_pod_eigh(1000, 32, dummy, dummy, dummy, dummy, dummy, need - 1, None) == 1
    assert b"workspace too small" in lib.desmo_last_error()
    assert lib.desmo_pod_eigh(1000, 32, None, dummy, dummy, dummy, dummy, need, None) == 1   # null pointer
