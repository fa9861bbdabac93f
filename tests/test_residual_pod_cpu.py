"""CPU-side checks of the residual POD: the argument checks of desmo_residual_gram / desmo_residual_modes that run before anything
touches a device, the scratch formula stated in include/desmo_b200.h, and the ctypes declarations of the new entry points."""
import ctypes as C

import pytest

from desmo_b200 import _lib

torch = pytest.importorskip("torch")

CHUNK_BYTES = 64 << 20  # kResidChunkBytes of csrc/gemm_path.cu


def _scratch(n, m, r, p, sms):
    """The formula of include/desmo_b200.h, restated."""
    shape = _lib.make_shape(n, m, r, p)
    T = _lib.load().desmo_num_terms(r, p)
    K = T + 3 * r
    A = lambda v: (v + 1023) // 1024 * 1024  # noqa: E731
    Kr, mp = (K + 63) // 64 * 64, (m + 127) // 128 * 128
    tiles = (mp // 128) * (mp // 128 + 1) // 2
    rows_c = min(max(CHUNK_BYTES // (6 * Kr + 4 * mp) // 128 * 128, 128), shape.ld)
    ns = min(max(sms // tiles, 1), 32, rows_c // 64)
    part = 131072 * ns * tiles
    total = (A(8 * T) + A(T) + A(6 * Kr * rows_c) + A(6 * Kr * mp) + A(4 * rows_c * mp) + A(512 * mp) + A(8 * sms) + A(part))
    return shape, total, rows_c


@pytest.mark.parametrize("n,m,r,p,sms", [
    (3 << 20, 1000, 4, 2, 148),
    (262144, 1000, 32, 2, 148),
    (1, 70, 8, 3, 148),
    (4100, 1300, 4, 2, 148),
    (700, 8192, 64, 1, 148),
    (100000, 300, 8, 2, 7),
])
def test_scratch_formula(n, m, r, p, sms):
    shape, want, rows_c = _scratch(n, m, r, p, sms)
    got = C.c_size_t(0)
    assert _lib.load().desmo_residual_gram_scratch_bytes(C.byref(shape), sms, C.byref(got)) == 0
    assert got.value == want
    # bounded by the chunk and m, never by n: the same scratch for 10x the points
    big = _lib.make_shape(10 * n, m, r, p)
    got10 = C.c_size_t(0)
    assert _lib.load().desmo_residual_gram_scratch_bytes(C.byref(big), sms, C.byref(got10)) == 0
    if rows_c < shape.ld:
        assert got10.value == got.value
    if (n, m) == (3 << 20, 1000):
        assert want < 128e6 and want < 0.01 * 4 * n * m, want  # not an m x n buffer (12.6 GB in fp32)


def test_scratch_bytes_rejects_bad_arguments():
    shape = _lib.make_shape(1000, 50, 4, 2)
    got = C.c_size_t(0)
    lib = _lib.load()
    assert lib.desmo_residual_gram_scratch_bytes(C.byref(shape), 0, C.byref(got)) == 1
    assert lib.desmo_residual_gram_scratch_bytes(C.byref(shape), 148, None) == 1


# dummy device pointers: every case below is rejected on the host before a device is touched
def _gram(shape, U=16, u_dtype=_lib.DTYPE_F32, Cp=16, scratch=16, nbytes=1 << 40):
    lib = _lib.load()
    rc = lib.desmo_residual_gram(C.byref(shape), U, u_dtype, 16, 16, 16, 16, Cp, 16, scratch, nbytes, None)
    return rc, lib.desmo_last_error().decode()


def _modes(shape, k, V=16, u_dtype=_lib.DTYPE_F32, nbytes=1 << 40, scratch=16):
    lib = _lib.load()
    rc = lib.desmo_residual_modes(C.byref(shape), 16, u_dtype, 16, 16, 16, 16, k, V, 16, 16, scratch, nbytes, None)
    return rc, lib.desmo_last_error().decode()


def test_gram_rejects_bad_arguments_before_any_launch():
    shape = _lib.make_shape(1000, 50, 4, 2)
    for kw, msg in ((dict(U=None), "null"), (dict(Cp=None), "null"), (dict(scratch=None), "null"), (dict(u_dtype=7), "u_dtype"),
                    (dict(scratch=8), "aligned"), (dict(nbytes=1024), "scratch too small")):
        rc, err = _gram(shape, **kw)
        assert rc == 1, (kw, rc, err)
        assert msg in err, (kw, err)


@pytest.mark.parametrize("k,code,msg", [(0, 1, "k"), (-3, 1, "k"), (51, 1, "k"), (65, 2, "k")])
def test_modes_rejects_bad_k_before_any_launch(k, code, msg):
    shape = _lib.make_shape(1000, 50 if k != 65 else 100, 4, 2)
    rc, err = _modes(shape, k)
    assert rc == code and msg in err, (rc, err)


def test_modes_rejects_null_dtype_misaligned_and_small_scratch():
    shape = _lib.make_shape(1000, 50, 4, 2)
    rc, err = _modes(shape, 4, V=None)
    assert rc == 1 and "null" in err
    rc, err = _modes(shape, 4, u_dtype=1)
    assert rc == 1 and "u_dtype" in err
    rc, err = _modes(shape, 4, nbytes=0)
    assert rc == 1 and "scratch too small" in err
    rc, err = _modes(shape, 4, scratch=24)
    assert rc == 1 and "aligned" in err


def test_signatures_declared():
    declared = set(_lib.declared_symbols())
    for name in ("desmo_residual_gram_scratch_bytes", "desmo_residual_gram", "desmo_residual_modes"):
        assert name in declared and name in _lib.SIGNATURES
    res, args = _lib.SIGNATURES["desmo_residual_gram"]
    assert len(args) == 12 and args[-2] is C.c_size_t
    res, args = _lib.SIGNATURES["desmo_residual_modes"]
    assert len(args) == 14 and args[7] is C.c_int32 and args[-2] is C.c_size_t

