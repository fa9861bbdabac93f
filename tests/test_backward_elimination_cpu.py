"""CPU-side checks of backward elimination: the argument checks of desmo_elimination_pass / desmo_elimination_greedy that run before
anything touches a device, the scratch formula stated in include/desmo_b200.h, the ctypes declarations, and a numpy statement of the
greedy rule (zero rows first, ties to the lowest index, the F update) against brute-force recomputation of ||R_S||^2."""
import ctypes as C
import re

import numpy as np
import pytest

from desmo_b200 import _lib

torch = pytest.importorskip("torch")

CHUNK_BYTES = 64 << 20  # kElimChunkBytes of csrc/gemm_path.cu


def _scratch(n, m, r, p, sms):
    """The formula of include/desmo_b200.h, restated."""
    shape = _lib.make_shape(n, m, r, p)
    T = _lib.load().desmo_num_terms(r, p)
    K = T + 3 * r
    A = lambda v: (v + 1023) // 1024 * 1024  # noqa: E731
    Kr, Kp16, mp = (K + 127) // 128 * 128, (K + 15) // 16 * 16, (m + 127) // 128 * 128
    TK = Kr // 128
    tiles = TK * (TK + 1) // 2
    rows_c = min(max(CHUNK_BYTES // (6 * Kr + 4 * mp) // 128 * 128, 128), shape.ld)
    ns = lambda x: min(max(sms // x, 1), 32, rows_c // 64)  # noqa: E731
    nsg, nse = ns(tiles), ns(TK * mp // 128)
    total = (A(8 * T) + A(T) + A(6 * Kr * rows_c) + A(6 * Kr * mp) + A(4 * rows_c * mp) + A(4 * nse * Kp16 * shape.mld) + A(8 * sms)
             + A(131072 * nsg * tiles))
    return shape, total, rows_c, K


@pytest.mark.parametrize("n,m,r,p,sms", [
    (3 << 20, 1000, 4, 2, 148),
    (262144, 1000, 32, 2, 148),
    (1, 70, 8, 3, 148),
    (4100, 1300, 4, 2, 148),
    (700, 150, 64, 1, 148),
    (100000, 300, 8, 2, 7),
])
def test_scratch_formula(n, m, r, p, sms):
    shape, want, rows_c, K = _scratch(n, m, r, p, sms)
    got = C.c_size_t(0)
    assert _lib.load().desmo_elimination_scratch_bytes(C.byref(shape), sms, C.byref(got)) == 0
    assert got.value == want
    # bounded by the chunk, K and m, never by n
    big = _lib.make_shape(10 * n, m, r, p)
    got10 = C.c_size_t(0)
    assert _lib.load().desmo_elimination_scratch_bytes(C.byref(big), sms, C.byref(got10)) == 0
    if rows_c < shape.ld:
        assert got10.value == got.value
    if (n, m, r) == (262144, 1000, 32):
        assert want < 160e6, want
    # the greedy's head fits in it
    assert 256 + 2 * ((4 * K + 255) // 256 * 256) + (8 * K + 255) // 256 * 256 <= want


def test_scratch_bytes_rejects_bad_arguments():
    shape = _lib.make_shape(1000, 50, 4, 2)
    got = C.c_size_t(0)
    lib = _lib.load()
    assert lib.desmo_elimination_scratch_bytes(C.byref(shape), 0, C.byref(got)) == 1
    assert lib.desmo_elimination_scratch_bytes(C.byref(shape), 148, None) == 1


# dummy device pointers: every case below is rejected on the host before a device is touched
def _pass(shape, U=16, u_dtype=_lib.DTYPE_F32, A=16, scratch=16, nbytes=1 << 40):
    lib = _lib.load()
    rc = lib.desmo_elimination_pass(C.byref(shape), U, u_dtype, 16, 16, 16, 16, A, 16, 16, scratch, nbytes, None)
    return rc, lib.desmo_last_error().decode()


def _greedy(shape, steps, order=16, scratch=16, nbytes=1 << 40, F=16):
    lib = _lib.load()
    rc = lib.desmo_elimination_greedy(C.byref(shape), 16, F, 16, 16, steps, order, 16, scratch, nbytes, None)
    return rc, lib.desmo_last_error().decode()


def test_pass_rejects_bad_arguments_before_any_launch():
    shape = _lib.make_shape(1000, 50, 4, 2)
    for kw, msg in ((dict(U=None), "null"), (dict(A=None), "null"), (dict(scratch=None), "null"), (dict(u_dtype=7), "u_dtype"),
                    (dict(u_dtype=_lib.DTYPE_F64), "u_dtype"), (dict(scratch=8), "aligned"), (dict(nbytes=1024), "scratch too small")):
        rc, err = _pass(shape, **kw)
        assert rc == 1, (kw, rc, err)
        assert msg in err, (kw, err)


def test_greedy_rejects_bad_arguments_before_any_launch():
    shape = _lib.make_shape(1000, 50, 4, 2)
    K = 27
    for args, kw, msg in (((K + 1,), {}, "steps"), ((-1,), {}, "steps"), ((3,), dict(order=None), "null"), ((3,), dict(F=None), "null"),
                          ((3,), dict(scratch=None), "null"), ((3,), dict(scratch=24), "aligned"), ((3,), dict(nbytes=255), "too small")):
        rc, err = _greedy(shape, *args, **kw)
        assert rc == 1, (args, kw, rc, err)
        assert msg in err, (args, kw, err)


def test_signatures_declared():
    declared = set(_lib.declared_symbols())
    for name in ("desmo_elimination_scratch_bytes", "desmo_elimination_pass", "desmo_elimination_greedy"):
        assert name in declared and name in _lib.SIGNATURES
    res, args = _lib.SIGNATURES["desmo_elimination_pass"]
    assert len(args) == 13 and args[2] is C.c_int32 and args[-2] is C.c_size_t
    res, args = _lib.SIGNATURES["desmo_elimination_greedy"]
    assert len(args) == 11 and args[5] is C.c_int32 and args[-2] is C.c_size_t
    # parameter counts against the header's prototypes
    src = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)
    for name in ("desmo_elimination_scratch_bytes", "desmo_elimination_pass", "desmo_elimination_greedy"):
        proto = re.search(rf"\b{name}\s*\(([^)]*)\)", src).group(1)
        assert len(proto.split(",")) == len(_lib.SIGNATURES[name][1]), name


# ------------------------------------------------------------------------------------------------ the greedy rule, in numpy
def greedy(A, F, r2, W, steps):
    """The rule of desmo_elimination_greedy: zero W rows first in index order; then the least sum_t W_k (A_kk W_k - 2 F_k), ties to
    the lowest index; then F_l -= A_lk W_k for every l."""
    K = A.shape[0]
    F = F.copy()
    removed = np.zeros(K, bool)
    nz = (W != 0).any(1)
    order, pred = [], [r2]
    for _ in range(steps):
        zero = np.flatnonzero(~removed & ~nz)
        if zero.size:
            k = int(zero[0])
            pred.append(pred[-1])
        else:
            delta = (W * (np.diag(A)[:, None] * W - 2 * F)).sum(1)
            delta[removed] = np.inf
            k = int(np.argmin(delta))  # the first minimum: the lowest index on ties
            pred.append(pred[-1] + delta[k])
            F -= np.outer(A[:, k], W[k])
        removed[k] = True
        order.append(k)
    return order, np.array(pred)


def _case(seed, n=40, m=7, K=6):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((n, K))
    G[:, 3] = 0.9 * G[:, 1] + 0.1 * rng.standard_normal(n)  # correlated columns
    W = rng.standard_normal((K, m))
    U = G @ W + 0.3 * rng.standard_normal((n, m))
    return G, W, U


def _brute(G, W, U, removed):
    keep = [k for k in range(G.shape[1]) if k not in removed]
    return float(((G[:, keep] @ W[keep] - U) ** 2).sum())


@pytest.mark.parametrize("seed", range(6))
def test_greedy_rule_against_brute_force(seed):
    G, W, U = _case(seed)
    W[2] = 0.0  # a zero row: first, whatever its column
    R = G @ W - U
    order, pred = greedy(G.T @ G, G.T @ R, float((R ** 2).sum()), W, G.shape[1])
    assert order[0] == 2
    for s in range(len(order) + 1):
        assert abs(pred[s] - _brute(G, W, U, order[:s])) <= 1e-9 * max(1.0, pred[0])
    # every non-zero step is the brute-force argmin given the prefix
    for s in range(1, len(order)):
        errs = {k: _brute(G, W, U, order[:s] + [k]) for k in range(G.shape[1]) if k not in order[:s]}
        assert errs[order[s]] <= min(errs.values()) + 1e-9 * pred[0]


def test_ties_go_to_the_lowest_index_and_zero_rows_in_index_order():
    rng = np.random.default_rng(3)
    n, m = 30, 5
    g = rng.standard_normal(n)
    G = np.stack([g, rng.standard_normal(n), g, rng.standard_normal(n), rng.standard_normal(n)], axis=1)  # columns 0 and 2 equal
    W = rng.standard_normal((5, m))
    W[2] = W[0]
    W[4] = 0.0
    W[3] = 0.0
    U = G @ W
    R = G @ W - U
    order, pred = greedy(G.T @ G, G.T @ R, 0.0, W, 5)
    assert order[:2] == [3, 4]
    assert order.index(0) < order.index(2)  # equal increments: the lower index first
    assert np.all(np.diff(pred[:3]) == 0)


def test_negative_increments_are_taken():
    """A term that fits noise the wrong way: removing it lowers the error, Delta < 0 -- a finding, taken first."""
    rng = np.random.default_rng(4)
    G = rng.standard_normal((50, 3))
    W = rng.standard_normal((3, 4))
    U = G[:, :2] @ W[:2]  # term 2 is not in the data
    R = G @ W - U
    order, pred = greedy(G.T @ G, G.T @ R, float((R ** 2).sum()), W, 3)
    assert order[0] == 2 and pred[1] < pred[0] and abs(pred[1]) <= 1e-9
