"""CPU-side checks of the pruning profile: the term-order validation that runs before anything touches a device, the threshold ->
step mapping against the reference's threshold masks, and the scratch formula stated in include/desmo_b200.h."""
import ctypes as C
import os

import numpy as np
import pytest

from desmo_b200 import _lib
from desmo_b200.engine import pruning_order
from oracle import desmo_oracle as orc
from tests.helpers import golden_case

torch = pytest.importorskip("torch")

CHUNK_BYTES = 32 << 20  # kProfileChunkBytes of csrc/gemm_path.cu


# ------------------------------------------------------------------------------------------------ order validation
def test_python_order_validation():
    assert pruning_order([5, 0, 26], 27).tolist() == [5, 0, 26]
    got = pruning_order(torch.tensor([3, 1]), 27)
    assert got.dtype == np.int32 and got.flags.c_contiguous
    assert pruning_order([], 27).size == 0
    for bad in ([0, 1, 0], [27], [-1], list(range(28)), [0.5]):
        with pytest.raises(_lib.DesmoError):
            pruning_order(bad, 27)


def _call(shape, steps, order, U=16):
    lib = _lib.load()
    arr = (C.c_int32 * max(1, len(order)))(*order)
    # dummy device pointers: every case below is rejected on the host before a device is touched
    rc = lib.desmo_pruning_profile(C.byref(shape), U, _lib.DTYPE_F32, 16, 16, 16, 16, steps, C.addressof(arr), 16, 16, None)
    return rc, lib.desmo_last_error().decode()


@pytest.mark.parametrize("steps,order,msg", [
    (3, [0, 1, 0], "repeats"),
    (2, [4, 27], "outside"),
    (1, [-1], "outside"),
    (28, list(range(28)), "steps"),
    (-1, [0], "steps"),
])
def test_c_abi_rejects_bad_orders_before_any_launch(steps, order, msg):
    shape = _lib.make_shape(1000, 50, 4, 2)  # K = 27
    rc, err = _call(shape, steps, order)
    assert rc == 1 and msg in err, (rc, err)


def test_c_abi_rejects_bad_u_dtype_and_alignment():
    shape = _lib.make_shape(1000, 50, 4, 2)
    lib = _lib.load()
    arr = (C.c_int32 * 1)(0)
    rc = lib.desmo_pruning_profile(C.byref(shape), 16, 7, 16, 16, 16, 16, 1, C.addressof(arr), 16, 16, None)
    assert rc == 1 and b"u_dtype" in lib.desmo_last_error()
    rc, err = _call(shape, 1, [0], U=8)
    assert rc == 1 and "aligned" in err


# ------------------------------------------------------------------------------------------------ thresholds are prefixes
@pytest.mark.parametrize("name", ["traj_chan_r4p2", "traj_cyl_r4p3", "traj_fcyl_r2p2"])
def test_threshold_steps_reproduce_the_reference_masks(name):
    """On the trained parameters of the golden runs, every threshold of the reference's sweep removes a prefix of removal_order, and
    the prefix gives the reference's mask exactly."""
    from desmo_b200.sparsify import removal_order, threshold_steps

    fx, meta, modes, snap, prm = golden_case(name)
    for k in ("gates", "phi", "omega", "zall", "coefs", "periods"):
        if getattr(prm, k) is not None:
            setattr(prm, k, fx[f"step{meta['steps']}_{k}"].copy())
    norms = orc.term_norms(prm)
    order = removal_order(torch.from_numpy(norms), prm.T, prm.r)
    assert order == orc.removal_order(norms, prm.T, prm.r)
    steps = []
    for i, thr in enumerate(fx["sweep_thresholds"]):
        s = threshold_steps(norms, prm.gates, order, float(thr))
        mask = prm.gates != 0
        mask[order[:s]] = False
        assert np.array_equal(mask, fx["sweep_masks"][i]), thr
        assert int(mask.sum()) == int(fx["sweep_nonzero"][i])
        steps.append(s)
    assert steps == sorted(steps) and len(set(steps)) >= 4
    i = next(i for i, s in enumerate(steps) if 0 < s < prm.K and len(set(order[:s]) & set(order[::-1][:s])) < s)
    with pytest.raises(_lib.DesmoError):  # a threshold that removes terms out of this order's sequence
        threshold_steps(norms, prm.gates, order[::-1], float(fx["sweep_thresholds"][i]))


# ------------------------------------------------------------------------------------------------ scratch formula
def _scratch(n, m, r, p, steps, sms):
    """The formula of include/desmo_b200.h, restated."""
    shape = _lib.make_shape(n, m, r, p)
    T = _lib.load().desmo_num_terms(r, p)
    K = T + 3 * r
    A = lambda v: (v + 1023) // 1024 * 1024  # noqa: E731
    Kr, mp = (K + 63) // 64 * 64, (m + 127) // 128 * 128
    tiles_m = mp // 128
    gpt = min(max(sms // tiles_m, 1), shape.ld // 128)
    unit = 128 * gpt
    rows_c = min(max(CHUNK_BYTES // (6 * Kr + 4 * (steps + 1)) // unit * unit, unit), shape.ld)
    part = 1024 * tiles_m * gpt * (steps + 2)
    total = A(8 * T) + A(T) + A(6 * Kr * rows_c) + A(6 * Kr * mp) + A(4 * (steps + 1) * rows_c) + A(4 * (steps + 1) * mp) + A(part)
    return shape, total, part, tiles_m


@pytest.mark.parametrize("n,m,r,p,steps,sms", [
    (3 << 20, 1000, 4, 2, 27, 148),
    (262144, 1000, 32, 2, 657, 148),
    (262144, 1000, 32, 2, 100, 148),
    (1, 70, 8, 3, 189, 148),
    (4100, 1300, 4, 2, 0, 148),
    (700, 20000, 64, 1, 257, 148),
    (100000, 300, 8, 2, 69, 7),
])
def test_scratch_formula(n, m, r, p, steps, sms):
    shape, want, part, tiles_m = _scratch(n, m, r, p, steps, sms)
    got = C.c_size_t(0)
    assert _lib.load().desmo_pruning_profile_scratch_bytes(C.byref(shape), steps, sms, C.byref(got)) == 0
    assert got.value == want
    # bounded: one [steps + 2][128] fp64 partial per CTA, never one [steps + 2][m] per SM
    assert part <= (sms + tiles_m) * (steps + 2) * 1024
    if (n, m, steps) == (262144, 1000, 657):
        assert part < 100e6 and want < 200e6, (part, want)


def test_scratch_bytes_rejects_bad_arguments():
    shape = _lib.make_shape(1000, 50, 4, 2)
    got = C.c_size_t(0)
    lib = _lib.load()
    assert lib.desmo_pruning_profile_scratch_bytes(C.byref(shape), 28, 148, C.byref(got)) == 1
    assert lib.desmo_pruning_profile_scratch_bytes(C.byref(shape), 5, 0, C.byref(got)) == 1
    assert os.path.exists(_lib.HEADER_PATH)
