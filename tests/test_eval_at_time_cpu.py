"""CPU-side checks of evaluation at chosen instants: time_points against the t_point formula of csrc/library.cu, and the argument
validation that runs before anything touches a device."""
import ctypes as C

import numpy as np
import pytest

from desmo_b200 import _lib
from desmo_b200.engine import _instants, time_points

torch = pytest.importorskip("torch")


def _t_point(k, m):
    """t_point of csrc/library.cu in numpy fp32: step = m / (m - 1); k < m / 2 counts up from 0, the rest down from m."""
    f = np.float32
    step = f(m) / f(m - 1)
    return step * f(k) if k < m // 2 else f(m) - step * f(m - 1 - k)


@pytest.mark.parametrize("m", [2, 3, 1000, 1001])
def test_time_points_pin_the_device_formula(m):
    got = time_points(range(3 * m), m)
    assert got.dtype == np.float32 and got.shape == (3 * m,)
    for k in range(m):
        assert got[k] == _t_point(k, m), (m, k)
    step = np.float32(m) / np.float32(m - 1)
    for k in range(m, 3 * m):  # beyond the window the grid continues at the training spacing
        assert got[k] == step * np.float32(k), (m, k)
    assert got[0] == 0.0 and got[m - 1] == np.float32(m)
    assert np.all(np.diff(got) > 0)
    from oracle.desmo_oracle import t_points

    assert np.array_equal(got[:m], t_points(m))  # the reference's t_points as the oracle evaluates them


@pytest.mark.parametrize("m", [2, 3, 1000, 1001])
def test_agreement_with_torch_linspace_is_recorded_not_assumed(m):
    got = time_points(range(m), m)
    lin = torch.linspace(0, m, m).numpy()
    differ = np.flatnonzero(got != lin)
    if m <= 3:
        assert differ.size == 0  # every value is exact
    # where ATen's CPU kernel rounds differently it is by one ulp at most; the GPU tests check the device's own grid bit for bit
    assert np.all(np.abs(got[differ].astype(np.float64) - lin[differ]) <= np.spacing(np.float32(m)).astype(np.float64))
    print(f"m={m}: time_points differ from torch.linspace(0, m, m) at {differ.size} of {m} indices")


def test_time_points_reject_bad_input():
    with pytest.raises(_lib.DesmoError):
        time_points([0], 1)
    with pytest.raises(_lib.DesmoError):
        time_points([-1], 10)


def test_instants_validation():
    idx, t = _instants([3, 0, 3], None, 10, 0)
    assert t is None and idx.dtype == np.int32 and idx.tolist() == [3, 0, 3] and idx.flags.c_contiguous
    idx, t = _instants(None, [1.5, -2.0, 1e4], 10, 4)
    assert idx is None and t.dtype == np.float32
    assert _instants(range(2, 5), None, 10, 0)[0].tolist() == [2, 3, 4]
    assert _instants(torch.tensor([1, 2]), None, 10, 0)[0].tolist() == [1, 2]
    bad = [
        (None, None, 0), ([0], [0.0], 4),          # exactly one of index / times
        (None, [1.0], 0),                          # times on a free-row model
        ([10], None, 0), ([-1], None, 0),          # out of range
        ([], None, 0), (None, [], 4),              # empty
        ([1.5], None, 0),                          # not integers
        (None, [np.nan], 4), (None, [np.inf], 4), (None, [-np.inf], 4),
    ]
    for index, times, nF in bad:
        with pytest.raises(_lib.DesmoError):
            _instants(index, times, 10, nF)


def test_c_abi_validates_before_it_needs_a_device():
    lib = _lib.load()
    assert _lib.SIGNATURES["desmo_build_w_at"][1][5:7] == [_lib._i32, _lib._i32]
    fake = 1 << 12  # never dereferenced: every call below fails validation first
    s = _lib.make_shape(1000, 300, 4, 2, 0)
    sf = _lib.make_shape(1000, 300, 4, 2, 3)
    idx = np.array([0, 5, 299], np.int32)
    t = np.array([0.0, 1.0, 2.0], np.float32)

    def call(shape, m_out, mld_out, index, times, rows=fake, coefs=None, periods=None, gates=fake, W=fake):
        return lib.desmo_build_w_at(C.byref(shape), gates, rows, coefs, periods, m_out, mld_out,
                                    None if index is None else index.ctypes.data, None if times is None else times.ctypes.data, W, None, 0)

    cases = [
        (s, 0, 16, idx, None, {}),                                        # m_out >= 1
        (s, 3, 8, idx, None, {}),                                         # mld_out >= m_out ...
        (s, 3, 24, idx, None, {}),                                        # ... and a multiple of 16
        (s, 3, 16, None, None, {}),                                       # neither index nor times
        (sf, 3, 16, idx, t, {"coefs": fake, "periods": fake}),            # both
        (s, 3, 16, None, t, {}),                                          # times on DESMO
        (s, 3, 16, idx, None, {"rows": None}),                            # DESMO reads rows
        (sf, 3, 16, None, t, {"coefs": fake}),                            # Fourier needs periods
        (s, 3, 16, idx, None, {"W": None}),
        (s, 3, 16, np.array([0, 300, 1], np.int32), None, {}),            # index >= m
        (s, 3, 16, np.array([0, -1, 1], np.int32), None, {}),             # index < 0
        (sf, 3, 16, None, np.array([0.0, np.nan, 1.0], np.float32), {"coefs": fake, "periods": fake}),
        (sf, 3, 16, None, np.array([0.0, 1.0, np.inf], np.float32), {"coefs": fake, "periods": fake}),
    ]
    for shape, m_out, mld_out, index, times, kw in cases:
        assert call(shape, m_out, mld_out, index, times, **kw) == 1, (m_out, mld_out, kw, lib.desmo_last_error())
    assert b"index[1] = 300" in (call(s, 3, 16, np.array([0, 300, 1], np.int32), None) == 1 and lib.desmo_last_error())
    bad_shape = _lib.make_shape(1000, 1, 4, 2, 0)  # the model's shape is validated as everywhere else (m >= 2)
    assert call(bad_shape, 1, 16, np.array([0], np.int32), None) == 1
