"""CPU-side checks of training Fourier models at caller-given times: the host validation of desmo_time_points_prepare and of the
engine's time table, the ctypes declarations of the new entry points, the trainer's state_dict key, and tests/_times_oracle.py against
the existing oracle at the grid (bit for bit) and against fp64 finite differences elsewhere."""
import ctypes as C
import re

import numpy as np
import pytest

from desmo_b200 import _lib
from desmo_b200._lib import DesmoError
from desmo_b200.engine import _instants, time_table
from oracle import desmo_oracle as orc
from tests import _times_oracle as to

torch = pytest.importorskip("torch")


def _shape(nF=3, m=20, r=2, p=2, n=300):
    return _lib.make_shape(n, m, r, p, nF)


def _prepare(shape, times, count=None):
    lib = _lib.load()
    arr = (C.c_float * max(1, len(times)))(*times)
    # dummy device pointer: every case below is rejected on the host before anything is written
    rc = lib.desmo_time_points_prepare(C.byref(shape), C.addressof(arr), len(times) if count is None else count, 16, None)
    return rc, lib.desmo_last_error().decode()


# ------------------------------------------------------------------------------------------------ C ABI host validation
@pytest.mark.parametrize("case,msg", [
    ("desmo", "Fourier model"),
    ("short", "count = m"),
    ("long", "count = m"),
    ("nan", "not finite"),
    ("inf", "not finite"),
])
def test_prepare_rejects_bad_tables_on_the_host(case, msg):
    m = 20
    t = list(np.linspace(0.0, 1.0, m))
    shape = _shape()
    if case == "desmo":
        shape = _shape(nF=0)
    elif case == "short":
        t = t[:-1]
    elif case == "long":
        t = t + [2.0]
    elif case == "nan":
        t[7] = float("nan")
    elif case == "inf":
        t[m - 1] = float("-inf")
    rc, err = _prepare(shape, t)
    assert rc == 1 and msg in err, err  # DESMO_ERR_ARG


def test_prepare_null_pointers():
    lib = _lib.load()
    assert lib.desmo_time_points_prepare(C.byref(_shape()), None, 20, 16, None) == 1
    arr = (C.c_float * 20)()
    assert lib.desmo_time_points_prepare(C.byref(_shape()), C.addressof(arr), 20, None, None) == 1


@pytest.mark.parametrize("fn", ["desmo_build_w_times", "desmo_adamax_update_times", "desmo_assemble_grads_times"])
def test_times_entry_points_reject_a_table_on_free_rows(fn):
    lib = _lib.load()
    nargs = len(_lib.SIGNATURES[fn][1]) - 1
    args = [16] * nargs
    args[-2] = 16  # t_points: non-null
    rc = getattr(lib, fn)(C.byref(_shape(nF=0)), *args)
    assert rc == 1 and "Fourier model" in lib.desmo_last_error().decode()


# ------------------------------------------------------------------------------------------------ ctypes declarations
def _header_params(name):
    src = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^;]*)\)\s*;", src)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


@pytest.mark.parametrize("name", ["desmo_time_points_prepare", "desmo_build_w_times", "desmo_adamax_update_times",
                                  "desmo_assemble_grads_times"])
def test_ctypes_declarations_match_the_header(name):
    params = _header_params(name)
    res, args = _lib.SIGNATURES[name]
    assert res is C.c_int and len(args) == len(params)
    for decl, ct in zip(params, args):
        if decl.startswith("const desmo_shape*"):
            assert ct is _lib._SP
        elif "*" in decl:
            assert ct is C.c_void_p, decl
        elif decl.startswith("int32_t"):
            assert ct is C.c_int32, decl
        else:
            raise AssertionError(decl)
    # the extended calls take their base call's arguments, then (active, t_points, stream)
    base = {"desmo_build_w_times": "desmo_build_w", "desmo_adamax_update_times": "desmo_adamax_update",
            "desmo_assemble_grads_times": "desmo_assemble_grads"}.get(name)
    if base:
        assert params[:-3] == _header_params(base)[:-1]
        assert params[-3:] == ["const void* active", "const float* t_points", "void* stream"]
    assert name in _lib.declared_symbols()


# ------------------------------------------------------------------------------------------------ engine host validation
def test_time_table_validation():
    m = 6
    assert time_table([0, 1, 2, 3, 4, 5], m, 2).dtype == np.float32
    with pytest.raises(DesmoError, match="Fourier model"):
        time_table(np.arange(m, dtype=np.float32), m, 0)
    with pytest.raises(DesmoError, match="shape"):
        time_table(np.arange(m + 1, dtype=np.float32), m, 2)
    with pytest.raises(DesmoError, match="shape"):
        time_table(np.zeros((2, 3), np.float32), m, 2)
    with pytest.raises(DesmoError, match="finite"):
        time_table([0, 1, np.nan, 3, 4, 5], m, 2)
    with pytest.raises(DesmoError, match="real numbers"):
        time_table(np.ones(m, bool), m, 2)
    # fp64 input is rounded to nearest once; a tensor, an array and a sequence give the same table; order and repeats are free
    v = np.array([0.1, 1e-3, 7.3, 7.3, 2.0 / 3.0, -4.2])
    want = v.astype(np.float32)
    for x in (v, list(v), torch.from_numpy(v), torch.from_numpy(v).float()):
        assert np.array_equal(time_table(x, m, 2), want)


def test_instants_index_maps_to_the_table():
    table = np.array([0.5, 3.25, -1.0, 9.0], np.float32)
    idx, t = _instants(np.array([3, 0, 0]), None, 4, 2, table)
    assert idx is None and np.array_equal(t, table[[3, 0, 0]])
    with pytest.raises(DesmoError, match="0 .. 3"):
        _instants(np.array([4]), None, 4, 2, table)
    idx, t = _instants(None, [1.5], 4, 2, table)  # times= is not affected by the table
    assert idx is None and t.tolist() == [1.5]
    idx, t = _instants(np.array([1]), None, 4, 2, None)
    assert idx.tolist() == [1] and t is None


# ------------------------------------------------------------------------------------------------ trainer state_dict
class _Engine:
    """CPU stand-in with what DesmoTrainer's state_dict / load_state_dict touch (the real DesmoEngine needs a GPU)."""

    def __init__(self):
        self.n, self.m, self.r, self.polyorder, self.nF, self.n_global, self.K = 8, 4, 2, 2, 2, 8, 12
        z = lambda *s: torch.zeros(*s)  # noqa: E731
        for k in ("phi_m", "phi_u", "P"):
            setattr(self, k, z(self.r, 256))
        for k in ("gates_m", "gates_u", "periods_m", "periods_u"):
            setattr(self, k, z(self.K))
        self.rows_m, self.rows_u = z(self.K, 16), z(self.K, 16)
        self.coefs_m, self.coefs_u = z(self.K, 5), z(self.K, 5)
        self.omega_m, self.omega_u = z(6), z(6)
        self.step_dev = torch.zeros(1, dtype=torch.int32)
        self.device = torch.device("cpu")
        self.active_terms, self._active, self.t_points, self._times = None, None, None, None
        self.time_calls = []

    def set_hyper(self, *a):
        pass

    def set_active_terms(self, mask):
        self.active_terms = mask

    def set_time_points(self, t):
        self.time_calls.append(t)
        self.t_points = None if t is None else time_table(t, self.m, self.nF)


def test_trainer_state_dict_round_trip():
    from desmo_b200 import DesmoTrainer

    e = _Engine()
    tr = DesmoTrainer(e, use_cuda_graph=False)
    assert tr.state_dict()["t_points"] is None
    table = np.array([0.0, 0.7, 0.2, 5.5], np.float32)
    e.t_points = table.copy()
    sd = tr.state_dict()
    assert sd["t_points"].dtype == torch.float32 and np.array_equal(sd["t_points"].numpy(), table)
    e2 = _Engine()
    DesmoTrainer(e2, use_cuda_graph=False).load_state_dict(sd)
    assert np.array_equal(e2.t_points, table)
    # a checkpoint written before time tables existed loads as the grid
    old = {k: v for k, v in sd.items() if k != "t_points"}
    e3 = _Engine()
    e3.t_points = table.copy()
    DesmoTrainer(e3, use_cuda_graph=False).load_state_dict(old)
    assert e3.time_calls == [None] and e3.t_points is None


def test_sharded_checkpoint_keeps_the_table():
    from desmo_b200.checkpoint import scatter_trainer_state

    table = torch.tensor([0.0, 0.5, 2.0], dtype=torch.float32)
    sd = {"model": None, "optimizer": {"phi_m": torch.zeros(2, 10), "phi_u": torch.zeros(2, 10)}, "pod_modes": torch.zeros(2, 10),
          "shape": {"n": 10, "n_global": 10, "r": 2}, "t_points": table}
    for rank in range(3):
        assert torch.equal(scatter_trainer_state(sd, rank, 3)["t_points"], table)


# ------------------------------------------------------------------------------------------------ oracle
def _fourier_case(n=40, m=9, r=2, p=2, nF=3, period=None, seed=3):
    X = orc.synthetic_snapshots("cylinder", n, m, seed)
    modes, _, _, _ = orc.pod_analysis(X, r)
    prm = orc.perturb(orc.init_params(n, m, p, r, omega_init=10.0, nF=nF, period_init=period or 6.0), seed=5, rel=0.3)
    return modes, X.T.astype(np.float32), prm


def test_oracle_at_the_grid_is_the_existing_oracle_bit_for_bit():
    modes, snap, prm = _fourier_case()
    grid = orc.t_points(prm.m)
    a = orc.loss_and_grads(prm, modes, snap, 1e-3, 1e-4)
    b = to.loss_and_grads(prm, modes, snap, 1e-3, 1e-4, grid)
    assert a.mse == b.mse and a.total == b.total
    for k in a.grads:
        assert np.array_equal(a.grads[k], b.grads[k]), k
    assert np.array_equal(orc.temporal_rows(prm), to.fourier_rows(prm, grid))
    assert np.array_equal(orc.term_norms(prm), to.term_norms(prm, grid))
    ha, _, _ = orc.train(prm.copy(), modes, snap, 20, 1e-3, 1e-4, lrs=(1e-2, 1e-3, 1e-2, 1e-2, 1e-2))
    hb, _, _ = to.train(prm.copy(), modes, snap, 20, 1e-3, 1e-4, grid, lrs=(1e-2, 1e-3, 1e-2, 1e-2, 1e-2))
    assert np.array_equal(ha, hb)
    assert orc.t_points is not None and np.array_equal(orc.t_points(prm.m), grid)  # the oracle is restored


@pytest.mark.parametrize("kind", ["sorted_random", "seconds", "subset_unsorted_repeat"])
def test_oracle_gradients_at_other_times_match_finite_differences(kind):
    m = 9
    rng = np.random.default_rng(11)
    if kind == "sorted_random":
        t, period = np.sort(rng.uniform(0.0, m, m)), 6.0
    elif kind == "seconds":
        t, period = np.sort(rng.uniform(0.0, 1.3, m)), 1.0
    else:
        t = rng.permutation(orc.t_points(12))[:m].astype(np.float64)
        t[4] = t[1]
        period = 6.0
    t = t.astype(np.float32)
    modes, snap, prm = _fourier_case(m=m, period=period)
    q = prm.copy()
    for k in ("phi", "gates", "omega", "coefs", "periods"):
        setattr(q, k, getattr(q, k).astype(np.float64))
    g = to.loss_and_grads(q, modes.astype(np.float64), snap.astype(np.float64), 0.0, 0.0, t).grads
    # the table changes the answer: the rows are not the grid's
    assert not np.allclose(to.fourier_rows(prm, t), orc.temporal_rows(prm))
    for key, index in (("coefs", (0, 0)), ("coefs", (3, 1)), ("coefs", (prm.K - 1, 2 * prm.nF)), ("periods", 0), ("periods", prm.K - 2)):
        fd = to.finite_difference(prm, modes, snap, t, key, index, 1e-5 * max(1.0, abs(float(q.__dict__[key][index]))))
        an = float(g[key][index])
        assert abs(an - fd) <= 1e-6 * max(1.0, np.abs(g[key]).max()) + 1e-5 * abs(fd), (key, index, an, fd)
