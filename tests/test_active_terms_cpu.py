"""CPU-side checks of training on an active set of library terms: the host validation of desmo_active_terms_prepare and of
set_active_terms' mask, the table-size formula, the trainer's state_dict round trip, and the oracle's masked gradients against
finite differences."""
import ctypes as C

import numpy as np
import pytest

from desmo_b200 import _lib
from desmo_b200.engine import active_indices
from oracle import desmo_oracle as orc
from tests import _active_oracle as ao

torch = pytest.importorskip("torch")


def _shape(r=4, p=2, n=300, m=20):
    return _lib.make_shape(n, m, r, p)


def _prepare(shape, idx, count=None):
    lib = _lib.load()
    arr = (C.c_int32 * max(1, len(idx)))(*idx)
    # dummy device pointer: every case below is rejected on the host before anything is written
    rc = lib.desmo_active_terms_prepare(C.byref(shape), C.addressof(arr), len(idx) if count is None else count, 16, None)
    return rc, lib.desmo_last_error().decode()


@pytest.mark.parametrize("idx,msg", [
    ([], "1 .. K"),
    ([0, 27], "outside"),
    ([-1, 3], "outside"),
    ([2, 2, 5], "repeats"),
    ([5, 2], "strictly increasing"),
])
def test_prepare_rejects_bad_sets_on_the_host(idx, msg):
    rc, err = _prepare(_shape(), idx)
    assert rc == 1 and msg in err, err  # DESMO_ERR_ARG


def test_prepare_rejects_more_terms_than_the_library():
    rc, err = _prepare(_shape(), list(range(27)), count=28)
    assert rc == 1 and "1 .. K" in err


def test_prepare_null_pointers():
    lib = _lib.load()
    arr = (C.c_int32 * 1)(0)
    assert lib.desmo_active_terms_prepare(C.byref(_shape()), None, 1, 16, None) == 1
    assert lib.desmo_active_terms_prepare(C.byref(_shape()), C.addressof(arr), 1, None, None) == 1


@pytest.mark.parametrize("r,p", [(2, 2), (4, 2), (4, 3), (8, 2), (32, 2)])
def test_table_size_formula(r, p):
    lib = _lib.load()
    K = lib.desmo_num_terms(r, p) + 3 * r
    for count in (1, K // 2 or 1, K):
        nb = C.c_size_t(0)
        assert lib.desmo_active_terms_bytes(C.byref(_shape(r, p)), count, C.byref(nb)) == 0
        assert nb.value == 4 * (K + count)
    for bad in (0, K + 1):
        assert lib.desmo_active_terms_bytes(C.byref(_shape(r, p)), bad, C.byref(nb)) == 1


def test_mask_validation():
    K = 27
    m = np.zeros(K, bool)
    m[[0, 5, 26]] = True
    got = active_indices(m, K)
    assert got.dtype == np.int32 and got.tolist() == [0, 5, 26]
    assert active_indices(torch.from_numpy(m), K).tolist() == [0, 5, 26]
    for bad in (np.ones(K - 1, bool), np.ones(K + 1, bool), np.ones(K, np.int32), np.ones(K, np.float32), np.zeros(K, bool),
                torch.ones(K, dtype=torch.uint8), np.ones((1, K), bool)):
        with pytest.raises(_lib.DesmoError):
            active_indices(bad, K)


# ------------------------------------------------------------------------------------------------ trainer state_dict
class _Engine:
    """CPU stand-in with what DesmoTrainer's state_dict / load_state_dict touch (the real DesmoEngine needs a GPU)."""

    def __init__(self):
        self.n, self.m, self.r, self.polyorder, self.nF, self.n_global, self.K = 8, 4, 2, 2, 0, 8, 12
        z = lambda *s: torch.zeros(*s)  # noqa: E731
        for k in ("phi_m", "phi_u", "P"):
            setattr(self, k, z(self.r, 256))
        for k in ("gates_m", "gates_u"):
            setattr(self, k, z(self.K))
        for k in ("rows_m", "rows_u"):
            setattr(self, k, z(self.K, 16))
        self.omega_m, self.omega_u = z(6), z(6)
        self.coefs_m = self.coefs_u = self.periods_m = self.periods_u = None
        self.step_dev = torch.zeros(1, dtype=torch.int32)
        self.device = torch.device("cpu")
        self.active_terms, self._active = None, None
        self.set_calls = []

    def set_hyper(self, *a):
        pass

    def set_active_terms(self, mask):
        self.set_calls.append(mask)
        self.active_terms = None if mask is None else mask.clone()


def test_trainer_state_dict_round_trip():
    from desmo_b200 import DesmoTrainer

    e = _Engine()
    tr = DesmoTrainer(e, use_cuda_graph=False)
    sd = tr.state_dict()
    assert sd["active_terms"] is None
    mask = torch.zeros(e.K, dtype=torch.bool)
    mask[[0, 3, 7]] = True
    e.active_terms = mask.clone()
    sd = tr.state_dict()
    assert torch.equal(sd["active_terms"], mask)
    e2 = _Engine()
    DesmoTrainer(e2, use_cuda_graph=False).load_state_dict(sd)
    assert torch.equal(e2.active_terms, mask)
    # a checkpoint written before active sets existed loads unmasked
    old = {k: v for k, v in sd.items() if k != "active_terms"}
    e3 = _Engine()
    e3.active_terms = mask.clone()
    DesmoTrainer(e3, use_cuda_graph=False).load_state_dict(old)
    assert e3.set_calls == [None] and e3.active_terms is None


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("nF", [None, 2])
def test_oracle_masked_gradients_match_finite_differences(nF):
    n, m, r, p = 40, 7, 2, 2
    X = orc.synthetic_snapshots("cylinder", n, m, 3)
    modes, _, _, _ = orc.pod_analysis(X, r)
    snap = X.T.astype(np.float64)
    prm = orc.perturb(orc.init_params(n, m, p, r, omega_init=2.0, nF=nF, period_init=9.0, dtype=np.float64), seed=5, rel=0.2)
    K = prm.K
    active = np.ones(K, bool)
    active[[1, 4, prm.T + 1, prm.T + r + 0]] = False  # two monomials, a sin and a cos term
    beta, lam = 1e-3, 1e-4
    out = ao.loss_and_grads(prm, modes, snap, beta, lam, active=active)
    fms = ao.frozen_masks(prm, active)
    h = 1e-6
    for name in ("gates", "omega", "phi", "coefs" if nF else "zall") + (("periods",) if nF else ()):
        arr = getattr(prm, name)
        g = out.grads[name]
        if name in fms:
            assert np.all(g[~fms[name]] == 0.0), name
        flat = arr.reshape(-1)
        for j in np.random.default_rng(0).choice(flat.size, size=min(flat.size, 12), replace=False):
            if name in fms and not fms[name].reshape(-1)[j]:
                continue
            old = flat[j]
            flat[j] = old + h
            up = ao.loss_and_grads(prm, modes, snap, beta, lam, want_grads=False, active=active).total
            flat[j] = old - h
            dn = ao.loss_and_grads(prm, modes, snap, beta, lam, want_grads=False, active=active).total
            flat[j] = old
            fd = (up - dn) / (2 * h)
            assert abs(fd - g.reshape(-1)[j]) <= 1e-5 * max(1.0, abs(fd)), (name, j, fd, g.reshape(-1)[j])
    # the frozen entries do not enter the loss at all
    q = prm.copy()
    q.gates[~active] = 123.0
    q.omega[~fms["omega"]] = -7.0
    assert ao.loss_and_grads(q, modes, snap, beta, lam, want_grads=False, active=active).total == out.total


def test_oracle_adamax_leaves_frozen_entries_alone():
    n, m, r, p = 30, 6, 2, 2
    X = orc.synthetic_snapshots("cylinder", n, m, 1)
    modes, _, _, _ = orc.pod_analysis(X, r)
    prm = orc.perturb(orc.init_params(n, m, p, r, omega_init=2.0), seed=2, rel=0.2)
    active = np.zeros(prm.K, bool)
    active[[0, 2, prm.T + 2 * r + 1]] = True
    before = prm.copy()
    opt = orc.Adamax(prm)
    opt.exp_avg["gates"][:] = 0.5  # old momentum must not move a frozen gate
    opt.exp_inf["gates"][:] = 1.0
    ao.train(prm, modes, X.T.astype(np.float32), 3, 1e-3, 1e-4, active=active, opt=opt)
    fms = ao.frozen_masks(before, active)
    for k, fm in fms.items():
        assert np.array_equal(getattr(prm, k)[~fm], getattr(before, k)[~fm]), k
        assert np.all(opt.exp_avg[k][~fm] == (0.5 if k == "gates" else 0.0)), k
        assert not np.array_equal(getattr(prm, k)[fm], getattr(before, k)[fm]), k
    assert not np.array_equal(prm.phi, before.phi)
