"""Training DESMOFourier at caller-given times (DesmoEngine.set_time_points, desmo_*_times): a table equal to the grid is bit for bit
no table on every path, gradients and a 1000-step trajectory at non-uniform / physical / window / subset times against
tests/_times_oracle.py, evaluation, term norms, active sets, autograd, graphs, checkpoints, validation in fit, rejections, two GPUs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import desmo_oracle as orc
from tests import _times_oracle as to
from tests.helpers import engine_params, golden_case, load_engine, make_case, rel

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRAD_TOL = {"gates": 1e-5, "coefs": 1e-5, "periods": 5e-5, "phi": 5e-5, "omega": 5e-5}
BETA, LAM = 1e-3, 1e-4
STATE = ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "omega", "omega_m", "omega_u", "coefs", "coefs_m", "coefs_u",
         "periods", "periods_m", "periods_u", "losses", "step_dev", "W")
U32 = 2.0 ** -24
SNAP_BOUND, ETA = 9 * U32, 2.0 ** -14  # desmo_residual_profile's documented bound; recon of the fp32 paths vs exact (f6)


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _engine(prm, modes, snap, path=0, t_points=None, snapshot_dtype=torch.float32):
    from desmo_b200 import DesmoEngine

    e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF, device=_dev(), path=path, snapshot_dtype=snapshot_dtype,
                    t_points=t_points)
    load_engine(e, prm, modes, snap)
    return e


def _f64(prm):
    q = prm.copy()
    for k, v in q.__dict__.items():
        if isinstance(v, np.ndarray):
            setattr(q, k, v.astype(np.float64))
    return q


def _times(kind, M, seed=0):
    """(time table, snapshot rows of the M-snapshot grid data it belongs to, or None when the data are taken as they are)."""
    rng = np.random.default_rng(seed)
    grid = orc.t_points(M)
    if kind == "sorted_random":
        return np.sort(rng.uniform(0.0, M, M)).astype(np.float32), None
    if kind == "seconds":  # the same flow sampled over 1.3 s, periods near 1
        return np.sort(rng.uniform(0.0, 1.3, M)).astype(np.float32), None
    m = int(0.8 * M)
    if kind == "first80":
        return grid[:m].copy(), np.arange(m)
    if kind == "subset80":  # a random 80 % of the snapshots, unsorted, one of them twice
        rows = rng.permutation(M)[:m]
        rows[m // 2] = rows[1]
        return grid[rows], rows
    raise KeyError(kind)


def _case(name, kind):
    """A Fourier case at a kind of times: (modes, snapshot rows, params with m = the table's length, table)."""
    if name.startswith("grad_"):
        _, meta, modes, snap, prm = golden_case(name)
    else:  # a GEMM-path Fourier library
        _, modes, snap, prm = make_case("cylinder", 900, 120, 4, 3, 3, period_init=60.0, omega_init=2.0, perturb_rel=0.2)
    t, rows = _times(kind, prm.m)
    if kind == "seconds":
        prm.periods = (prm.periods / np.float32(prm.periods.mean())).astype(np.float32)
    if rows is not None:
        snap = np.ascontiguousarray(snap[rows])
        prm.m = len(rows)
    return modes, snap, prm, t


def _check_grads(e, prm, modes, snap, t, active=None):
    out = to.loss_and_grads(_f64(prm), modes, snap.astype(np.float64), BETA, LAM, t, active=active)
    # dphi and d omega do not see the table (the spatial chain rule is generic in W); their fp32 sums cancel, and the fp32 oracle itself
    # misses fp64 by up to 2e-4 on these cases, at the grid too: their gate is the larger of 5e-5 and twice that floor
    out32 = to.loss_and_grads(prm, modes.astype(np.float32), snap, BETA, LAM, t, active=active)
    g = e.gradients(beta=BETA, l1_lambda=LAM)
    losses = e.losses.cpu().numpy()
    assert abs(losses[0] - out.mse) <= 1e-5 * abs(out.mse)
    assert abs(losses[3] - out.total) <= 1e-5 * abs(out.total)
    for k, ref in out.grads.items():
        got = np.asarray(g[k].cpu().numpy(), np.float64)
        tol = GRAD_TOL[k]
        if k in ("phi", "omega"):
            tol = max(tol, 2.0 * np.linalg.norm(out32.grads[k] - ref) / max(np.linalg.norm(ref), 1e-300))
        scale = np.linalg.norm(ref)
        if active is not None and k == "periods":  # as tests/test_active_terms.py: relative to the whole library's period gradient
            scale = max(scale, np.linalg.norm(to.loss_and_grads(_f64(prm), modes, snap.astype(np.float64), BETA, LAM, t).grads[k]))
        err = np.linalg.norm(got - ref) / max(scale, 1e-300)
        assert err < tol, (k, err, tol)


def _equal_state(a, b, keys=STATE):
    for k in keys:
        x, y = getattr(a, k), getattr(b, k)
        if x is not None:
            assert torch.equal(x, y), k


# ------------------------------------------------------------------------------------------------ 1. the grid table is no table
@pytest.mark.parametrize("path,m", [(1, 60), (2, 90), (3, 90)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_grid_table_is_bit_identical_to_no_table(path, m, dtype):
    from desmo_b200 import DesmoTrainer

    # m < 128 on the FFMA path: one time slab (its multi-slab launches add with float atomics)
    _, modes, snap, prm = make_case("cylinder", 700, m, 2, 2, 4, omega_init=2.0, perturb_rel=0.2)
    ea = _engine(prm, modes, snap, path, snapshot_dtype=dtype)
    eb = _engine(prm, modes, snap, path, t_points=orc.t_points(m), snapshot_dtype=dtype)
    assert ea.path_used == path
    lrs = (1e-2, 1e-3, 1e-2, 1e-2, 1e-2)
    ta, tb = (DesmoTrainer(e, lrs=lrs, beta=BETA, l1_lambda=LAM, sched_every=10) for e in (ea, eb))
    for _ in range(50):
        ta.step()
        tb.step()
    torch.cuda.synchronize()
    _equal_state(ea, eb)
    assert [h[1:] for h in ta.history] == [h[1:] for h in tb.history]


# ------------------------------------------------------------------------------------------------ 2. gradients
@pytest.mark.parametrize("kind", ["sorted_random", "seconds", "first80", "subset80"])
@pytest.mark.parametrize("name,path", [("grad_fcyl_r2p2", 0), ("grad_faneu_r2p2", 0), ("gemm_fr4p3", 3)])
def test_gradients_match_oracle(name, path, kind):
    modes, snap, prm, t = _case(name, kind)
    e = _engine(prm, modes, snap, path, t_points=t)
    if path == 0:
        assert e.path_used == 2  # the fused tcgen05 kernel
    _check_grads(e, prm, modes, snap, t)


@pytest.mark.parametrize("path", [1, 3])
def test_gradients_on_an_active_set_match_oracle(path):
    modes, snap, prm, t = _case("grad_fcyl_r2p2" if path == 1 else "gemm_fr4p3", "subset80")
    mask = np.random.default_rng(2).random(prm.K) < 0.5
    mask[0] = True
    e = _engine(prm, modes, snap, path, t_points=t)
    e.set_active_terms(mask)
    before = (e.coefs.clone(), e.periods.clone())
    _check_grads(e, prm, modes, snap, t, active=mask)
    from desmo_b200 import DesmoTrainer

    tr = DesmoTrainer(e, lrs=(1e-2, 1e-3, 1e-2, 1e-2, 1e-2))
    for _ in range(10):
        tr.step()
    torch.cuda.synchronize()
    fz = torch.from_numpy(~mask).to(e.device)
    assert torch.equal(e.coefs[fz], before[0][fz]) and torch.equal(e.periods[fz], before[1][fz])  # absent terms stay frozen


# ------------------------------------------------------------------------------------------------ 3. trajectory
@pytest.mark.parametrize("path", [0, 3])
def test_trajectory_matches_oracle(path):
    from desmo_b200 import DesmoTrainer

    _, modes, snap, prm = make_case("cylinder", 180, 60, 2, 2, 3, period_init=20.0, omega_init=10.0, perturb_seed=43, perturb_rel=0.02)
    t = np.sort(np.random.default_rng(5).uniform(0.0, 60.0, 60)).astype(np.float32)
    lrs = (1e-2, 1e-3, 1e-2, 1e-2, 1e-2)
    e = _engine(prm, modes, snap, path, t_points=t)
    tr = DesmoTrainer(e, lrs=lrs, beta=BETA, l1_lambda=LAM, patience=50, sched_every=10)
    ref = prm.copy()
    to.train(ref, modes, snap, 1000, BETA, LAM, t, patience=50, sched_every=10, lrs=lrs)
    for _ in range(1000):
        tr.step()
    torch.cuda.synchronize()
    got = engine_params(e)
    for k in ("gates", "phi", "omega", "coefs", "periods"):
        assert rel(got[k], getattr(ref, k)) < 1e-3, (k, rel(got[k], getattr(ref, k)))


# ------------------------------------------------------------------------------------------------ 4. evaluation
@pytest.mark.parametrize("path", [0, 3])
def test_evaluation_at_the_table(path):
    from desmo_b200._lib import DesmoError

    modes, snap, prm, t = _case("grad_fcyl_r2p2" if path == 0 else "gemm_fr4p3", "subset80")
    e = _engine(prm, modes, snap, path, t_points=t)
    rec = e.reconstruct()
    rows = e.rows[:, :e.m].clone()
    k = np.array([3, 0, e.m - 1, 3])
    assert torch.equal(e.reconstruct_at(index=k), rec[k])
    assert torch.equal(e.temporal_rows_at(index=np.arange(e.m)), rows)
    assert np.array_equal(e.time_points(k), t[k])
    with pytest.raises(DesmoError):
        e.time_points([e.m])
    with pytest.raises(DesmoError):
        e.reconstruct_at(index=[e.m])
    # times= between and beyond the table agree with fp64
    ts = np.array([-3.5, 0.25, 17.125, 1.5 * float(t.max())], np.float32)
    q = _f64(prm)
    q.m = ts.size
    assert rel(e.temporal_rows_at(times=ts).cpu().numpy(), to.fourier_rows(q, ts)) < 1e-5
    # the rows against fp64 at the table itself
    assert rel(rows.cpu().numpy(), to.fourier_rows(_f64(prm), t)) < 1e-5


def test_held_out_profile_on_the_left_out_snapshots():
    """Train on a random 80 % at their true times, then score the other 20 % against fp64 sums."""
    _, modes, snap_all, prm = make_case("cylinder", 900, 120, 4, 3, 3, period_init=60.0, omega_init=2.0, perturb_rel=0.2)
    M = prm.m
    rows = np.random.default_rng(4).permutation(M)
    fit, out = np.sort(rows[:int(0.8 * M)]), rows[int(0.8 * M):]
    grid = orc.t_points(M)
    prm.m = fit.size
    e = _engine(prm, modes, np.ascontiguousarray(snap_all[fit]), 3, t_points=grid[fit])
    held = torch.from_numpy(np.ascontiguousarray(snap_all[out]))
    got = e.residual_profile_at(held, times=grid[out])
    q = _f64(prm)
    q.m = out.size
    with to.at_times(grid[out]):
        recon, _, _ = orc.forward(q, modes.astype(np.float64))
    r = recon - snap_all[out].astype(np.float64)
    ref_r2, ref_u2 = (r ** 2).sum(axis=1), (snap_all[out].astype(np.float64) ** 2).sum(axis=1)
    recon2 = (recon ** 2).sum(axis=1)
    g_r2, g_u2 = got["snapshot_residual2"].cpu().numpy(), got["snapshot_norm2"].cpu().numpy()
    assert np.all(np.abs(g_u2 - ref_u2) <= SNAP_BOUND * ref_u2)
    bound = SNAP_BOUND * ref_r2 + 2 * ETA * np.sqrt(ref_r2 * recon2) + ETA ** 2 * recon2
    assert np.all(np.abs(g_r2 - ref_r2) <= bound), np.max(np.abs(g_r2 - ref_r2) / bound)


# ------------------------------------------------------------------------------------------------ 5. term norms and masks
@pytest.mark.parametrize("path", [0, 3])
def test_term_norms_and_threshold_masks_at_the_table(path):
    from desmo_b200 import DESMOFourier
    from desmo_b200.sparsify import threshold_sweep

    modes, snap, prm, t = _case("grad_fcyl_r2p2" if path == 0 else "gemm_fr4p3", "sorted_random")
    model = DESMOFourier(prm.n, prm.m, prm.polyorder, prm.r, 2.0, prm.nF, pod_modes=modes, device=_dev(), path=path, t_points=t)
    load_engine(model.engine, prm, modes, snap)
    got = model.engine.term_norms().cpu().numpy()
    # against the fp32 oracle, the gate of the golden term norms (tests/test_gpu_parity.py); the fp32 library itself is 1.3e-5 off fp64 here
    ref = to.term_norms(prm, t)
    assert rel(got, ref) < 5e-6
    assert not np.allclose(ref, orc.term_norms(prm))  # the times matter
    thresholds = list(np.quantile(ref, [0.1, 0.3, 0.5, 0.7, 0.9]))
    for thr, _, _, mask in threshold_sweep(model, float((snap.astype(np.float64) ** 2).sum()), thresholds):
        want = orc.active_mask(got.astype(np.float64), prm.gates, thr)
        assert np.array_equal(mask.cpu().numpy(), want)
        assert np.array_equal(want, orc.active_mask(ref, prm.gates, thr)) or np.min(np.abs(ref - thr)) < 1e-4 * thr


# ------------------------------------------------------------------------------------------------ 6. combinations
def test_autograd_module_route_at_the_table():
    from desmo_b200 import DESMOFourier

    modes, snap, prm, t = _case("grad_fcyl_r2p2", "sorted_random")
    model = DESMOFourier(prm.n, prm.m, prm.polyorder, prm.r, 2.0, prm.nF, pod_modes=modes, device=_dev(), t_points=torch.from_numpy(t))
    load_engine(model.engine, prm, modes, snap)
    x = torch.from_numpy(snap).to(model.engine.device)
    recon, _, _ = model(x)
    torch.nn.functional.mse_loss(recon, x).backward()
    ref = to.loss_and_grads(_f64(prm), modes, snap.astype(np.float64), 0.0, 0.0, t).grads
    T = prm.T
    got_c = np.stack([p.grad.cpu().numpy() for p in model.z_list])
    got_p = np.concatenate([p.grad.cpu().numpy() for p in model.period_list])
    assert rel(got_c, ref["coefs"][:T]) < 1e-5 and rel(got_p, ref["periods"][:T]) < 5e-5
    assert rel(model.c_coef.grad.cpu().numpy(), ref["gates"][:T]) < 1e-5


def test_graph_replay_equals_eager_and_follows_an_in_place_table():
    from desmo_b200 import DesmoTrainer

    modes, snap, prm, t = _case("grad_faneu_r2p2", "sorted_random")
    t2 = (t * np.float32(1.5)).astype(np.float32)
    ea, eb = _engine(prm, modes, snap, 0, t_points=t), _engine(prm, modes, snap, 0, t_points=t)
    ta, tb = DesmoTrainer(ea, use_cuda_graph=True), DesmoTrainer(eb, use_cuda_graph=False)
    for i in range(20):
        if i == 10:  # rewritten in place: the captured graph reads the new table without a re-capture
            graph = ta._graph
            ea.set_time_points(t2)
            eb.set_time_points(t2)
        ta.step()
        tb.step()
    torch.cuda.synchronize()
    assert ta._graph is graph
    _equal_state(ea, eb)


def test_graph_is_recaptured_and_none_restores_the_grid():
    from desmo_b200 import DesmoTrainer

    modes, snap, prm, t = _case("grad_faneu_r2p2", "sorted_random")
    ea, eb = _engine(prm, modes, snap, 0, t_points=t), _engine(prm, modes, snap, 0)
    ta, tb = DesmoTrainer(ea), DesmoTrainer(eb)
    ta.step()
    g1 = ta._graph
    load_engine(ea, prm, modes, snap)
    ea.set_time_points(None)
    assert ea.t_points is None and ea.time_points([1]).tolist() == orc.t_points(prm.m)[[1]].tolist()
    ta.epoch, ta.history = 0, []
    for _ in range(10):
        ta.step()
        tb.step()
    torch.cuda.synchronize()
    assert ta._graph is not g1
    _equal_state(ea, eb)


def test_checkpoint_resume_is_exact_and_old_checkpoints_load_as_the_grid():
    from desmo_b200 import DESMOFourier, DesmoTrainer

    modes, snap, prm, t = _case("grad_fcyl_r2p2", "first80")

    def fresh(table):
        model = DESMOFourier(prm.n, prm.m, prm.polyorder, prm.r, 2.0, prm.nF, pod_modes=modes, device=_dev(), t_points=table)
        load_engine(model.engine, prm, modes, snap)
        return model, DesmoTrainer(model)

    ma, ta = fresh(t)
    for _ in range(20):
        ta.step()
    mb, tb = fresh(t)
    for _ in range(10):
        tb.step()
    sd = tb.state_dict()
    assert np.array_equal(sd["t_points"].numpy(), t)
    mc, tc = fresh(None)
    tc.load_state_dict(sd)
    assert np.array_equal(mc.t_points, t)
    for _ in range(10):
        tc.step()
    torch.cuda.synchronize()
    _equal_state(ma.engine, mc.engine)
    old = {k: v for k, v in sd.items() if k != "t_points"}
    md, td = fresh(t)
    td.load_state_dict(old)
    assert md.t_points is None and md.engine._times is None


def test_validation_curve_in_fit():
    from desmo_b200 import DesmoTrainer
    from desmo_b200.trainer import Validation

    _, modes, snap_all, prm = make_case("cylinder", 700, 90, 2, 2, 4, omega_init=2.0, perturb_rel=0.2)
    rows = np.random.default_rng(1).permutation(90)
    fit, out = rows[:72], rows[72:]
    grid = orc.t_points(90)
    prm.m = fit.size
    snap = np.ascontiguousarray(snap_all[fit])
    e = _engine(prm, modes, snap, 0, t_points=grid[fit])
    held = torch.from_numpy(np.ascontiguousarray(snap_all[out]))
    tr = DesmoTrainer(e)
    for _ in range(3):
        hist = tr.fit(torch.from_numpy(snap), 4, validation=(held, grid[out]), val_every=2)
        v = hist[-1]
        assert isinstance(v, Validation) and v.epoch == tr.epoch
        prof = e.residual_profile_at(held, times=grid[out])
        r2, u2 = float(prof["snapshot_residual2"].sum()), float(prof["snapshot_norm2"].sum())
        assert (v.residual2, v.norm2, v.rel_error) == (r2, u2, (r2 / u2) ** 0.5)
    vals = [h for h in tr.history if isinstance(h, Validation)]
    assert [v.epoch for v in vals] == [2, 4, 6, 8, 10, 12]
    assert len([h for h in tr.history if not isinstance(h, Validation)]) == 2  # the loss entries are unchanged (epochs 0, 10)


def test_bad_input_raises_before_anything_is_written():
    from desmo_b200 import DESMO, DesmoEngine
    from desmo_b200._lib import DesmoError

    modes, snap, prm, t = _case("grad_faneu_r2p2", "sorted_random")
    e = _engine(prm, modes, snap, 0, t_points=t)
    buf = e._times.clone()
    for bad in (np.r_[t[:-1], np.nan], t[:-1], np.r_[t, 1.0], np.full(prm.m, np.inf)):
        with pytest.raises(DesmoError):
            e.set_time_points(bad)
        torch.cuda.synchronize()
        assert torch.equal(e._times, buf) and np.array_equal(e.t_points, t)
    with pytest.raises(DesmoError):
        DESMO(prm.n, prm.m, 2, 2, device=_dev(), t_points=t)
    with pytest.raises(DesmoError):
        DesmoEngine(prm.n, prm.m, 2, 2, device=_dev(), t_points=t)


def test_ops_route_equals_engine():
    from desmo_b200 import ops

    modes, snap, prm, t = _case("gemm_fr4p3", "subset80")
    ea, eb = _engine(prm, modes, snap, 3, t_points=t), _engine(prm, modes, snap, 3, t_points=t)
    mask = np.ones(prm.K, bool)
    mask[5] = False
    ea.set_active_terms(mask)
    eb.set_active_terms(mask)
    for _ in range(5):
        ea.train_step()
        ops.engine_step_via_ops(eb)
    torch.cuda.synchronize()
    _equal_state(ea, eb)
    assert rel(ops.engine_term_norms_via_ops(eb).cpu().numpy(), ea.term_norms().cpu().numpy()) < 1e-6  # colnorm2 sums with float atomics
    table = torch.empty(prm.m, device=ea.device)
    torch.ops.desmo_b200.time_points_prepare(torch.from_numpy(t), table, *ops._shape_args(ea))
    assert torch.equal(table, ea._times)


def test_sharded_steps_share_the_table():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29681", os.path.join(ROOT, "tests", "_time_points_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("TIMES_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("TIMES_RESULT "):])
    assert res["rel_vs_unsharded"] < 1e-4, res
    assert res["identical_across_ranks"] and res["mismatch_raised"], res
