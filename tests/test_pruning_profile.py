"""Pruning profile (DesmoEngine.pruning_profile, sparsify.pruning_profile, desmo_pruning_profile): sum_x r_s(x, t)^2 for every step s of
a term-removal order, in one pass over U.

Error model (u = 2^-24, fp32 unit roundoff).  Let r_s be what the kernel forms for element (x, t) at step s and q_s the residual that
residual_profile() forms with the gates of order[:s] zeroed (or the exact fp64 residual, for the reference checks).
  - Each step is one FFMA, r_s = fl(r_{s-1} - a_s b_s): one rounding of at most u |r_s|, so s steps add at most u sum_{j<=s} |r_j|.
  - Both routes run GEMM 1 on the split-bf16 planes; each product sum is within EPS_GEMM * sum_k |G_k W_k| of the exact sum (the three
    plane products the split drops are 2^-23 of it; the tensor core's truncating fp32 accumulation stays below 2^-18 of it for these
    K).  Against residual_profile the two GEMMs (with and without the removed terms) both err: 2 EPS_GEMM.
  - r_0 = fl(Rec - U): one more u |r_0| on each side.
So |r_s - q_s| <= delta = 2u sum_{j<=s} |r_j| + 2 EPS_GEMM sum_k |G_k W_k| (+ the library's own fp32 evaluation, (p + 4) u per term,
against fp64 POOL_DATA; absolute for sin / cos / tanh).  With D = sum_x delta^2, Cauchy-Schwarz bounds the sums of squares: |sum r^2 - sum q^2| <= 2 sqrt(D Q) + D.
Summation: the kernel sums fp32 over a thread's 64 points (8 chains of 8 and a 3-level tree, plus the square: 12u), fp64 beyond;
residual_profile's own sums are within 9u.  Both are added to the bound."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import desmo_oracle as orc
from tests.helpers import golden_case, load_engine, make_case

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U32 = 2.0 ** -24
EPS_GEMM = 2.0 ** -18
SUM_P, SUM_R = 12 * U32, 9 * U32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _engine(kind, n, m, r, p, nF=None, dtype=torch.float32, perturb_rel=0.3):
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case(kind, n, m, r, p, nF=nF, omega_init=10.0, perturb_rel=perturb_rel)
    e = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF, device=torch.device(DEV), snapshot_dtype=dtype)
    load_engine(e, prm, modes, snap)
    return e


def _random_engine(n, m, r, p, seed=0):
    """Seeded parameters and data for shapes POD cannot give (n < r): U = recon(params) * (1 + 0.3 noise)."""
    from desmo_b200 import DesmoEngine

    g = torch.Generator(device=DEV).manual_seed(seed)
    e = DesmoEngine(n, m, p, r, omega_init=3.0, device=torch.device(DEV))
    e.P[:, :n] = torch.randn(r, n, device=DEV, generator=g) * 0.5
    e.phi[:, :n] = 1.0 + 0.2 * torch.randn(r, n, device=DEV, generator=g)
    e.gates.copy_(1.0 + 0.2 * torch.randn(e.K, device=DEV, generator=g))
    e.rows[:, :m] = torch.randn(e.K, m, device=DEV, generator=g)
    e.set_snapshot(torch.zeros(m, n))
    rec = e.reconstruct()
    e.set_snapshot(rec * (1.0 + 0.3 * torch.randn(m, n, device=DEV, generator=g)))
    return e


def _library64(e):
    """The library in fp64, (n, K) in packed K order: the oracle's POOL_DATA, then sin / cos / tanh of omega * Phi per mode."""
    lat = (e.phi[:, :e.n].double() * e.P[:, :e.n].double()).t().cpu().numpy()
    om = e.omega.double().cpu().numpy()
    cols = [orc.pool_data(lat, e.polyorder)]
    for b, f in enumerate((np.sin, np.cos, np.tanh)):
        cols.append(np.stack([f(om[3 * i + b] * lat[:, i]) for i in range(e.r)], axis=1))
    return torch.from_numpy(np.concatenate(cols, axis=1)).to(DEV)


def _order(e, S=None, seed=1):
    """The greedy removal order, or a seeded shuffle of the terms cut to S."""
    from desmo_b200.sparsify import removal_order

    order = removal_order(e.term_norms(), e.T, e.r)
    if S is not None:
        order = np.random.default_rng(seed).permutation(order)[:S].tolist()
    return [int(k) for k in order]


def _peel64(e, order):
    """fp64 quantities of the error model for every step: Q_exact[s][t] = sum_x (G W_s - U)^2, A[s][t] = sum_x delta_s^2 terms."""
    G = _library64(e)  # (n, K)
    e.build_w(False)
    W = e.W[:e.K, :e.m].double()
    u = e.U[:, :e.n].double().t()  # (n, m)
    r = G @ W - u
    absgw = G.abs() @ W.abs()
    q, run, abs_sum = [(r ** 2).sum(0)], r.clone(), torch.zeros_like(r)
    rs_abs = [abs_sum.clone()]
    for k in order:
        run -= torch.outer(G[:, k], W[k])
        abs_sum += run.abs()
        q.append((run ** 2).sum(0))
        rs_abs.append(abs_sum.clone())
    return torch.stack(q), rs_abs, absgw, r


def _cs_bound(Q, D):
    return 2 * torch.sqrt(Q * D) + D


def _prof(e, order):
    out = e.pruning_profile(order)
    torch.cuda.synchronize()
    return out


# ------------------------------------------------------------------------------------------------ 1. against the per-mask route
CASES = [
    ("r4p2-K27", ("channel", 2000, 300, 4, 2), None),
    ("r4p3-K47", ("cylinder", 1500, 200, 4, 3), None),
    ("r8p2-K69", ("cylinder", 1200, 150, 8, 2), None),
    ("r8p3-K189", ("cylinder", 1500, 200, 8, 3), None),
    ("r64p1-K257", ("channel", 700, 150, 64, 1), None),
    ("r32p2-K657", ("channel", 1000, 300, 32, 2), None),
    ("fourier-r2p2", ("cylinder", 900, 120, 2, 2, 4), None),
    ("m1300-r4p2", ("aneurysm", 600, 1300, 4, 2), None),
    ("n4100-r8p3-S40", ("channel", 4100, 130, 8, 3), 40),
    ("r32p2-S100", ("channel", 1000, 300, 32, 2), 100),
]


def _check_against_masks(e, order):
    got = _prof(e, order)
    S = len(order)
    assert got["snapshot_residual2"].shape == (S + 1, e.m) and got["snapshot_residual2"].dtype == torch.float64
    assert got["snapshot_norm2"].shape == (e.m,)
    _, rs_abs, absgw, _ = _peel64(e, order)
    saved = e.gates.clone()
    worst = 0.0
    try:
        for s in range(S + 1):
            e.gates.copy_(saved)
            if s:
                e.gates[order[:s]] = 0.0
            ref = e.residual_profile()["snapshot_residual2"]
            delta = 2 * U32 * rs_abs[s] + 2 * EPS_GEMM * absgw
            bound = _cs_bound(ref, (delta ** 2).sum(0)) + SUM_R * ref + SUM_P * got["snapshot_residual2"][s]
            err = (got["snapshot_residual2"][s] - ref).abs()
            worst = max(worst, float((err / bound.clamp_min(1e-300)).max()))
            assert bool((err <= bound).all()), (s, float((err / bound.clamp_min(1e-300)).max()))
        e.gates.copy_(saved)
        rp = e.residual_profile()
    finally:
        e.gates.copy_(saved)
    # sum_x U^2: the same values in two summation orders
    assert bool(((got["snapshot_norm2"] - rp["snapshot_norm2"]).abs() <= (SUM_P + SUM_R) * rp["snapshot_norm2"]).all())
    return got, worst


@pytest.mark.parametrize("label,args,S", CASES, ids=[c[0] for c in CASES])
def test_every_step_matches_residual_profile_with_the_gates_zeroed(label, args, S):
    e = _engine(*args)
    got, worst = _check_against_masks(e, _order(e, S))
    print(label, "worst error / bound", worst)


@pytest.mark.parametrize("n,r,p", [(1, 4, 2), (1, 8, 3), (129, 4, 2)])
def test_edge_point_counts(n, r, p):
    e = _random_engine(n, 70, r, p)
    _check_against_masks(e, _order(e))


# ------------------------------------------------------------------------------------------------ 2. against fp64 POOL_DATA
@pytest.mark.parametrize("args", [("channel", 1500, 200, 4, 2), ("cylinder", 1000, 150, 8, 2), ("cylinder", 900, 130, 8, 3)],
                         ids=["K27", "K69", "K189"])
def test_against_fp64_reference(args):
    e = _engine(*args)
    order = _order(e)
    got = _prof(e, order)
    Q, rs_abs, absgw, r0 = _peel64(e, order)
    # fp32 library values: (p + 4) u relative for the monomials, (p + 4) u absolute for sin / cos / tanh of |omega Phi| <~ 1
    G = _library64(e)
    libgw = (G.abs() + 1.0) @ e.W[:e.K, :e.m].double().abs()
    for s in range(len(order) + 1):
        delta = 2 * U32 * rs_abs[s] + U32 * r0.abs() + EPS_GEMM * absgw + (e.polyorder + 4) * U32 * libgw
        bound = _cs_bound(Q[s], (delta ** 2).sum(0)) + SUM_P * got["snapshot_residual2"][s]
        err = (got["snapshot_residual2"][s] - Q[s]).abs()
        assert bool((err <= bound).all()), (s, float((err / bound).max()))
    u2 = (e.U[:, :e.n].double() ** 2).sum(1)
    assert bool(((got["snapshot_norm2"] - u2).abs() <= SUM_P * u2).all())


# ------------------------------------------------------------------------------------------------ 3. against the existing sweeps
def test_curve_equals_greedy_removal():
    from desmo_b200 import DESMO
    from desmo_b200.sparsify import greedy_removal, pruning_profile

    _, modes, snap, prm = make_case("channel", 700, 72, 4, 2, omega_init=10.0, perturb_rel=0.3)
    prm.gates[3] = 0.0  # an already-pruned term: norm 0, removed first, never counted
    model = DESMO(prm.n, prm.m, 2, 4, 10.0, pod_modes=modes, device=torch.device(DEV))
    load_engine(model.engine, prm, modes, snap)
    x2 = float((snap.astype(np.float64) ** 2).sum())
    want = greedy_removal(model, x2)
    pp = pruning_profile(model, snapshot_norm2=x2)
    assert len(pp.relative_error) == prm.K + 1
    assert pp.nonzero_terms == [w[2] for w in want]
    for s, w in enumerate(want):
        assert abs(pp.relative_error[s] - w[1]) < 1e-4 * max(w[1], 1e-3), (s, pp.relative_error[s], w)
    assert abs(pp.relative_error[-1] - 1.0) < 1e-6  # every term removed: recon = 0
    # the default denominator is the stored U's sum of squares
    assert abs(pruning_profile(model).relative_error[-1] - 1.0) < 1e-6
    assert torch.equal(model.engine.gates.cpu(), torch.from_numpy(prm.gates))


@pytest.mark.parametrize("name", ["traj_chan_r4p2", "traj_fcyl_r2p2", "traj_cyl_r4p3"])
def test_thresholds_read_off_the_curve_match_the_golden_sweep(name):
    from desmo_b200 import DESMO, DESMOFourier
    from desmo_b200.sparsify import pruning_profile, threshold_sweep

    fx, meta, modes, snap, prm = golden_case(name)
    dev = torch.device(DEV)
    if prm.fourier:
        model = DESMOFourier(prm.n, prm.m, prm.polyorder, prm.r, 10.0, prm.nF, period_init=meta["period_init"], pod_modes=modes, device=dev)
    else:
        model = DESMO(prm.n, prm.m, prm.polyorder, prm.r, 10.0, pod_modes=modes, device=dev)
    q = prm.copy()
    for k in ("gates", "phi", "omega", "zall", "coefs", "periods"):
        if getattr(q, k) is not None:
            setattr(q, k, fx[f"step{meta['steps']}_{k}"].copy())
    load_engine(model.engine, q, modes, snap)
    x2 = float((snap.astype(np.float64) ** 2).sum())
    pp = pruning_profile(model, snapshot_norm2=x2)
    thr = list(fx["sweep_thresholds"])
    ref = threshold_sweep(model, x2, thr)
    for i, ((t, err, n_active, mask), (_, err_ref, _, _)) in enumerate(zip(pp.threshold_sweep(thr), ref)):
        assert np.array_equal(mask.cpu().numpy(), fx["sweep_masks"][i]), t
        assert n_active == int(fx["sweep_nonzero"][i])
        assert abs(err - fx["sweep_err"][i]) < 2e-5, (t, err, fx["sweep_err"][i])
        assert abs(err - err_ref) < 2e-5


# ------------------------------------------------------------------------------------------------ 4./5. storage, reproducibility
@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3)], ids=["r4p2", "r8p3"])
def test_bf16_equals_fp32_storage_of_uq_and_calls_repeat_bit_for_bit(args):
    from desmo_b200 import DesmoEngine

    kind, n, m, r, p = args
    _, modes, snap, prm = make_case(kind, n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    out = []
    for dt, s in ((torch.bfloat16, snap), (torch.float32, torch.from_numpy(snap).bfloat16().float().numpy())):
        e = DesmoEngine(n, m, p, r, omega_init=10.0, device=torch.device(DEV), snapshot_dtype=dt)
        load_engine(e, prm, modes, s)
        out.append(_prof(e, _order(e)))
    again = _prof(e, _order(e))
    for k in ("snapshot_residual2", "snapshot_norm2"):
        assert torch.equal(out[0][k], out[1][k]), k
        assert torch.equal(out[1][k], again[k]), k


# ------------------------------------------------------------------------------------------------ 6. no side effects
def _buffers(e):
    return {k: v.clone() for k, v in vars(e).items() if torch.is_tensor(v)}


@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3), ("cylinder", 900, 120, 2, 2, 4)],
                         ids=["fusedtc", "gemm", "fourier"])
def test_no_side_effects(args):
    e = _engine(*args)
    e.train_step()
    e.build_w(False)
    torch.cuda.synchronize()
    before = _buffers(e)
    _prof(e, _order(e))
    after = _buffers(e)
    for k in before:
        assert torch.equal(before[k], after[k]), k


@pytest.mark.parametrize("path", [0, 3])
def test_profile_between_training_steps_changes_nothing(path):
    from desmo_b200 import DesmoEngine, DesmoTrainer

    fx, meta, modes, snap, prm = golden_case("traj_chan_r4p2")
    runs = []
    for with_profile in (False, True):
        e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device(DEV), path=path)
        load_engine(e, prm, modes, snap)
        tr = DesmoTrainer(e, lrs=meta["lrs"], beta=meta["beta"], l1_lambda=meta["l1_lambda"], patience=2, sched_every=3,
                          use_cuda_graph=True, device_scheduler=True)
        losses = []
        for i in range(20):
            if with_profile and i == 10:
                e.pruning_profile(_order(e))
            tr.step()
            losses.append(e.losses.clone())
        torch.cuda.synchronize()
        runs.append((e, torch.stack(losses)))
    (e0, l0), (e1, l1) = runs
    assert torch.equal(l0, l1)
    for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "omega", "omega_m", "omega_u",
              "hyper", "step_dev", "losses", "red", "dphi", "U"):
        assert torch.equal(getattr(e0, k), getattr(e1, k)), k


# ------------------------------------------------------------------------------------------------ 7. validation, ops route, sharding
def test_validation_and_ops_route():
    import desmo_b200.ops as ops
    from desmo_b200 import _lib

    e = _engine("cylinder", 1500, 200, 8, 3)
    order = _order(e, 50)
    step = e.step_dev.clone()
    a = _prof(e, order)
    b = ops.engine_pruning_profile_via_ops(e, order)
    torch.cuda.synchronize()
    for k in ("snapshot_residual2", "snapshot_norm2"):
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(e.step_dev, step)
    empty = _prof(e, [])  # S = 0: step 0 only
    assert torch.equal(empty["snapshot_residual2"][0], a["snapshot_residual2"][0])
    for bad in ([order[0], order[0]], [e.K], [-1], list(range(e.K + 1))):
        with pytest.raises(_lib.DesmoError):
            e.pruning_profile(bad)
    sa = ops._shape_args(e)
    snap = torch.full((3, e.m), 3.0, dtype=torch.float64, device=DEV)
    norm = torch.full((e.m,), 3.0, dtype=torch.float64, device=DEV)
    for bad in ([1, 1], [1, e.K]):
        with pytest.raises(_lib.DesmoError):
            torch.ops.desmo_b200.pruning_profile(e.U, e.P, e.phi, e.omega, e.W, torch.tensor(bad, dtype=torch.int32), snap, norm, *sa)
    with pytest.raises(_lib.DesmoError):  # the order lives on the host
        torch.ops.desmo_b200.pruning_profile(e.U, e.P, e.phi, e.omega, e.W, torch.tensor([0, 1], dtype=torch.int32, device=DEV), snap,
                                             norm, *sa)
    torch.cuda.synchronize()
    assert bool((snap == 3.0).all()) and bool((norm == 3.0).all())  # nothing was launched


def test_sharded_profile_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29674", os.path.join(ROOT, "tests", "_pruning_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("PRUNING_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("PRUNING_RESULT "):])
    # the sharded and unsharded sums group the same fp32 terms differently: within twice the summation bound (+ a tiny absolute floor)
    assert res["rel_vs_unsharded"] <= 2 * SUM_P, res
    assert res["identical_across_ranks"], res
