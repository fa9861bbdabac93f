"""Backward elimination by error (DesmoEngine.backward_elimination, sparsify.backward_elimination, desmo_elimination_pass /
desmo_elimination_greedy): the removal order that raises ||U - recon||^2 least at every step, from A = G^T G and F = G^T R.

Error model (u = 2^-24).  g is the device's fp32 library value, G the fp64 POOL_DATA of the same lat = fl(phi * P): |g - G| <= d with
d = (p + 4) u |G| for a monomial and (|omega lat| + 4) 2u for sin / cos / tanh (the rounding of the argument, then of the function).
  - A: three bf16 planes per operand, six products (the dropped ones and the split remainder <= 4u |g_i g_j|); the tensor core's
    truncating adds, 48 per chain (<= 48 * 2^-23 of the chain's sum of |products|), fp32 sums of the chains in a slice, fp64 beyond:
    below 2^-15 sum_x |g_i||g_j| together.  So |A - A64| <= BA = 2^-15 |G|^T |G| + d^T |G| + |G|^T d + d^T d.
  - F: r = fl(Rec - U) with Rec from GEMM 1 (six products, chains of 96 MMAs: <= 2^-16 sum_k |g_k W_k|) differs from the fp64 R by
    dr <= 2^-16 |G||W| + d |W| + u |R|.  GEMM 4 multiplies two bf16 planes of g and of r (three products: 3 * 2^-16) in chains of 384
    MMAs (<= 384 * 2^-23 < 2^-14), fp32 within a chunk's slice, fp64 beyond.  So |F - F64| <= BF = 2^-13 |G|^T |R| + (|G| + d)^T dr
    + d^T |R|.
  - An increment sum_t W_k (A_kk W_k - 2 F_k) then errs by at most b_k = sum_t |W_k| (BA_kk |W_k| + 2 BF_k), with BF_k growing by
    BA_lk |W_l| for every term l removed before (the F update).  fp64 rounding of the sums is far below that.
A choice is correct when its fp64 increment is within b_chosen + b_best of the fp64 minimum; where the fp64 margin exceeds that, it is
fp64's choice."""
import ctypes as C
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
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _engine(kind, n, m, r, p, nF=None, dtype=torch.float32, perturb_rel=0.3):
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case(kind, n, m, r, p, nF=nF, omega_init=10.0, perturb_rel=perturb_rel)
    e = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF, device=torch.device(DEV), snapshot_dtype=dtype)
    load_engine(e, prm, modes, snap)
    return e


def _random_engine(n, m, r, p, seed=0):
    """Seeded parameters and data for shapes POD cannot give (n < r): U = recon * (1 + 0.3 noise)."""
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
    """(n, K) fp64 library of lat = fl(phi * P) in packed K order, and the bound d on |g - G| (see the module docstring)."""
    lat32 = (e.phi[:, :e.n] * e.P[:, :e.n]).t().contiguous()
    lat = lat32.double().cpu().numpy()
    om = e.omega.double().cpu().numpy()
    poly = orc.pool_data(lat, e.polyorder)
    cols, dev = [poly], [(e.polyorder + 4) * U32 * np.abs(poly)]
    for b, f in enumerate((np.sin, np.cos, np.tanh)):
        arg = np.stack([om[3 * i + b] * lat[:, i] for i in range(e.r)], axis=1)
        cols.append(f(arg))
        dev.append((np.abs(arg) + 4) * 2 * U32)
    G = torch.from_numpy(np.concatenate(cols, axis=1)).to(DEV)
    d = torch.from_numpy(np.concatenate(dev, axis=1)).to(DEV)
    return G, d


def _reference(e):
    G, d = _library64(e)
    e.build_w(False)
    W = e.W[:e.K, :e.m].double()
    R = G @ W - e.U[:, :e.n].double().t()  # (n, m)
    aG = G.abs()
    BA = 2.0 ** -15 * (aG.T @ aG) + d.T @ aG + aG.T @ d + d.T @ d
    dr = 2.0 ** -16 * (aG @ W.abs()) + d @ W.abs() + U32 * R.abs()
    BF = 2.0 ** -13 * (aG.T @ R.abs()) + (aG + d).T @ dr + d.T @ R.abs()
    return {"A": G.T @ G, "F": G.T @ R, "r2": float((R ** 2).sum()), "BA": BA, "BF": BF, "W": W, "dr": dr, "R": R}


def _pass(e):
    """A, F, r2 straight from desmo_elimination_pass."""
    f64 = dict(dtype=torch.float64, device=DEV)
    scratch = e._elimination_scratch()
    A, F, r2 = torch.empty(e.K, e.K, **f64), torch.empty(e.K, e.mld, **f64), torch.empty(1, **f64)
    e.build_w(False)
    from desmo_b200._lib import check

    check(e.lib.desmo_elimination_pass(C.byref(e.shape), e.U.data_ptr(), e._u_dtype(), e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(),
                                       e.W.data_ptr(), A.data_ptr(), F.data_ptr(), r2.data_ptr(), scratch.data_ptr(), scratch.numel(),
                                       torch.cuda.current_stream().cuda_stream), "desmo_elimination_pass")
    torch.cuda.synchronize()
    return A, F, float(r2.item())


def _elim(e, steps=None):
    out = e.backward_elimination(steps)
    torch.cuda.synchronize()
    return out


def _check_pass(e, ref):
    A, F, r2 = _pass(e)
    assert torch.equal(A, A.T)
    errA = (A - ref["A"]).abs()
    assert bool((errA <= ref["BA"]).all()), float((errA / ref["BA"]).max())
    assert bool((F[:, e.m:] == 0).all())
    errF = (F[:, :e.m] - ref["F"]).abs()
    assert bool((errF <= ref["BF"]).all()), float((errF / ref["BF"]).max())
    r2_tol = float((2 * ref["R"].abs() * ref["dr"] + ref["dr"] ** 2).sum()) + 64 * U32 * ref["r2"]
    assert abs(r2 - ref["r2"]) <= r2_tol, (r2, ref["r2"], r2_tol)
    return float((errA / ref["BA"]).max()), float((errF / ref["BF"].clamp_min(1e-300)).max())


def _check_steps(e, got, ref):
    """Every step of the device's order against fp64, given the device's own prefix.  Returns the fp64 totals along the order, their
    accumulated bounds, and how many steps were decided by a margin above the bound."""
    A, F, W, BA = ref["A"], ref["F"].clone(), ref["W"], ref["BA"]
    BF = ref["BF"].clone()
    aW = W.abs()
    order = got["order"].tolist()
    removed = torch.zeros(e.K, dtype=torch.bool, device=DEV)
    nz = (W != 0).any(1)
    total, cum, totals, bounds, decided = ref["r2"], 0.0, [ref["r2"]], [0.0], 0
    for s, k in enumerate(order):
        rem = ~removed
        zero_left = torch.nonzero(rem & ~nz).flatten()
        if zero_left.numel():  # zero rows first, in index order
            assert k == int(zero_left[0]), (s, k, zero_left[:4].tolist())
            removed[k] = True
            totals.append(total)
            bounds.append(cum)
            continue
        assert bool(rem[k]) and bool(nz[k])
        Akk = torch.diagonal(A)
        delta = (W * (Akk[:, None] * W - 2 * F)).sum(1)
        b = (aW * (torch.diagonal(BA)[:, None] * aW + 2 * BF)).sum(1) + 1e-12 * abs(ref["r2"])
        cand = torch.where(rem, delta, torch.full_like(delta, float("inf")))
        best = int(torch.argmin(cand))
        assert float(delta[k]) <= float(cand[best]) + float(b[k]) + float(b[best]), (s, k, best)
        srt = torch.sort(cand).values
        if srt.numel() > 1 and torch.isfinite(srt[1]) and float(srt[1] - srt[0]) > 2 * float(b[rem].max()):
            assert k == best, (s, k, best)
            decided += 1
        total += float(delta[k])
        cum += float(b[k])
        totals.append(total)
        bounds.append(cum)
        F -= torch.outer(A[:, k], W[k])
        BF += torch.outer(BA[:, k], aW[k])
        removed[k] = True
    return np.array(totals), np.array(bounds), decided


# ------------------------------------------------------------------------------------------------ 1-3. against fp64
CASES = [
    ("r4p2-K27", ("channel", 2000, 300, 4, 2)),
    ("r4p3-K47", ("cylinder", 1500, 200, 4, 3)),
    ("r8p2-K69", ("cylinder", 1200, 150, 8, 2)),
    ("r8p3-K189", ("cylinder", 1500, 200, 8, 3)),
    ("r32p2-K657", ("channel", 1000, 300, 32, 2)),
    ("r64p1-K257", ("channel", 700, 150, 64, 1)),
    ("fourier-r2p2", ("cylinder", 900, 120, 2, 2, 4)),
    ("m1300-r4p2", ("aneurysm", 600, 1300, 4, 2)),
]
# several chunks of points ending in a short one: F adds the chunks in fp64, the Gram keeps the first chunk's slice layout
MULTI = [
    ("3chunks-r32p2-K657", ("channel", 30000, 120, 32, 2)),  # rows_c = 13 056 at m = 120: 2 x 13 056 + 4 096 points
    ("chunks-r4p2-K27", ("channel", 150000, 300, 4, 2)),     # rows_c = 47 104: 3 x 47 104 + 8 704 points
]


def _chunks(e):
    Kr, mp = (e.K + 127) // 128 * 128, (e.m + 127) // 128 * 128
    rows_c = min(max((64 << 20) // (6 * Kr + 4 * mp) // 128 * 128, 128), e.ld)
    return [min(rows_c, e.ld - x0) for x0 in range(0, e.ld, rows_c)]


@pytest.mark.parametrize("label,args", CASES + MULTI, ids=[c[0] for c in CASES + MULTI])
def test_pass_and_every_step_against_fp64(label, args):
    e = _engine(*args)
    if label in dict(MULTI):
        pts = _chunks(e)
        assert len(pts) >= 3 and pts[-1] < pts[0], pts
    ref = _reference(e)
    wa, wf = _check_pass(e, ref)
    got = _elim(e)
    order = got["order"].tolist()
    assert sorted(order) == list(range(e.K))
    totals, bounds, decided = _check_steps(e, got, ref)
    pred = got["predicted_residual2"].cpu().numpy()
    # the predicted totals are the fp64 algebra on the device's A and F: within the accumulated bounds (+ the r2 error) of fp64's
    r2_err = abs(pred[0] - ref["r2"])
    assert np.all(np.abs(pred - totals) <= bounds + r2_err + 1e-12 * np.abs(totals).max()), float(np.max(np.abs(pred - totals) - bounds))
    # and of the exact profile of the same order (pruning_profile's own error is bounded in test_pruning_profile.py, here 2^-14 of it)
    prof = e.pruning_profile(order)["snapshot_residual2"].sum(1).cpu().numpy()
    assert np.all(np.abs(pred - prof) <= bounds + r2_err + 2.0 ** -14 * np.maximum(prof, totals) + 1e-12 * prof.max()), \
        float(np.max(np.abs(pred - prof) / (bounds + r2_err + 2.0 ** -14 * prof + 1e-300)))
    print(label, "A err/bound", wa, "F err/bound", wf, "steps decided by margin", decided, "of", e.K)


@pytest.mark.parametrize("n,r,p", [(1, 4, 2), (129, 8, 3)])
def test_edge_point_counts(n, r, p):
    e = _random_engine(n, 70, r, p)
    ref = _reference(e)
    _check_pass(e, ref)
    got = _elim(e)
    _check_steps(e, got, ref)


# ------------------------------------------------------------------------------------------------ 4. small libraries, brute force
@pytest.mark.parametrize("args", [("cylinder", 1500, 200, 2, 2), ("cylinder", 900, 120, 2, 2, 4)], ids=["r2p2", "fourier-r2"])
def test_small_library_against_brute_force(args):
    from desmo_b200 import sparsify

    e = _engine(*args)
    ref = _reference(e)
    got = _elim(e)
    order = got["order"].tolist()
    prof = e.pruning_profile(order)["snapshot_residual2"]
    saved = e.gates.clone()
    for s in (1, 2, e.K // 2, e.K):  # pruning_profile(order) against residual_profile() with the gates of order[:s] zeroed
        e.gates.copy_(saved)
        e.gates[order[:s]] = 0.0
        rp = e.residual_profile()["snapshot_residual2"]
        assert float((prof[s] - rp).abs().sum()) <= 2.0 ** -12 * float(rp.sum()) + 1e-9, s
    e.gates.copy_(saved)
    # step 1 by brute force: every candidate's exact error, one profile each
    first = np.array([float(e.pruning_profile([k])["snapshot_residual2"][1].sum()) for k in range(e.K)])
    totals, bounds, _ = _check_steps(e, got, ref)
    assert first[order[0]] <= first.min() + 2 * bounds[1] + 2.0 ** -14 * first.min()
    # the error order's first step is no worse than the norm order's, within the ranking bound
    norm_first = sparsify.pruning_profile(_Model(e)).relative_error[1]
    elim = sparsify.backward_elimination(_Model(e))
    assert elim.order == order
    total = float(prof[0].sum()) / elim.relative_error[0] ** 2  # ||U||^2 as the profile normalises
    assert elim.relative_error[1] ** 2 <= norm_first ** 2 + (2 * bounds[1] + 2.0 ** -14 * first.min()) / total, (elim.relative_error[1], norm_first)


class _Model:
    def __init__(self, e):
        self.engine = e


# ------------------------------------------------------------------------------------------------ 5. a planted case
def test_planted_small_norm_term_is_kept():
    """r = 2, p = 1 (K = 9), a perfect fit.  The reference's term norms evaluate the library on the raw phi, forward() on phi * POD:
    with mode 0's POD mode 100x larger, phi_0 (term 1) with a 20x smaller row has the smallest norm but the largest single field, so
    the norm order removes it first and the error order keeps it until only the cancelling pair is left.  The pair: phi_1 and
    sin(omega phi_1) at omega = 0.01, weighted 4 z and -400 z, each a large field, their sum a small cubic remainder -- removing either
    alone costs most of the signal, so the greedy takes neither before the others."""
    from desmo_b200 import DesmoEngine, sparsify

    n, m, r, p = 3000, 120, 2, 1
    g = torch.Generator(device=DEV).manual_seed(7)
    e = DesmoEngine(n, m, p, r, omega_init=3.0, device=torch.device(DEV))
    e.P[0, :n] = 100.0 * (1.0 + 0.1 * torch.randn(n, device=DEV, generator=g))
    e.P[1, :n] = 1.0 + 0.1 * torch.randn(n, device=DEV, generator=g)
    e.phi[:, :n] = 1.0 + 0.3 * torch.randn(r, n, device=DEV, generator=g)
    e.rows[:, :m] = 0.3 * torch.randn(e.K, m, device=DEV, generator=g)
    c, lin1, sin1 = 1, 2, e.T + 1  # phi_0; phi_1 and sin(omega_1 phi_1) (packed order: sin_i at T + i)
    e.rows[c, :m] = 0.015 * torch.randn(m, device=DEV, generator=g)
    e.omega[3] = 0.01
    z = torch.randn(m, device=DEV, generator=g)
    e.rows[lin1, :m] = 4.0 * z
    e.rows[sin1, :m] = -4.0 * z / 0.01
    e.set_snapshot(torch.zeros(m, n))
    e.set_snapshot(e.reconstruct())
    model = _Model(e)
    norm = sparsify.pruning_profile(model)
    elim = sparsify.backward_elimination(model)
    assert norm.order[0] == c, norm.order
    assert elim.order.index(c) >= e.K - 3, elim.order
    assert set(elim.order[-2:]) == {lin1, sin1}, elim.order
    assert elim.relative_error[1] < 0.5 * norm.relative_error[1], (elim.relative_error[:3], norm.relative_error[:3])
    assert all(a <= b * (1 + 2.0 ** -10) for a, b in zip(elim.relative_error[1:3], norm.relative_error[1:3]))


# ------------------------------------------------------------------------------------------------ 6. zero gates, active sets, edges
def test_zero_gates_and_active_set_come_first():
    from desmo_b200 import sparsify

    e = _engine("cylinder", 1500, 200, 8, 3)
    mask = torch.rand(e.K, generator=torch.Generator().manual_seed(5)) < 0.6
    mask[0] = True
    e.gates[[3, 11]] = 0.0
    e.set_active_terms(mask)
    gates, rows, step = e.gates.clone(), e.rows.clone(), e.step_dev.clone()
    absent = sorted(set(np.flatnonzero(~mask.numpy()).tolist()) | {3, 11})
    got = _elim(e)
    order = got["order"].tolist()
    assert order[:len(absent)] == absent
    pred = got["predicted_residual2"].cpu().numpy()
    assert np.all(pred[:len(absent) + 1] == pred[0])
    prof = sparsify.backward_elimination(_Model(e))
    assert prof.order == order
    nz = int((gates != 0).sum())
    assert prof.nonzero_terms[:len(absent) + 1] == [nz] * (len(absent) + 1)
    assert prof.nonzero_terms[-1] == 0 and all(a - b in (0, 1) for a, b in zip(prof.nonzero_terms, prof.nonzero_terms[1:]))
    assert abs(prof.relative_error[-1] - 1.0) <= 1e-4
    assert torch.equal(e.gates, gates) and torch.equal(e.rows, rows) and torch.equal(e.step_dev, step)
    assert torch.equal(e.active_terms, mask)
    am = prof.active_mask(len(absent) + 3)
    assert not bool(am[order[:len(absent) + 3]].any())


def test_fewer_steps_and_a_perfect_fit():
    e = _engine("cylinder", 1500, 200, 8, 3)  # K = 189: reconstruct() is GEMM 1's Rec, bit for bit
    full = _elim(e)
    part = _elim(e, 25)
    assert torch.equal(part["order"], full["order"][:25])
    assert torch.equal(part["predicted_residual2"], full["predicted_residual2"][:26])
    assert _elim(e, 0)["order"].numel() == 0
    e.set_snapshot(e.reconstruct())
    got = _elim(e)
    pred = got["predicted_residual2"].cpu().numpy()
    assert pred[0] == 0.0 and np.all(np.isfinite(pred)) and sorted(got["order"].tolist()) == list(range(e.K))


# ------------------------------------------------------------------------------------------------ 7. invariants
def _same(a, b):
    for k in ("order", "predicted_residual2", "gram"):
        assert torch.equal(a[k], b[k]), k


def test_bit_reproducible_and_bf16_equals_fp32_of_uq():
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case("cylinder", 1500, 200, 8, 3, omega_init=10.0, perturb_rel=0.3)
    out = []
    for dt, s in ((torch.bfloat16, snap), (torch.float32, torch.from_numpy(snap).bfloat16().float().numpy())):
        e = DesmoEngine(1500, 200, 3, 8, omega_init=10.0, device=torch.device(DEV), snapshot_dtype=dt)
        load_engine(e, prm, modes, s)
        out.append(_elim(e))
        _same(out[-1], _elim(e))
    _same(*out)


@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3), ("cylinder", 900, 120, 2, 2, 4)],
                         ids=["fusedtc", "gemm", "fourier"])
def test_no_side_effects(args):
    e = _engine(*args)
    e.train_step()
    e.build_w(False)
    torch.cuda.synchronize()
    before = {k: v.clone() for k, v in vars(e).items() if torch.is_tensor(v)}
    _elim(e)
    for k, v in vars(e).items():
        if torch.is_tensor(v):
            assert torch.equal(before[k], v), k


@pytest.mark.parametrize("path", [0, 3])
def test_elimination_between_training_steps_changes_nothing(path):
    from desmo_b200 import DesmoEngine, DesmoTrainer

    fx, meta, modes, snap, prm = golden_case("traj_chan_r4p2")
    runs = []
    for with_call in (False, True):
        e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device(DEV), path=path)
        load_engine(e, prm, modes, snap)
        tr = DesmoTrainer(e, lrs=meta["lrs"], beta=meta["beta"], l1_lambda=meta["l1_lambda"], patience=2, sched_every=3,
                          use_cuda_graph=True, device_scheduler=True)
        losses = []
        for i in range(20):
            if with_call and i == 10:
                e.backward_elimination()
            tr.step()
            losses.append(e.losses.clone())
        torch.cuda.synchronize()
        runs.append((e, torch.stack(losses)))
    (e0, l0), (e1, l1) = runs
    assert torch.equal(l0, l1)
    for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "omega", "omega_m", "omega_u",
              "hyper", "step_dev", "losses", "red", "dphi", "P"):
        assert torch.equal(getattr(e0, k), getattr(e1, k)), k


# ------------------------------------------------------------------------------------------------ 8. routes and bad input
def test_ops_route_and_model_pass_through():
    import desmo_b200.ops as ops
    from desmo_b200 import DESMO

    e = _engine("channel", 1000, 300, 32, 2)
    step = e.step_dev.clone()
    a = _elim(e)
    b = ops.engine_backward_elimination_via_ops(e)
    torch.cuda.synchronize()
    _same(a, b)
    assert torch.equal(e.step_dev, step)
    _, modes, snap, prm = make_case("channel", 1000, 300, 32, 2, omega_init=10.0, perturb_rel=0.3)
    model = DESMO(1000, 300, 2, 32, 10.0, pod_modes=modes, device=torch.device(DEV))
    load_engine(model.engine, prm, modes, snap)
    _same(model.backward_elimination(), a)


def test_bad_arguments_raise_before_any_launch():
    from desmo_b200 import DesmoEngine, _lib

    e = DesmoEngine(1000, 50, 2, 4, device=torch.device(DEV))
    with pytest.raises(_lib.DesmoError):
        e.backward_elimination()  # no snapshot
    e.set_snapshot(torch.randn(50, 1000))
    for s in (-1, e.K + 1):
        with pytest.raises(_lib.DesmoError):
            e.backward_elimination(s)
    scratch = e._elimination_scratch()
    f64 = dict(dtype=torch.float64, device=DEV)
    A, F, r2 = torch.full((e.K, e.K), 7.0, **f64), torch.full((e.K, e.mld), 7.0, **f64), torch.full((1,), 7.0, **f64)
    order, pred = torch.full((e.K,), 7, dtype=torch.int32, device=DEV), torch.full((e.K + 1,), 7.0, **f64)
    st = torch.cuda.current_stream().cuda_stream
    args = (C.byref(e.shape), e.U.data_ptr(), e._u_dtype(), e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(), e.W.data_ptr())
    outs = (A.data_ptr(), F.data_ptr(), r2.data_ptr())
    assert e.lib.desmo_elimination_pass(*args, *outs, scratch.data_ptr(), scratch.numel() - 1, st) == 1
    assert b"scratch too small" in e.lib.desmo_last_error()
    assert e.lib.desmo_elimination_pass(*args, *outs, scratch.data_ptr() + 8, scratch.numel() - 8, st) == 1
    assert b"aligned" in e.lib.desmo_last_error()
    assert e.lib.desmo_elimination_pass(*args[:2], 7, *args[3:], *outs, scratch.data_ptr(), scratch.numel(), st) == 1
    assert e.lib.desmo_elimination_pass(*args, A.data_ptr(), None, r2.data_ptr(), scratch.data_ptr(), scratch.numel(), st) == 1
    g = (C.byref(e.shape), A.data_ptr(), F.data_ptr(), r2.data_ptr(), e.W.data_ptr())
    assert e.lib.desmo_elimination_greedy(*g, e.K + 1, order.data_ptr(), pred.data_ptr(), scratch.data_ptr(), scratch.numel(), st) == 1
    assert e.lib.desmo_elimination_greedy(*g, -1, order.data_ptr(), pred.data_ptr(), scratch.data_ptr(), scratch.numel(), st) == 1
    assert e.lib.desmo_elimination_greedy(*g, 3, None, pred.data_ptr(), scratch.data_ptr(), scratch.numel(), st) == 1
    assert e.lib.desmo_elimination_greedy(*g, 3, order.data_ptr(), pred.data_ptr(), scratch.data_ptr(), 16, st) == 1
    torch.cuda.synchronize()
    assert bool((A == 7.0).all()) and bool((F == 7.0).all()) and bool((r2 == 7.0).all())  # nothing was launched
    assert bool((order == 7).all()) and bool((pred == 7.0).all())


# ------------------------------------------------------------------------------------------------ 9. point-sharded
def test_sharded_order_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29681", os.path.join(ROOT, "tests", "_elimination_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("ELIM_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("ELIM_RESULT "):])
    assert res["identical_across_ranks"], res
    assert res["gram_rel_vs_unsharded"] <= 1e-6, res
    assert res["same_prefix_as_unsharded"] >= 1, res
    assert res["pred_rel_vs_unsharded"] <= 1e-4, res
