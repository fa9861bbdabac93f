"""Evaluation at chosen instants (DesmoEngine.temporal_rows_at / reconstruct_at / residual_profile_at, desmo_build_w_at).

Error model (u = 2^-24).  On the training grid every value is bit for bit what desmo_build_w / desmo_reconstruct give.  Off the grid a
Fourier term is z(t) = a0 + sum_h a_h cos(theta_h) + b_h sin(theta_h), theta_h = 2 pi h t / period, and the device evaluates
theta~ = fl(fl(fl32(2 pi h) * t) / period): three roundings, |theta~ - theta| <= 3u |theta| (+ O(u^2)).  cos / sin move by at most
that much, and are themselves accurate to 2 ulp (<= 2^-23 absolute, |value| <= 1).  The fp32 products and the running sum add at most
(2 nF + 2) u of the sum of the term magnitudes.  So, per term k,
  |z~(t) - z(t)| <= sum_h (|a_h| + |b_h|) (3u |theta_h| + 2^-23) + (2 nF + 2) u (|a0| + sum_h (|a_h| + |b_h|))
with z(t) the fp64 value of the reference's fourier_series (FCYL:487-506) at the fp32 time t."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import load_engine, make_case

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U32 = 2.0 ** -24
SNAP_BOUND, POINT_BOUND = 9 * U32, 70 * U32  # desmo_residual_profile's documented bounds
ETA_FFMA = 2.0 ** -14  # |recon_ffma - recon_gemm| <= eta |recon| (tests/test_residual_profile.py)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("snapshot_residual2", "snapshot_norm2", "point_residual2", "point_norm2")


def _engine(kind, n, m, r, p, nF=None, dtype=torch.float32, period_init=60.0):
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case(kind, n, m, r, p, nF=nF, omega_init=10.0, perturb_rel=0.3, period_init=period_init)
    e = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF, device=torch.device(DEV), snapshot_dtype=dtype, period_init=period_init)
    load_engine(e, prm, modes, snap)
    return e


def _is_gemm_recon(e):
    return not (e.r <= 8 and e.K <= 80)  # desmo_reconstruct's FFMA kernel covers r <= 8, K <= 80


def _indices(m, count, seed):
    """Unsorted, with repeats, always including 0 and m - 1."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, m, size=count)
    k[0] = m - 1
    if count > 2:
        k[count // 2] = 0
        k[-1] = k[1]
    return k


# ------------------------------------------------------------------------------------------------ 1. grid identity
GRID = [
    ("desmo-r4p2-K27", ("channel", 1000, 300, 4, 2)),
    ("desmo-r8p2-K69", ("cylinder", 777, 150, 8, 2)),
    ("desmo-r8p3-K189", ("cylinder", 1500, 200, 8, 3)),
    ("desmo-r32p2-K657", ("channel", 1000, 300, 32, 2)),
    ("fourier-r2p2", ("cylinder", 900, 120, 2, 2, 4)),
    ("fourier-r8p3-K189", ("cylinder", 700, 90, 8, 3, 3)),
    ("desmo-m1300-r4p2", ("aneurysm", 600, 1300, 4, 2)),
    ("fourier-m1300-r4p2", ("aneurysm", 600, 1300, 4, 2, 3)),
]


@pytest.mark.parametrize("label,args", GRID, ids=[g[0] for g in GRID])
def test_grid_instants_are_bit_identical_to_the_training_evaluation(label, args):
    e = _engine(*args)
    e.build_w(False)
    W_full, rows_full = e.W.clone(), e.rows.clone()
    rec_full = e.reconstruct()
    for count in (1, 7, 130, 1300):
        k = _indices(e.m, count, seed=count)
        kt = torch.from_numpy(k).long().to(DEV)
        W = e._w_at(*_host(e, k), round_up16(count))
        torch.cuda.synchronize()
        assert torch.equal(W[:, :count], W_full[:, kt]), (label, count)
        assert int((W[:, count:] != 0).sum()) == 0 and int((W[e.K:] != 0).sum()) == 0
        z = e.temporal_rows_at(index=k)
        assert z.shape == (e.K, count)
        assert torch.equal(z, rows_full[:e.K, kt]), (label, count)
        if e.nF:
            assert torch.equal(e.temporal_rows_at(times=e.time_points(k)), z)
            assert torch.equal(e.reconstruct_at(times=e.time_points(k)), rec_full[kt])
        rec = e.reconstruct_at(index=k)
        assert rec.shape == (count, e.n)
        assert torch.equal(rec, rec_full[kt]), (label, count, _is_gemm_recon(e))
    # no buffer of the model moved
    assert torch.equal(e.W, W_full) and torch.equal(e.rows, rows_full)


def round_up16(v):
    return (v + 15) // 16 * 16


def _host(e, k):
    from desmo_b200.engine import _instants

    return _instants(k, None, e.m, e.nF)


@pytest.mark.parametrize("n", [1, 129])
def test_grid_identity_at_edge_point_counts(n):
    from desmo_b200 import DesmoEngine

    g = torch.Generator(device=DEV).manual_seed(n)
    for r, p in ((4, 2), (8, 3)):
        e = DesmoEngine(n, 70, p, r, omega_init=3.0, device=torch.device(DEV))
        e.P[:, :n] = torch.randn(r, n, device=DEV, generator=g) * 0.5
        e.phi[:, :n] = 1.0 + 0.2 * torch.randn(r, n, device=DEV, generator=g)
        e.gates.copy_(1.0 + 0.2 * torch.randn(e.K, device=DEV, generator=g))
        e.rows[:, :70] = torch.randn(e.K, 70, device=DEV, generator=g)
        full = e.reconstruct()
        for count in (1, 7, 130):
            k = _indices(70, count, seed=count)
            assert torch.equal(e.reconstruct_at(index=k), full[torch.from_numpy(k).long().to(DEV)]), (n, r, p, count)


# ------------------------------------------------------------------------------------------------ 2./3. off the grid, periodicity
def _fp64_series(coefs, periods, t):
    """fp64 fourier_series (FCYL:487-506) of every term at the fp32 times t (given as float64 values): (K, len(t)), and the bound."""
    c = coefs.double().cpu().numpy()
    per = periods.double().cpu().numpy()[:, None]
    tt = np.asarray(t, dtype=np.float64)[None, :]
    nF = (c.shape[1] - 1) // 2
    z = np.repeat(c[:, 0:1], tt.shape[1], axis=1)
    mag = np.abs(c).sum(axis=1, keepdims=True)
    bound = (2 * nF + 2) * U32 * np.repeat(mag, tt.shape[1], axis=1)
    for h in range(1, nF + 1):
        th = 2.0 * np.pi * h * tt / per
        a, b = c[:, 2 * h - 1:2 * h], c[:, 2 * h:2 * h + 1]
        z = z + a * np.cos(th) + b * np.sin(th)
        bound = bound + (np.abs(a) + np.abs(b)) * (3 * U32 * np.abs(th) + 2.0 ** -23)
    return z, bound


def test_off_grid_fourier_values_against_fp64():
    e = _engine("cylinder", 900, 120, 2, 2, nF=4)
    m = e.m
    grid = e.time_points(range(m))
    rng = np.random.default_rng(3)
    t = np.concatenate([
        rng.uniform(0, m, 200),                              # inside the window
        0.5 * (grid[:-1] + grid[1:])[::7],                   # half-way between grid points
        rng.uniform(m, 3 * m, 200), [3.0 * m],               # beyond the window, up to 3m
        -rng.uniform(0, 2 * m, 100), [-0.0, 1e-30],          # before 0
    ]).astype(np.float32)
    z = e.temporal_rows_at(times=t).double().cpu().numpy()
    ref, bound = _fp64_series(e.coefs, e.periods, t.astype(np.float64))
    err = np.abs(z - ref)
    assert (err <= bound).all(), float((err / bound).max())
    # W' = gate * z: one more rounding
    import desmo_b200.ops  # noqa: F401  (registers the op)

    W = torch.zeros(e.Kp, round_up16(t.size), device=DEV)
    torch.ops.desmo_b200.build_w_at(e.gates, e.rows, e.coefs, e.periods, None, torch.from_numpy(t), W, None,
                                    e.n, e.n_global, e.m, e.r, e.polyorder, e.nF, e.shape.path)
    g = e.gates.double().cpu().numpy()[:, None]
    Wd = W[:e.K, :t.size].double().cpu().numpy()
    assert (np.abs(Wd - g * ref) <= np.abs(g) * (bound + U32 * (np.abs(ref) + bound)) + 1e-300).all()


def test_periodicity():
    e = _engine("cylinder", 700, 90, 8, 3, nF=3)
    T0 = 37.25
    e.periods.fill_(T0)
    rng = np.random.default_rng(5)
    t = np.concatenate([rng.uniform(-90, 180, 300), e.time_points(range(90))]).astype(np.float32)
    t2 = (t + np.float32(T0)).astype(np.float32)  # one fp32 rounding on the host
    za = e.temporal_rows_at(times=t).double().cpu().numpy()
    zb = e.temporal_rows_at(times=t2).double().cpu().numpy()
    _, ba = _fp64_series(e.coefs, e.periods, t.astype(np.float64))
    _, bb = _fp64_series(e.coefs, e.periods, t2.astype(np.float64))
    c = e.coefs.double().cpu().numpy()
    nF = (c.shape[1] - 1) // 2
    shift = np.abs(t2.astype(np.float64) - t.astype(np.float64) - T0)[None, :]  # how far t2 is from t + T0 exactly
    moved = sum((np.abs(c[:, 2 * h - 1:2 * h]) + np.abs(c[:, 2 * h:2 * h + 1])) * 2 * np.pi * h / T0 for h in range(1, nF + 1)) * shift
    err = np.abs(za - zb)
    assert (err <= ba + bb + moved).all(), float((err / (ba + bb + moved)).max())
    assert float(np.abs(za).max()) > 0.1


# ------------------------------------------------------------------------------------------------ 4. held-out profile
def _reference(rec, Ub):
    rec, u = rec.double(), Ub.double()
    r2, u2, c2 = (rec - u) ** 2, u ** 2, rec ** 2
    return {"snapshot_residual2": r2.sum(1), "snapshot_norm2": u2.sum(1), "point_residual2": r2.sum(0), "point_norm2": u2.sum(0),
            "snapshot_recon2": c2.sum(1), "point_recon2": c2.sum(0)}


def _check_profile(e, got, ref):
    for k in KEYS:
        assert got[k].shape == ref[k].shape, k
        assert torch.isfinite(got[k]).all(), k
    for k, b in (("snapshot_norm2", SNAP_BOUND), ("point_norm2", POINT_BOUND)):
        err = (got[k].double() - ref[k]).abs()
        assert bool((err <= b * ref[k] + 1e-300).all()), k
    for k, b, c2 in (("snapshot_residual2", SNAP_BOUND, "snapshot_recon2"), ("point_residual2", POINT_BOUND, "point_recon2")):
        g, r = got[k].double(), ref[k]
        bound = b * r
        if not _is_gemm_recon(e):
            bound = bound + 2 * ETA_FFMA * torch.sqrt(r * ref[c2]) + ETA_FFMA ** 2 * ref[c2]
        assert bool(((g - r).abs() <= bound + 1e-300).all()), (k, float(((g - r).abs() / bound.clamp_min(1e-300)).max()))


HELD = [
    ("r4p2-K27", ("channel", 2000, 300, 4, 2), 200),
    ("r8p2-K69", ("cylinder", 1200, 150, 8, 2), 77),
    ("r8p3-K189", ("cylinder", 1500, 200, 8, 3), 130),
    ("r32p2-K657", ("channel", 1000, 300, 32, 2), 200),
    ("fourier-r2p2", ("cylinder", 900, 120, 2, 2, 4), 1),
    ("fourier-r8p3", ("cylinder", 700, 90, 8, 3, 3), 250),
]


@pytest.mark.parametrize("label,args,count", HELD, ids=[h[0] for h in HELD])
def test_held_out_profile_against_fp64_sums(label, args, count):
    e = _engine(*args)
    m = e.m
    # a held-out block: other data of the same kind (a later stretch of the synthetic flow), at unsorted training indices
    X, _, _, _ = make_case(args[0], args[1], 2 * m, *args[3:5], omega_init=10.0)
    k = _indices(m, count, seed=11)
    block = torch.from_numpy(np.ascontiguousarray(X.T[m + k].astype(np.float32)))
    kw = {"times": e.time_points(m + k)} if e.nF else {"index": k}
    got = e.residual_profile_at(block, **kw)
    rec = e.reconstruct_at(**kw)
    torch.cuda.synchronize()
    _check_profile(e, got, _reference(rec, block.to(DEV)))
    # fp64 and device input store the same fp32 values
    got64 = e.residual_profile_at(block.double().to(DEV), **kw)
    for key in KEYS:
        assert torch.equal(got[key], got64[key]), key


@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3), ("cylinder", 700, 90, 8, 3, 3)],
                         ids=["r4p2", "r8p3", "fourier"])
def test_held_out_bf16_storage_equals_fp32_storage_of_uq(args):
    eb = _engine(*args, dtype=torch.bfloat16)
    ef = _engine(*args, dtype=torch.float32)
    m = eb.m
    X, _, _, _ = make_case(args[0], args[1], 2 * m, *args[3:5], omega_init=10.0)
    k = _indices(m, 150, seed=2)
    block = torch.from_numpy(np.ascontiguousarray(X.T[m + k].astype(np.float32)))
    kw = {"times": eb.time_points(m + k)} if eb.nF else {"index": k}
    a = eb.residual_profile_at(block, **kw)                       # rounded to bf16 by desmo_snapshot_to_bf16
    b = ef.residual_profile_at(block.bfloat16().float(), **kw)    # fp32 storage of U'_q
    c = eb.residual_profile_at(block.bfloat16(), **kw)            # stored as it is
    for key in KEYS:
        assert torch.equal(a[key], b[key]) and torch.equal(a[key], c[key]), key


@pytest.mark.parametrize("args", [("cylinder", 900, 120, 2, 2, 4), ("cylinder", 700, 90, 8, 3, 3)], ids=["ffma", "gemm"])
def test_model_generated_future_block_has_a_rounding_level_residual(args):
    e = _engine(*args)
    t = e.time_points(range(e.m, 3 * e.m))
    block = e.reconstruct_at(times=t)
    got = e.residual_profile_at(block, times=t)
    torch.cuda.synchronize()
    if _is_gemm_recon(e):  # the profile's GEMM 1 is the reconstruction's: r is exactly zero
        assert float(got["snapshot_residual2"].abs().max()) == 0.0
    else:
        assert bool((got["snapshot_residual2"] <= (1 + SNAP_BOUND) * ETA_FFMA ** 2 * got["snapshot_norm2"]).all())
    assert float(got["snapshot_norm2"].min()) > 0.0


# ------------------------------------------------------------------------------------------------ 5. no side effects
def _buffers(e):
    return {k: v.clone() for k, v in vars(e).items() if torch.is_tensor(v)}


@pytest.mark.parametrize("name", ["traj_chan_r4p2", "traj_fcyl_r2p2", "traj_cyl_r4p3"])
def test_graph_replayed_training_is_unchanged_by_evaluation(name):
    from desmo_b200 import DesmoEngine, DesmoTrainer
    from tests.helpers import golden_case

    fx, meta, modes, snap, prm = golden_case(name)
    runs = []
    for with_eval in (False, True):
        e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device(DEV))
        load_engine(e, prm, modes, snap)
        tr = DesmoTrainer(e, lrs=meta["lrs"], beta=meta["beta"], l1_lambda=meta["l1_lambda"], patience=2, sched_every=3,
                          use_cuda_graph=True, device_scheduler=True)
        losses = []
        for i in range(20):
            if with_eval and i in (5, 10, 15):
                k = _indices(e.m, 37, seed=i)
                block = torch.from_numpy(snap[k])
                before = _buffers(e)
                kw = {"times": e.time_points(k + e.m)} if e.nF else {"index": k}
                e.reconstruct_at(**kw)
                e.temporal_rows_at(**kw)
                e.residual_profile_at(block, **kw)
                torch.cuda.synchronize()
                after = _buffers(e)
                for key in before:
                    assert torch.equal(before[key], after[key]), key
            tr.step()
            losses.append(e.losses.clone())
        torch.cuda.synchronize()
        runs.append((e, torch.stack(losses)))
    (e0, l0), (e1, l1) = runs
    assert torch.equal(l0, l1)
    for key in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "coefs", "coefs_m", "coefs_u",
                "periods", "periods_m", "periods_u", "omega", "omega_m", "omega_u", "hyper", "step_dev", "losses", "red", "dphi", "W"):
        a, b = getattr(e0, key), getattr(e1, key)
        assert (a is None and b is None) or torch.equal(a, b), key


# ------------------------------------------------------------------------------------------------ 6. input checks
def test_bad_inputs_raise_before_a_launch():
    import ctypes as C

    from desmo_b200 import _lib

    d = _engine("channel", 1000, 300, 4, 2)
    f = _engine("cylinder", 900, 120, 2, 2, nF=4)
    before = {id(e): _buffers(e) for e in (d, f)}
    block = torch.zeros(3, d.n)
    cases = [
        lambda: d.reconstruct_at(times=[1.0, 2.0]),                           # times on a free-row model
        lambda: d.reconstruct_at(index=[0, 300]),                             # index out of range
        lambda: d.temporal_rows_at(index=[-1]),
        lambda: f.reconstruct_at(times=[1.0, float("nan")]),                  # non-finite times
        lambda: f.temporal_rows_at(times=[float("inf")]),
        lambda: d.residual_profile_at(block, index=[0, 1]),                   # wrong block shape
        lambda: d.residual_profile_at(block.T.contiguous(), index=[0, 1, 2]),
        lambda: d.residual_profile_at(block.half(), index=[0, 1, 2]),         # fp16 block
        lambda: d.residual_profile_at(block.half().to(DEV), index=[0, 1, 2]),
        lambda: d.reconstruct_at(index=[0], times=[0.0]),                     # both
        lambda: d.reconstruct_at(),                                           # neither
    ]
    for i, fn in enumerate(cases):
        with pytest.raises(_lib.DesmoError):
            fn()
    torch.cuda.synchronize()
    for e in (d, f):
        after = _buffers(e)
        for key, v in before[id(e)].items():
            assert torch.equal(v, after[key]), key
    # the C ABI checks by itself, before it launches: a sentinel W_out stays untouched
    W = torch.full((d.Kp, 16), 7.0, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    idx = np.array([0, 300], np.int32)
    t = np.array([1.0, np.nan], np.float32)
    lib = d.lib
    assert lib.desmo_build_w_at(C.byref(d.shape), d.gates.data_ptr(), d.rows.data_ptr(), None, None, 2, 16, idx.ctypes.data, None,
                                W.data_ptr(), None, st) == 1
    assert b"index[1]" in lib.desmo_last_error()
    assert lib.desmo_build_w_at(C.byref(d.shape), d.gates.data_ptr(), d.rows.data_ptr(), None, None, 2, 16, None, t.ctypes.data,
                                W.data_ptr(), None, st) == 1
    assert lib.desmo_build_w_at(C.byref(f.shape), f.gates.data_ptr(), None, f.coefs.data_ptr(), f.periods.data_ptr(), 2, 16, None,
                                t.ctypes.data, W.data_ptr(), None, st) == 1
    assert b"not finite" in lib.desmo_last_error()
    torch.cuda.synchronize()
    assert bool((W == 7.0).all())


# ------------------------------------------------------------------------------------------------ 7. ops route
@pytest.mark.parametrize("args", [("cylinder", 1500, 200, 8, 3), ("cylinder", 700, 90, 8, 3, 3)], ids=["desmo", "fourier"])
def test_ops_route_equals_the_engine(args):
    import desmo_b200.ops  # noqa: F401  (registers the op)

    e = _engine(*args)
    k = _indices(e.m, 600, seed=4)
    idx, t = _host(e, k)
    W_e = e._w_at(idx, t, round_up16(k.size))
    z_e = e.temporal_rows_at(index=k)
    W_o = torch.zeros_like(W_e)
    z_o = torch.zeros(e.K, W_e.shape[1], device=DEV)
    torch.ops.desmo_b200.build_w_at(e.gates, e.rows, e.coefs, e.periods, torch.from_numpy(idx), None, W_o, z_o,
                                    e.n, e.n_global, e.m, e.r, e.polyorder, e.nF, e.shape.path)
    torch.cuda.synchronize()
    assert torch.equal(W_o, W_e) and torch.equal(z_o[:, :k.size], z_e)
    if e.nF:
        tt = torch.from_numpy(e.time_points(k))
        W_t = torch.zeros_like(W_e)
        torch.ops.desmo_b200.build_w_at(e.gates, e.rows, e.coefs, e.periods, None, tt, W_t, None,
                                        e.n, e.n_global, e.m, e.r, e.polyorder, e.nF, e.shape.path)
        assert torch.equal(W_t, W_e)
    from desmo_b200 import _lib

    with pytest.raises(_lib.DesmoError):  # device indices are refused: the instants are host arrays
        torch.ops.desmo_b200.build_w_at(e.gates, e.rows, e.coefs, e.periods, torch.from_numpy(idx).to(DEV), None, W_o, None,
                                        e.n, e.n_global, e.m, e.r, e.polyorder, e.nF, e.shape.path)


def test_model_pass_throughs():
    from desmo_b200 import DESMOFourier

    _, modes, snap, prm = make_case("cylinder", 700, 90, 8, 3, nF=3, omega_init=10.0, perturb_rel=0.3)
    model = DESMOFourier(prm.n, prm.m, prm.polyorder, prm.r, 10.0, nF=3, pod_modes=modes, device=torch.device(DEV))
    load_engine(model.engine, prm, modes, snap)
    with torch.no_grad():
        model.zsin_list[0].data = model.zsin_list[0].data.clone() * 2.0  # detached, as the reference's sweep does
    t = model.time_points(range(90, 120))
    z = model.temporal_rows_at(times=t)
    assert torch.equal(z, model.engine.temporal_rows_at(times=t))
    assert model.zsin_list[0].data_ptr() == model.engine.coefs[model.engine.T].data_ptr()  # re-aliased by sync_parameters
    rec = model.reconstruct_at(times=t)
    prof = model.residual_profile_at(rec, times=t)
    assert rec.shape == (30, prm.n) and prof["snapshot_residual2"].shape == (30,)


# ------------------------------------------------------------------------------------------------ 8. point-sharded
def test_sharded_held_out_profile_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29674", os.path.join(ROOT, "tests", "_eval_at_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("EVAL_AT_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("EVAL_AT_RESULT "):])
    assert res["snapshot_rel_vs_unsharded"] <= 2 * SNAP_BOUND, res
    assert res["snapshot_identical_across_ranks"], res
    assert res["point_slabs_bit_identical"], res
    assert res["recon_slabs_bit_identical"], res
