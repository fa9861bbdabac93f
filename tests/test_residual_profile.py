"""Residual profile (DesmoEngine.residual_profile, desmo_residual_profile): the per-snapshot and per-point marginals of r^2, r = recon - U,
in one pass over U without materialising recon.

Error model (u = 2^-24).  For libraries with K > 80 or r > 8, desmo_reconstruct runs the same GEMM 1 as the profile, so each fp32 r is
bit for bit reconstruct() - U and only the summation differs from fp64 sums of reconstruct().double() - U.double():
  - r itself is one fp32 rounding of that difference (<= u |r|), r^2 one more (__fmul_rn): 3u relative per term;
  - per snapshot: a 5-level tree over 32 points in fp32 (5u), everything after in fp64  -> |err| <= 8u * value (9u stated);
  - per point: 64 fp32 terms in sequence (63u), the two column halves (u), fp64 over the tiles, one fp32 rounding (u) -> 68u (70u stated).
For the libraries the FFMA reconstruction covers (r <= 8, K <= 80) the two recons differ by the fp32 rounding of two different
evaluations of G W; with |recon_profile - recon_ffma| <= eta |recon| entrywise, Cauchy-Schwarz gives
  |sum r_a^2 - sum r_b^2| <= 2 eta sqrt(sum r^2 sum recon^2) + eta^2 sum recon^2, with eta = 2^-14 (fp32-class) stated here."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import GOLDEN, golden_case, load_engine, make_case

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U32 = 2.0 ** -24
SNAP_BOUND, POINT_BOUND = 9 * U32, 70 * U32
ETA_FFMA = 2.0 ** -14
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("snapshot_residual2", "snapshot_norm2", "point_residual2", "point_norm2")


def _engine(kind, n, m, r, p, nF=None, path=0, dtype=torch.float32, perturb_rel=0.3):
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case(kind, n, m, r, p, nF=nF, omega_init=10.0, perturb_rel=perturb_rel)
    e = DesmoEngine(n, m, p, r, omega_init=10.0, nF=nF, device=torch.device(DEV), path=path, snapshot_dtype=dtype)
    load_engine(e, prm, modes, snap)
    return e


def _random_engine(n, m, r, p, seed=0):
    """Seeded parameters and data for shapes POD cannot give (n < r): U = recon(params) * (1 + 0.3 noise) so r is a fraction of U."""
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


def _reference(e):
    """fp64 marginals of reconstruct().double() - U.double() and of U, on the device; also the marginals of recon^2."""
    rec = e.reconstruct().double()
    u = e.U[:, :e.n].double()
    r2, u2, c2 = (rec - u) ** 2, u ** 2, rec ** 2
    return {"snapshot_residual2": r2.sum(1), "snapshot_norm2": u2.sum(1), "point_residual2": r2.sum(0), "point_norm2": u2.sum(0),
            "snapshot_recon2": c2.sum(1), "point_recon2": c2.sum(0)}


def _profile(e):
    out = e.residual_profile()
    torch.cuda.synchronize()
    return out


# ------------------------------------------------------------------------------------------------ 1. against the materialised recon
# (label, builder args): every path of desmo_reconstruct / the training step, ragged and edge sizes
CASES = [
    ("r4p2-K27-fusedtc", ("channel", 2000, 300, 4, 2)),
    ("r4p3-K47", ("cylinder", 1500, 200, 4, 3)),
    ("r8p2-K69", ("cylinder", 1200, 150, 8, 2)),
    ("r8p3-K189", ("cylinder", 1500, 200, 8, 3)),
    ("r32p2-K657", ("channel", 1000, 300, 32, 2)),
    ("r64p1-K257", ("channel", 700, 150, 64, 1)),
    ("fourier-r2p2", ("cylinder", 900, 120, 2, 2, 4)),
    ("fourier-r8p3", ("cylinder", 700, 90, 8, 3, 3)),
    ("m1300-r4p2", ("aneurysm", 600, 1300, 4, 2)),
    ("m1300-r8p3", ("aneurysm", 600, 1300, 8, 3)),
    ("n4100-r4p2", ("channel", 4100, 130, 4, 2)),
    ("n4100-r32p2", ("channel", 4100, 130, 32, 2)),
]


def _is_gemm_recon(e):
    return not (e.r <= 8 and e.K <= 80)  # desmo_reconstruct's FFMA kernel covers r <= 8, K <= 80


def _check_against_reference(e):
    got, ref = _profile(e), _reference(e)
    for k in KEYS:
        assert got[k].shape == ref[k].shape, k
        assert torch.isfinite(got[k]).all(), k
    assert got["snapshot_residual2"].dtype == torch.float64 and got["point_residual2"].dtype == torch.float32
    # the U marginals never depend on the recon
    for k, b in (("snapshot_norm2", SNAP_BOUND), ("point_norm2", POINT_BOUND)):
        err = (got[k].double() - ref[k]).abs()
        assert bool((err <= b * ref[k] + 1e-300).all()), (k, float((err / ref[k].clamp_min(1e-300)).max()))
    worst = {}
    for k, b, c2 in (("snapshot_residual2", SNAP_BOUND, "snapshot_recon2"), ("point_residual2", POINT_BOUND, "point_recon2")):
        g, r = got[k].double(), ref[k]
        bound = b * r
        if not _is_gemm_recon(e):
            bound = bound + 2 * ETA_FFMA * torch.sqrt(r * ref[c2]) + ETA_FFMA ** 2 * ref[c2]
        err = (g - r).abs()
        worst[k] = float((err / bound.clamp_min(1e-300)).max())
        assert bool((err <= bound).all()), (k, worst[k])
    # r is not trivially small: the test exercises cancellation in the recon
    assert float(ref["snapshot_residual2"].sum()) > 1e-4 * float(ref["snapshot_norm2"].sum())
    return got, worst


@pytest.mark.parametrize("label,args", CASES, ids=[c[0] for c in CASES])
def test_profile_matches_fp64_sums_of_the_reconstruction(label, args):
    e = _engine(*args)
    got, worst = _check_against_reference(e)
    print(label, "worst error / bound", worst)
    # pad columns of the point map are exactly 0
    snap = torch.empty(2, e.m, dtype=torch.float64, device=DEV)
    point = torch.full((2, e.ld), 7.0, dtype=torch.float32, device=DEV)
    import ctypes as C

    from desmo_b200._lib import check

    check(e.lib.desmo_residual_profile(C.byref(e.shape), e.U.data_ptr(), e._u_dtype(), e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(),
                                       e.W.data_ptr(), snap.data_ptr(), point.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert e.ld > e.n
    assert int((point[:, e.n:] != 0).sum()) == 0
    assert torch.equal(point[0, :e.n], got["point_residual2"]) and torch.equal(snap[0], got["snapshot_residual2"])


@pytest.mark.parametrize("n,r,p", [(1, 4, 2), (1, 8, 3), (129, 4, 2)])
def test_edge_point_counts(n, r, p):
    e = _random_engine(n, 70, r, p)
    _check_against_reference(e)


# ------------------------------------------------------------------------------------------------ 2. against the oracle
@pytest.mark.parametrize("name", sorted(os.path.basename(f)[:-4] for f in os.listdir(GOLDEN) if f.startswith("grad_") and f.endswith(".npz")))
def test_totals_match_golden_loss_and_residual_norm2(name):
    from desmo_b200 import DesmoEngine

    fx, meta, modes, snap, prm = golden_case(name)
    e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device(DEV))
    load_engine(e, prm, modes, snap)
    got = _profile(e)
    want = float(fx["mse"]) * prm.n * prm.m
    s_snap, s_point = float(got["snapshot_residual2"].sum()), float(got["point_residual2"].double().sum())
    assert abs(s_snap - want) <= 1e-5 * want, (s_snap, want)
    rn2 = e.residual_norm2()
    assert abs(s_snap - rn2) <= 1e-5 * s_snap and abs(s_point - s_snap) <= 1e-5 * s_snap
    u = torch.from_numpy(snap).to(DEV).double()  # the stored fp32 U
    u2t, u2x = (u ** 2).sum(1), (u ** 2).sum(0)
    assert bool(((got["snapshot_norm2"] - u2t).abs() <= SNAP_BOUND * u2t).all())
    assert bool(((got["point_norm2"].double() - u2x).abs() <= POINT_BOUND * u2x).all())


# ------------------------------------------------------------------------------------------------ 3. no side effects, reproducible
def _buffers(e):
    return {k: v.clone() for k, v in vars(e).items() if torch.is_tensor(v)}


@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3), ("cylinder", 900, 120, 2, 2, 4)],
                         ids=["fusedtc", "gemm", "fourier"])
def test_no_side_effects_and_bit_reproducible(args):
    e = _engine(*args)
    e.train_step()  # red, dphi, losses, Adamax state and the step counter hold real values
    e.build_w(False)  # W (and its planes in the workspace) of the current parameters, as residual_profile rebuilds them
    torch.cuda.synchronize()
    before = _buffers(e)
    a = _profile(e)
    after = _buffers(e)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    b = _profile(e)
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k


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
                e.residual_profile()
            tr.step()
            losses.append(e.losses.clone())
        torch.cuda.synchronize()
        runs.append((e, torch.stack(losses)))
    (e0, l0), (e1, l1) = runs
    assert torch.equal(l0, l1)
    for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "omega", "omega_m", "omega_u",
              "hyper", "step_dev", "losses", "red", "dphi"):
        assert torch.equal(getattr(e0, k), getattr(e1, k)), k


# ------------------------------------------------------------------------------------------------ 4. bf16 storage
@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3)], ids=["r4p2", "r8p3"])
def test_bf16_equals_fp32_storage_of_uq(args):
    from desmo_b200 import DesmoEngine

    kind, n, m, r, p = args
    _, modes, snap, prm = make_case(kind, n, m, r, p, omega_init=10.0, perturb_rel=0.3)
    out = []
    for dt, s in ((torch.bfloat16, snap), (torch.float32, torch.from_numpy(snap).bfloat16().float().numpy())):
        e = DesmoEngine(n, m, p, r, omega_init=10.0, device=torch.device(DEV), snapshot_dtype=dt)
        load_engine(e, prm, modes, s)
        out.append(_profile(e))
    for k in KEYS:
        assert torch.equal(out[0][k], out[1][k]), k


# ------------------------------------------------------------------------------------------------ 5. masks
@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3)], ids=["r4p2", "r8p3"])
def test_masked_gates_total_matches_residual_norm2(args):
    e = _engine(*args)
    norms = e.term_norms()
    saved = e.gates.clone()
    for thr in (float(norms.median()), float(norms.quantile(0.9))):
        e.gates.copy_(saved)
        e.gates.mul_((norms >= thr).to(e.gates.dtype))  # what threshold_sweep does for one threshold
        total = float(_profile(e)["snapshot_residual2"].sum())
        rn2 = e.residual_norm2()
        assert abs(total - rn2) <= 1e-5 * total, (thr, total, rn2)
    e.gates.copy_(saved)


# ------------------------------------------------------------------------------------------------ 6. torch.ops route, dtypes
def test_ops_route_is_bitwise_equal_and_rejects_other_dtypes():
    import desmo_b200.ops as ops
    from desmo_b200 import _lib

    e = _engine("cylinder", 1500, 200, 8, 3)
    step = e.step_dev.clone()
    a = _profile(e)
    b = ops.engine_residual_profile_via_ops(e)
    torch.cuda.synchronize()
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(e.step_dev, step)
    sa = ops._shape_args(e)
    snap = torch.full((2, e.m), 3.0, dtype=torch.float64, device=DEV)
    point = torch.full((2, e.ld), 3.0, dtype=torch.float32, device=DEV)
    for dt in (torch.float16, torch.float64):
        e.U = torch.zeros(e.m, e.ld, dtype=dt, device=DEV)
        with pytest.raises(_lib.DesmoError):
            e.residual_profile()
        with pytest.raises(_lib.DesmoError):
            torch.ops.desmo_b200.residual_profile(e.U, e.P, e.phi, e.omega, e.W, snap, point, *sa)
    torch.cuda.synchronize()
    assert bool((snap == 3.0).all()) and bool((point == 3.0).all())  # nothing was launched
    # the C ABI rejects an unknown u_dtype by itself
    import ctypes as C

    rc = e.lib.desmo_residual_profile(C.byref(e.shape), e.U.data_ptr(), 7, e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(),
                                      e.W.data_ptr(), snap.data_ptr(), point.data_ptr(), 0)
    assert rc == 1 and b"u_dtype" in e.lib.desmo_last_error()


# ------------------------------------------------------------------------------------------------ 7. point-sharded
def test_sharded_profile_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29673", os.path.join(ROOT, "tests", "_profile_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("PROFILE_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("PROFILE_RESULT "):])
    # both snapshot sums are within SNAP_BOUND of the exact sums of the same fp32 r: they differ by at most twice that
    assert res["snapshot_rel_vs_unsharded"] <= 2 * SNAP_BOUND, res
    assert res["snapshot_identical_across_ranks"], res
    assert res["point_slabs_bit_identical"], res
