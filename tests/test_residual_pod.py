"""Residual POD (DesmoEngine.residual_pod, desmo_residual_gram / desmo_residual_modes): the singular spectrum and leading modes of
R = recon - U, from the Gram C_R = R R^T accumulated over chunks of points without forming R.

Error model.  GEMM 1 forms r exactly as the training step does (for K > 80 or r > 8 bit for bit reconstruct() - U, otherwise within
eta |recon| of it, eta = 2^-14 as in test_residual_profile.py).  The Gram GEMM multiplies the two bf16 planes r = b1 + b2 + e
(|e| <= 2^-16 |r|) with three products (b1 b1 + b1 b2 + b2 b1; the omitted b2 b2 <= 2^-16 |r r'|): 3 * 2^-16 of sum_x |r r'|.  The
tensor core's truncating adds (48 MMAs per chain, <= 2^-23 each), the fp32 sums of the chains, fp64 beyond and the final fp32 rounding
add < 2^-16 more, so |C - C64| <= B = 2^-14 |R| |R|^T (+ the eta terms), entrywise, and ||C - C64||_2 <= ||B||_2.  Eigenvalues then obey
Weyl's bound |lambda_i - lambda64_i| <= ||C - C64||_2 (plus the solver's floor 2^-23 trace for a mode reported as 0), eigenvectors
Davis-Kahan's sin(theta_i) <= 2 ||C - C64||_2 / gap_i.  So the spectrum is resolved down to about ||B||_2 <= 2^-14 trace(C_R)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import golden_case, load_engine, make_case

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BETA = 2.0 ** -14
ETA_FFMA = 2.0 ** -14
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ("singular_values", "sigma", "temporal_modes", "spatial_modes", "energy", "cumulative_energy", "gram")


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


def _is_gemm_recon(e):
    return not (e.r <= 8 and e.K <= 80)  # desmo_reconstruct's FFMA kernel covers r <= 8, K <= 80


def _pod(e, k):
    out = e.residual_pod(k)
    torch.cuda.synchronize()
    return out


def _reference(e):
    """fp64 R = reconstruct() - U (m, n), its Gram, the entrywise bound B of |C - C64| and its spectral norm."""
    rec = e.reconstruct().double()
    R = rec - e.U[:, :e.n].double()
    A = R.abs()
    B = BETA * (1 + 2.0 ** -10) * (A @ A.T)
    if not _is_gemm_recon(e):
        Q = rec.abs()
        B = B + ETA_FFMA * (A @ Q.T + Q @ A.T) + ETA_FFMA ** 2 * (Q @ Q.T)
    lam = np.linalg.svd(R.cpu().numpy(), compute_uv=False) ** 2
    lam = np.concatenate([lam, np.zeros(e.m - lam.size)])
    return {"R": R, "rec": rec, "C64": R @ R.T, "B": B, "Bnorm": float(torch.linalg.matrix_norm(B, ord=2)), "lam": lam}


def _check_gram(e, got, ref):
    Cg = got["gram"].double()
    assert torch.equal(got["gram"], got["gram"].T)  # mirrored from the upper tiles
    err = (Cg - ref["C64"]).abs()
    worst = float((err / ref["B"].clamp_min(1e-300)).max())
    assert bool((err <= ref["B"]).all()), worst
    tr64 = float(ref["C64"].diagonal().sum())
    trb = float(ref["B"].diagonal().sum())
    assert abs(got["residual_norm2"] - tr64) <= trb, (got["residual_norm2"], tr64, trb)
    return worst, float(torch.linalg.matrix_norm(Cg - ref["C64"], ord=2))


def _check_spectrum(e, got, ref, E2):
    S = got["singular_values"].numpy()
    lam, tr = ref["lam"], got["residual_norm2"]
    assert S.shape == (e.m,) and np.all(np.diff(S) <= 0) and np.all(np.isfinite(S))
    bound = E2 + np.where(S == 0, 2.0 ** -23 * tr, 0.0) + 1e-12 * lam[0]
    assert np.all(np.abs(S ** 2 - lam) <= bound), float(np.max(np.abs(S ** 2 - lam) / bound))
    k = got["sigma"].numel()
    assert torch.equal(got["sigma"].cpu(), torch.from_numpy(S[:k]).float())
    assert np.allclose(got["energy"].numpy(), S[:k] ** 2 / tr, rtol=1e-6, atol=0)


def _check_modes(e, got, ref, E2):
    """Temporal and spatial modes against fp64 for well-separated sigma_i, orthonormality, and the rank-k reconstruction."""
    R, lam, Eb = ref["R"], ref["lam"], ref["Bnorm"]
    k = got["sigma"].numel()
    U64, s64, Vh64 = torch.linalg.svd(R, full_matrices=False)  # R = U64 diag(s64) Vh64: v_i = U64[:, i], psi_i = Vh64[i]
    V, Psi, sig = got["temporal_modes"].double(), got["spatial_modes"].double(), got["sigma"].double()
    assert bool(torch.allclose(V.norm(dim=1), torch.ones(k, dtype=torch.float64, device=DEV), atol=1e-5))
    eta = 0.0 if _is_gemm_recon(e) else ETA_FFMA
    checked = 0
    for i in range(min(k, s64.numel())):
        gap = min(lam[i - 1] - lam[i] if i > 0 else np.inf, lam[i] - lam[i + 1] if i + 1 < lam.size else np.inf)
        if not gap > 10 * E2 or lam[i] < 100 * Eb:
            continue
        sin_t = 2 * E2 / gap
        sg = torch.sign(V[i] @ U64[:, i])
        dv = float((V[i] - sg * U64[:, i]).norm())
        assert dv <= np.sqrt(2) * sin_t + 1e-5, (i, dv, sin_t)
        s_i = float(s64[i])
        gemm = (4 * 2.0 ** -16 * float((R.abs().T @ V[i].abs()).norm()) + eta * float((ref["rec"].abs().T @ V[i].abs()).norm())) / s_i
        tol = (float(s64[0]) / s_i) * (dv + 1e-6) + abs(float(sig[i]) - s_i) / s_i + gemm + 1e-5
        dpsi = float((Psi[i] - sg * Vh64[i]).norm())
        assert dpsi <= tol, (i, dpsi, tol)
        checked += 1
    # orthonormal spatial modes (those well above the Gram's rounding level)
    big = [i for i in range(k) if float(sig[i]) ** 2 > 100 * Eb]
    if big:
        G = Psi[big] @ Psi[big].T
        sb = sig[big]
        tol = 3 * Eb / torch.outer(sb, sb) + 1e-5
        assert bool(((G - torch.eye(len(big), dtype=torch.float64, device=DEV)).abs() <= tol).all())
    # R ~ sum_i sigma_i v_i psi_i^T: ||R - V V^T R~||_F <= sqrt(tail + 2 k ||E||) + split error of GEMM 3 (+ eta)
    Rk = (V * sig[:, None]).T @ Psi
    tail = float(lam[k:].sum())
    lhs = float((R - Rk).norm())
    rhs = np.sqrt(tail + 2 * k * Eb) + 2.0 ** -13 * float(R.norm()) + eta * float(ref["rec"].norm())
    assert lhs <= rhs, (lhs, rhs)
    return checked


# ------------------------------------------------------------------------------------------------ 1-2. against fp64
CASES = [
    ("r4p2-K27-fusedtc", ("channel", 2000, 300, 4, 2)),
    ("r4p3-K47", ("cylinder", 1500, 200, 4, 3)),
    ("r8p2-K69", ("cylinder", 1200, 150, 8, 2)),
    ("r32p2-K657", ("channel", 1000, 300, 32, 2)),
    ("r64p1-K257", ("channel", 700, 150, 64, 1)),
    ("fourier-r2p2", ("cylinder", 900, 120, 2, 2, 4)),
    ("m1300-r4p2", ("aneurysm", 600, 1300, 4, 2)),
    ("n4100-r8p3", ("channel", 4100, 130, 8, 3)),
]


@pytest.mark.parametrize("label,args", CASES, ids=[c[0] for c in CASES])
def test_gram_spectrum_and_modes_against_fp64(label, args):
    e = _engine(*args)
    got = _pod(e, 8)
    ref = _reference(e)
    worst, E2 = _check_gram(e, got, ref)
    _check_spectrum(e, got, ref, E2)
    checked = _check_modes(e, got, ref, E2)
    print(label, "gram worst err / bound", worst, "||E||_2 / lambda_1", E2 / ref["lam"][0], "modes checked", checked)
    # the trace is ||R||_F^2: the training step's residual_norm2 up to the split error and the order of the sums
    rn2 = e.residual_norm2()
    assert abs(got["residual_norm2"] - rn2) <= 2.0 ** -13 * rn2 + (0 if _is_gemm_recon(e) else 4 * ETA_FFMA * rn2 ** 0.5 * float(ref["rec"].norm()))
    assert got["spatial_modes"].shape == (8, e.n) and got["temporal_modes"].shape == (8, e.m)


# ------------------------------------------------------------------------------------------------ several chunks of points
def _chunks(e):
    """The point chunks and the Gram's slice layout as csrc/gemm_path.cu (residual_pod_layout) lays them out."""
    sms = torch.cuda.get_device_properties(e.device).multi_processor_count
    Kr, mp = (e.K + 63) // 64 * 64, (e.m + 127) // 128 * 128
    tiles = (mp // 128) * (mp // 128 + 1) // 2
    rows_c = min(max((64 << 20) // (6 * Kr + 4 * mp) // 128 * 128, 128), e.ld)
    ns = min(max(sms // tiles, 1), 32, rows_c // 64)
    pts = [min(rows_c, e.ld - x0) for x0 in range(0, e.ld, rows_c)]
    return pts, ns


# The C_R slice partials accumulate over the chunks in fp64 (first chunk stores, later chunks add), every chunk uses the first chunk's
# slice layout (a short last chunk leaves trailing slices with no k-block: they must add +0), and GEMM 3 of the modes pass writes each
# chunk's points at x0 > 0.  These shapes run several chunks and end in a short one.
MULTI = [
    ("3chunks+128-r32p2-K657", ("channel", 35000, 300, 32, 2)),       # rows_c = 11 648: 3 x 11 648 + 128 points, 22 of 24 slices empty
    ("2chunks+short-r4p2-K27", ("channel", 80000, 300, 4, 2)),        # rows_c = 34 944: 2 x 34 944 + 10 240 points
]


@pytest.mark.parametrize("label,args", MULTI, ids=[c[0] for c in MULTI])
def test_several_chunks_against_fp64(label, args):
    e = _engine(*args)
    pts, ns = _chunks(e)
    assert len(pts) >= 3 and pts[-1] < pts[0], pts
    if label.startswith("3chunks"):
        assert pts == [11648] * 3 + [128] and ns - pts[-1] // 64 == 22, (pts, ns)
    got = _pod(e, 8)
    ref = _reference(e)
    worst, E2 = _check_gram(e, got, ref)
    _check_spectrum(e, got, ref, E2)
    checked = _check_modes(e, got, ref, E2)
    assert checked >= 1
    print(label, "chunks", pts, "slices", ns, "gram worst err / bound", worst, "||E||_2 / lambda_1", E2 / ref["lam"][0],
          "modes checked", checked)
    # the chunked sums against one that is not split: the trace is ||R||_F^2 within the split error
    rn2 = float((ref["R"] ** 2).sum())
    assert abs(got["residual_norm2"] - rn2) <= 2.0 ** -13 * rn2 + (0 if _is_gemm_recon(e) else 4 * ETA_FFMA * rn2 ** 0.5 * float(ref["rec"].norm()))
    _same(got, _pod(e, 8))


@pytest.mark.parametrize("n,r,p", [(1, 4, 2), (129, 8, 3)])
def test_edge_point_counts(n, r, p):
    e = _random_engine(n, 70, r, p)
    got = _pod(e, 4)
    ref = _reference(e)
    _, E2 = _check_gram(e, got, ref)
    _check_spectrum(e, got, ref, E2)
    if n == 1:  # rank one: everything beyond sigma_1 at the floor
        assert float(got["singular_values"][1:].abs().max()) ** 2 <= E2 + 2.0 ** -23 * got["residual_norm2"]


# ------------------------------------------------------------------------------------------------ 3. planted structure
def test_planted_rank_two_residual():
    e = _engine("cylinder", 1500, 200, 8, 3)  # K = 189: reconstruct() runs GEMM 1 itself, so R is exactly the planted part + rounding
    rec = e.reconstruct().double()
    g = torch.Generator().manual_seed(3)
    psi, _ = torch.linalg.qr(torch.randn(e.n, 2, generator=g, dtype=torch.float64))
    v, _ = torch.linalg.qr(torch.randn(e.m, 2, generator=g, dtype=torch.float64))
    psi, v = psi.to(DEV), v.to(DEV)
    a = 1e-2 * float(rec.norm())
    b = 0.4 * a
    U = rec + a * torch.outer(v[:, 0], psi[:, 0]) + b * torch.outer(v[:, 1], psi[:, 1])
    e.set_snapshot(U.float())
    got = _pod(e, 4)
    R = rec - e.U[:, :e.n].double()
    delta = float((R + a * torch.outer(v[:, 0], psi[:, 0]) + b * torch.outer(v[:, 1], psi[:, 1])).norm())  # fp32 rounding of U
    assert delta <= 2.0 ** -23 * float(U.norm())
    Eb = float(torch.linalg.matrix_norm(BETA * (R.abs() @ R.abs().T), ord=2))
    S = got["singular_values"].numpy()
    for i, want in enumerate((a, b)):
        assert abs(S[i] - want) <= delta + Eb / want, (i, S[i], want)
    assert float(np.max(S[2:])) <= delta + np.sqrt(Eb + 2.0 ** -23 * got["residual_norm2"]), S[:6]
    pert = 2 * a * delta + delta ** 2 + Eb
    for i, gap in enumerate((a * a - b * b, min(a * a - b * b, b * b))):
        sin_t = 2 * pert / gap
        cv = abs(float(got["temporal_modes"][i].double() @ v[:, i]))
        cp = abs(float(got["spatial_modes"][i].double() @ psi[:, i]))
        assert cv >= 1 - sin_t - 1e-6, (i, cv, sin_t)
        assert cp >= 1 - 4 * sin_t * a / b - 2.0 ** -13, (i, cp, sin_t)


# ------------------------------------------------------------------------------------------------ 4. cross-check with POD
def test_all_gates_zero_matches_pod_analysis():
    e = _engine("cylinder", 3000, 100, 8, 2)
    e.pod_analysis()
    torch.cuda.synchronize()
    Sp, P, Cpod = e.pod_singular_values.numpy(), e.P[:, :e.n].clone(), e.pod_gram.double()
    e.gates.zero_()  # R = -U exactly
    got = _pod(e, e.r)
    u = e.U[:, :e.n].double()
    C64 = u @ u.T
    E2 = float(torch.linalg.matrix_norm(got["gram"].double() - C64, ord=2))
    Ep = float(torch.linalg.matrix_norm(Cpod - C64, ord=2))
    S, tr = got["singular_values"].numpy(), got["residual_norm2"]
    bound = E2 + Ep + 2.0 ** -23 * tr + 1e-12 * S[0] ** 2
    assert np.all(np.abs(S ** 2 - Sp ** 2) <= bound), float(np.max(np.abs(S ** 2 - Sp ** 2) / bound))
    lam = Sp ** 2
    for i in range(e.r):
        gap = min(lam[i - 1] - lam[i] if i > 0 else np.inf, lam[i] - lam[i + 1])
        if not gap > 10 * (E2 + Ep) or lam[i] < 1e-6 * lam[0]:
            continue
        psi = got["spatial_modes"][i].double()
        sg = torch.sign(psi @ -P[i].double())
        d = float((psi + sg * P[i].double()).norm())
        tol = (S[0] / S[i]) * 4 * np.sqrt(2) * (E2 + Ep) / gap + 2.0 ** -12
        assert d <= tol, (i, d, tol)


# ------------------------------------------------------------------------------------------------ 5. edge cases
def test_perfect_fit_gives_zeros_and_no_nan():
    e = _engine("cylinder", 1500, 200, 8, 3)  # K = 189: reconstruct() is GEMM 1's Rec, bit for bit
    e.set_snapshot(e.reconstruct())
    got = _pod(e, 8)
    assert got["residual_norm2"] == 0.0
    for k in KEYS:
        t = got[k]
        assert bool(torch.isfinite(t).all()) and float(t.abs().max()) == 0.0, k


def test_k_equals_m():
    e = _random_engine(3000, 50, 4, 2)
    got = _pod(e, 50)
    ref = _reference(e)
    _, E2 = _check_gram(e, got, ref)
    _check_spectrum(e, got, ref, E2)
    V = got["temporal_modes"].double()
    assert bool(((V @ V.T - torch.eye(50, dtype=torch.float64, device=DEV)).abs() <= 1e-5).all())


def test_bad_arguments_raise_before_any_launch():
    from desmo_b200 import DesmoEngine, _lib

    e = DesmoEngine(1000, 50, 2, 4, device=torch.device(DEV))
    with pytest.raises(_lib.DesmoError):
        e.residual_pod(4)  # no snapshot
    e.set_snapshot(torch.randn(50, 1000))
    for k in (0, 51, 65, -1):
        with pytest.raises(_lib.DesmoError):
            e.residual_pod(k)
    scratch = e._residual_pod_scratch()
    Cm = torch.full((50, 50), 7.0, device=DEV)
    tr = torch.full((1,), 7.0, dtype=torch.float64, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    args = (C.byref(e.shape), e.U.data_ptr(), e._u_dtype(), e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(), e.W.data_ptr())
    assert e.lib.desmo_residual_gram(*args, Cm.data_ptr(), tr.data_ptr(), scratch.data_ptr(), scratch.numel() - 1, st) == 1
    assert b"scratch too small" in e.lib.desmo_last_error()
    modes = torch.full((4, e.ld), 7.0, device=DEV)
    V, sg = torch.zeros(4, 50, device=DEV), torch.ones(4, device=DEV)
    assert e.lib.desmo_residual_modes(*args, 4, V.data_ptr(), sg.data_ptr(), modes.data_ptr(), scratch.data_ptr(), 1024, st) == 1
    assert e.lib.desmo_residual_modes(*args, 0, V.data_ptr(), sg.data_ptr(), modes.data_ptr(), scratch.data_ptr(), scratch.numel(), st) == 1
    torch.cuda.synchronize()
    assert bool((Cm == 7.0).all()) and bool((tr == 7.0).all()) and bool((modes == 7.0).all())  # nothing was launched


# ------------------------------------------------------------------------------------------------ 6. invariants
def _same(a, b):
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k
    assert a["residual_norm2"] == b["residual_norm2"]


@pytest.mark.parametrize("args", [("channel", 2000, 300, 4, 2), ("cylinder", 1500, 200, 8, 3), ("cylinder", 900, 120, 2, 2, 4)],
                         ids=["fusedtc", "gemm", "fourier"])
def test_no_side_effects_and_bit_reproducible(args):
    e = _engine(*args)
    e.train_step()
    e.pod_analysis()
    e.build_w(False)
    torch.cuda.synchronize()
    before = {k: v.clone() for k, v in vars(e).items() if torch.is_tensor(v)}
    pod_attrs = {k: v for k, v in vars(e).items() if k.startswith("pod_")}
    a = _pod(e, 8)
    for k, v in vars(e).items():
        if torch.is_tensor(v):
            assert torch.equal(before[k], v), k
    for k, v in pod_attrs.items():
        assert getattr(e, k) is v, k
    _same(a, _pod(e, 8))


def test_bf16_equals_fp32_storage_of_uq():
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case("cylinder", 1500, 200, 8, 3, omega_init=10.0, perturb_rel=0.3)
    out = []
    for dt, s in ((torch.bfloat16, snap), (torch.float32, torch.from_numpy(snap).bfloat16().float().numpy())):
        e = DesmoEngine(1500, 200, 3, 8, omega_init=10.0, device=torch.device(DEV), snapshot_dtype=dt)
        load_engine(e, prm, modes, s)
        out.append(_pod(e, 8))
    _same(*out)


def test_active_set_equals_zeroed_gates():
    a = _engine("cylinder", 1500, 200, 8, 3)
    b = _engine("cylinder", 1500, 200, 8, 3)
    mask = torch.rand(a.K, generator=torch.Generator().manual_seed(5)) < 0.5
    mask[0] = True
    a.set_active_terms(mask)
    b.gates.mul_(mask.to(DEV, torch.float32))
    _same(_pod(a, 8), _pod(b, 8))


@pytest.mark.parametrize("path", [0, 3])
def test_pod_between_training_steps_changes_nothing(path):
    from desmo_b200 import DesmoEngine, DesmoTrainer

    fx, meta, modes, snap, prm = golden_case("traj_chan_r4p2")
    runs = []
    for with_pod in (False, True):
        e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device(DEV), path=path)
        load_engine(e, prm, modes, snap)
        tr = DesmoTrainer(e, lrs=meta["lrs"], beta=meta["beta"], l1_lambda=meta["l1_lambda"], patience=2, sched_every=3,
                          use_cuda_graph=True, device_scheduler=True)
        losses = []
        for i in range(20):
            if with_pod and i == 10:
                e.residual_pod(4)
            tr.step()
            losses.append(e.losses.clone())
        torch.cuda.synchronize()
        runs.append((e, torch.stack(losses)))
    (e0, l0), (e1, l1) = runs
    assert torch.equal(l0, l1)
    for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "omega", "omega_m", "omega_u",
              "hyper", "step_dev", "losses", "red", "dphi", "P"):
        assert torch.equal(getattr(e0, k), getattr(e1, k)), k


def test_ops_route_is_bitwise_equal_and_model_passes_through():
    import desmo_b200.ops as ops
    from desmo_b200 import DESMO

    e = _engine("channel", 1000, 300, 32, 2)
    step = e.step_dev.clone()
    a = _pod(e, 8)
    b = ops.engine_residual_pod_via_ops(e, 8)
    torch.cuda.synchronize()
    for k in ("singular_values", "sigma", "temporal_modes", "spatial_modes", "gram"):
        assert torch.equal(a[k], b[k]), k
    assert a["residual_norm2"] == b["residual_norm2"]
    assert torch.equal(e.step_dev, step)
    _, modes, snap, prm = make_case("channel", 1000, 300, 32, 2, omega_init=10.0, perturb_rel=0.3)
    model = DESMO(1000, 300, 2, 32, 10.0, pod_modes=modes, device=torch.device(DEV))
    load_engine(model.engine, prm, modes, snap)
    _same(model.residual_pod(8), a)


# ------------------------------------------------------------------------------------------------ 7. point-sharded
def test_sharded_residual_pod_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29679", os.path.join(ROOT, "tests", "_residual_pod_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("RPOD_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("RPOD_RESULT "):])
    assert res["gram_rel_vs_unsharded"] <= 1e-6, res
    assert res["sv2_err_over_trace"] <= 1e-6, res
    assert res["identical_across_ranks"], res
    assert res["slab_rel_vs_unsharded"] <= 1e-4, res
