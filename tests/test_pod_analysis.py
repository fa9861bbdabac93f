"""POD for up to 64 modes with the full spectrum: the dense fp64 eigensolver (desmo_pod_eigh) and DesmoEngine.pod_analysis().

1  Solver alone, against np.linalg.eigh of the device's own Gram in fp64: all m values of S, floor, sign, orthonormality, residuals,
   Weyl and Davis-Kahan bounds, and the workspace report.
2  pod_analysis() end to end against np.linalg.svd of the fp64 data; agreement with pod_from_snapshot at r <= 14.
3  Floor on rank-deficient data.  4  Storage, determinism, ops route, a failing call.  5  Training from the new modes.  6  Two GPUs.
Each bound is derived where it is used.  u = 2^-53 (fp64) and U32 = 2^-24 (fp32) are the unit roundoffs."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_pod_reference import SPECTRA, _clusters, _e2e_data, _engine, _gram, _spectral, _spectrum, _upload

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U32 = 2.0 ** -24
U64 = 2.0 ** -53
EIGH_TOL = 2.0 ** -27


def _L():
    from desmo_b200 import _lib as L
    from desmo_b200 import ops  # noqa: F401  (registers torch.ops.desmo_b200.*)

    return L


def _eigh(Cm, r):
    L = _L()
    m = Cm.shape[0]
    nbytes = C.c_size_t(0)
    L.check(L.load().desmo_pod_eigh_workspace_bytes(m, r, C.byref(nbytes)), "desmo_pod_eigh_workspace_bytes")
    ws = torch.full((nbytes.value,), 0xFF, dtype=torch.uint8, device=DEV)
    S = torch.full((m,), float("nan"), dtype=torch.float64, device=DEV)
    V, sigma = torch.full((r, m), float("nan"), device=DEV), torch.full((r,), float("nan"), device=DEV)
    torch.ops.desmo_b200.pod_eigh(Cm, S, V, sigma, ws, m, r)
    torch.cuda.synchronize()
    status = int(ws[:4].view(torch.int32).item())
    return S.cpu().numpy(), V.double().cpu().numpy(), sigma.double().cpu().numpy(), status, float(ws[8:16].view(torch.float64).item())


def _solver_bound(m, lam1):
    """Backward error of the solver in fp64: Householder tridiagonalisation perturbs A by ||E|| <= c m u ||A|| (Higham, Accuracy and
    Stability, Thm 19.4; c a small constant, taken as 4 with the sums' rounding modelled as the worst case), bisection adds at most
    2 eps ||T|| and inverse iteration leaves a residual of the same order.  numpy's reference has the same order of error, so the
    two are compared at 2 * (4 m + 4) u lambda_1; at m = 4096 this is 3.6e-12 lambda_1, 5000x tighter than the subspace solver's
    2e-8 lambda_1."""
    return 2.0 * (4.0 * m + 4.0) * U64 * lam1


@pytest.fixture(scope="module")
def grams():
    cache = {}

    def get(kind, m):
        if (kind, m) not in cache:
            if len(cache) > 3:
                cache.clear()
            X = _spectral(m + 7, _spectrum(kind, m), seed=m)
            if m >= 2:
                Cm = _gram(_upload(X), m + 7, 0)
            else:   # the Gram entry points need m >= 2; the solver also takes the 1 x 1 Gram, formed here in fp64 and rounded once
                Cm = torch.as_tensor(X.T @ X, dtype=torch.float32, device=DEV)
            C64 = Cm.double().cpu().numpy()
            C64 = np.tril(C64) + np.tril(C64, -1).T   # the solver reads the lower triangle, as eigh(UPLO='L')
            lam, E = np.linalg.eigh(C64)
            cache[(kind, m)] = (Cm, C64, lam[::-1].copy(), E[:, ::-1].copy())
        return cache[(kind, m)]

    return get


def _check_solver(Cm, C64, lam, E, r):
    m = C64.shape[0]
    S, V, sigma, status, reported = _eigh(Cm, r)
    lam1, trace = lam[0], float(np.trace(C64))
    floor = 2.0 ** -23 * trace
    tol = _solver_bound(m, lam1)
    assert status == 0
    assert np.isfinite(S).all() and np.isfinite(V).all() and np.isfinite(sigma).all()
    assert np.all(np.diff(S) <= 0.0)                               # descending
    # every value of S: S_i^2 within the backward-error bound of lambda_i (+ the rounding of sqrt and of the square: 3u lambda_i)
    live_S = S > 0
    assert np.all(np.abs(S[live_S] ** 2 - lam[live_S]) <= tol + 3 * U64 * lam[live_S]), np.max(np.abs(S[live_S] ** 2 - lam[live_S])) / lam1
    # floor: S_i = 0 exactly for the values at the Gram's rounding level, and only for those (up to the solver's error)
    assert np.all(lam[~live_S] <= floor + tol) and np.all(lam[live_S] >= floor - tol)
    assert np.array_equal(sigma, S[:r].astype(np.float32).astype(np.float64))
    # orthonormal to fp32 rounding, floored rows included: (v + d).(w + e) - v.w <= |d| + |e| + |d||e| with |d|, |e| <= u |v|
    assert np.abs(V @ V.T - np.eye(r)).max() <= 4 * U32
    # sign convention: the largest-|.| entry of each V_i is positive
    assert all(V[i, np.argmax(np.abs(V[i]))] > 0 for i in range(r))
    live = sigma > 0
    res = np.zeros(r)
    theta = np.zeros(r)
    for i in np.flatnonzero(live):
        v = V[i]
        theta[i] = v @ C64 @ v / (v @ v)
        res[i] = np.linalg.norm(C64 @ v - theta[i] * v) / np.linalg.norm(v)
        # residual: the solver's error plus the fp32 rounding of v, ||(C - theta) dv|| <= lambda_1 U32 ||v||
        assert res[i] <= tol + U32 * lam1, (i, res[i] / lam1)
        # Weyl on the emitted sigma: solver error plus the fp32 rounding of sigma (2 U32 sigma^2 + U32^2 sigma^2)
        assert abs(sigma[i] ** 2 - lam[i]) <= tol + 3 * U32 * lam[i], (i, sigma[i] ** 2, lam[i])
    # the report: the device measured ||C x - lambda x|| / lambda_1 for the fp64 x; the host's value for fp32 v = x + dx differs by at most
    # ||(C - lambda) dx|| / lambda_1 <= U32 plus the Rayleigh-quotient shift (second order)
    host = max((np.linalg.norm(C64 @ V[i] - S[i] ** 2 * V[i]) / lam1 for i in np.flatnonzero(live)), default=0.0)
    assert 0.0 <= reported <= EIGH_TOL
    assert abs(host - reported) <= 2 * U32, (host, reported)
    # Davis-Kahan per cluster: ||(I - E E^T) V_K^T||_2 <= ||R_K||_F / gap_K (+ the fp32 rounding of V)
    nlive = int(live.sum())
    for K in _clusters(lam, 1e-6 * lam1):
        mine = [i for i in K if i < nlive]
        others = np.setdiff1d(np.arange(m), K)
        if not mine or others.size == 0:
            continue
        gap = min(np.min(np.abs(theta[i] - lam[others])) for i in mine)
        bound = np.linalg.norm(res[mine]) / gap + 2 * U32 * np.sqrt(len(mine))
        if bound >= 0.5:
            continue
        EK = E[:, K]
        VK = V[mine].T / np.linalg.norm(V[mine], axis=1)
        assert np.linalg.norm(VK - EK @ (EK.T @ VK), 2) <= bound, (K, bound)


@pytest.mark.parametrize("m", [1, 2, 10, 17, 200, 1000, 2100, 4096])
@pytest.mark.parametrize("kind", SPECTRA)
def test_eigh_against_fp64_eigh_of_device_gram(grams, kind, m):
    Cm, C64, lam, E = grams(kind, m)
    for r in (1, 8, 14, 15, 16, 32, 64):
        if r <= m:
            _check_solver(Cm, C64, lam, E, r)


# ------------------------------------------------------------------------------------------------ 2. end to end
def _svd(X):
    Xf = X.astype(np.float32).astype(np.float64)   # what U holds
    Us, S, _ = np.linalg.svd(Xf, full_matrices=False)
    return Xf, Us, S


def _check_modes(kind, X, Us, S, sigma, P, dC, res_bound):
    """Davis-Kahan of P against the SVD's left singular vectors (as test_pod_reference's end-to-end test): v_i is an eigenvector
    of C64 up to dC + the solver's residual; P_i = X v_i / sigma_i turns an angle phi into at most (S_0 / S_i) tan(phi)."""
    n = X.shape[0]
    lam = S ** 2
    live = sigma > 0
    nlive = int(live.sum())
    Pn = P[:nlive, :n] / np.linalg.norm(P[:nlive, :n], axis=1, keepdims=True)
    for K in _clusters(lam, 1e-3 * lam[0]):
        mine = [i for i in K if i < nlive]
        if not mine:
            continue
        others = np.setdiff1d(np.arange(len(lam)), K)
        gap = min(np.min(np.abs(sigma[i] ** 2 - lam[others])) for i in mine) if others.size else np.inf
        eps = np.sqrt(len(mine)) * (dC + res_bound + U32 * lam[0])
        if gap <= 2 * eps:
            continue
        sphi = eps / (gap - eps)
        bound = (S[0] / S[max(K)]) * sphi / np.sqrt(max(1e-30, 1 - sphi ** 2)) + 1e-5
        if bound >= 0.5:
            continue
        UK = Us[:, K]
        off = Pn[mine].T - UK @ (UK.T @ Pn[mine].T)
        assert np.linalg.norm(off, 2) <= bound, (kind, K, np.linalg.norm(off, 2), bound)


@pytest.mark.parametrize("r", [4, 14, 16, 32, 64])
@pytest.mark.parametrize("kind", ["cylinder", "channel", "aneurysm", "flat"])
def test_pod_analysis_against_fp64_svd(kind, r):
    X = _e2e_data(kind)
    n, m = X.shape
    Xf, Us, S = _svd(X)
    lam = S ** 2
    e = _engine(X, r, 0)
    sigma = e.pod_analysis().double().cpu().numpy()
    P = e.P.double().cpu().numpy()
    Sdev = e.pod_singular_values.numpy()
    assert e.pod_singular_values.dtype == torch.float64 and Sdev.shape == (m,)
    assert np.isfinite(P).all() and np.all(P[:, n:] == 0)
    assert np.array_equal(sigma, Sdev[:r].astype(np.float32).astype(np.float64))
    assert torch.equal(e.pod_V, e.pod_V) and e.pod_V.shape == (r, m) and e.pod_gram.shape == (m, m)
    Cdev = e.pod_gram.double().cpu().numpy()
    dC = np.linalg.norm(Cdev - Xf.T @ Xf, 2)           # measured ||C_dev - C64||_2
    trace = float(np.trace(Cdev))
    floor = 2.0 ** -23 * trace
    tol = _solver_bound(m, lam[0])
    # Weyl over the full spectrum: |S_i^2 - lambda_i| <= ||C_dev - C64||_2 + the solver's bound (+ the rounding of S^2)
    live_S = Sdev > 0
    assert np.all(np.abs(Sdev[live_S] ** 2 - lam[live_S]) <= dC + tol + 3 * U64 * lam[live_S])
    assert np.all(lam[~live_S] <= floor + dC + tol)
    live = sigma > 0
    weyl = dC + tol + 3 * U32 * lam[:r]
    assert np.all(np.abs(sigma[live] ** 2 - lam[:r][live]) <= weyl[live])
    assert np.all(P[~live] == 0)
    res_bound = EIGH_TOL * lam[0]
    _check_modes(kind, Xf, Us, S, sigma, P, dC, res_bound)
    # POD_analysis' diagnostics
    tot = float(np.sum(lam))
    en = lam[:r] / tot
    tol_e = (weyl + abs(trace - tot)) / tot + 1e-7
    assert np.all(np.abs(e.pod_energy.numpy()[live] - en[live]) <= tol_e[live] + en[live] * 1e-6)
    assert np.allclose(e.pod_cumulative_energy.numpy(), np.cumsum(e.pod_energy.numpy()), rtol=0, atol=1e-12)
    assert abs(e.pod_error ** 2 - max(0.0, 1.0 - float(np.sum(en)))) <= float(np.sum(tol_e)) + 1e-6
    assert set(e.pod_timing) == {"gram_ms", "eig_ms", "project_ms"}
    if r <= 14:
        # the subspace solver's result is within its own bounds (test_pod_reference) of the same references: both within Weyl and
        # Davis-Kahan of the SVD, so within the sum of the two bounds of each other
        P_eigh = P.copy()
        s_sub = e.pod_from_snapshot().double().cpu().numpy()
        P_sub = e.P.double().cpu().numpy()
        assert np.array_equal(s_sub > 0, live)
        assert np.all(np.abs(s_sub[live] ** 2 - sigma[live] ** 2) <= weyl[live] + dC + 2e-8 * lam[0] + 3 * U32 * lam[:r][live])
        _check_modes(kind, Xf, Us, S, s_sub, P_sub, dC, 1e-8 * lam[0])
        assert np.all(P_sub[~live] == 0) and np.all(P_eigh[~live] == 0)


def test_pod_analysis_rank_deficient_floor():
    """The aneurysm field has exact rank 8: at r = 16 the eight null modes come back as sigma = 0 and zero rows of P."""
    X = _e2e_data("aneurysm")
    e = _engine(X, 16, 0)
    sigma = e.pod_analysis().cpu().numpy()
    P = e.P.cpu().numpy()
    assert np.isfinite(P).all()
    assert np.all(sigma[:8] > 0) and np.all(sigma[8:] == 0), sigma
    assert np.all(P[8:] == 0) and np.all(np.linalg.norm(P[:8], axis=1) > 0.5)
    S = e.pod_singular_values.numpy()
    assert np.all(S[:8] > 0) and np.all(S[8:] == 0)
    V = e.pod_V.double().cpu().numpy()
    assert np.abs(V @ V.T - np.eye(16)).max() <= 4 * U32     # floored rows are orthonormal too


# ------------------------------------------------------------------------------------------------ 4. storage, determinism, ops
def test_bf16_storage_equals_fp32_of_rounded():
    from desmo_b200 import DesmoEngine

    X = _e2e_data("channel")
    n, m = X.shape
    Uq = torch.as_tensor(np.ascontiguousarray(X.T), dtype=torch.float32).bfloat16().float()
    out = []
    for dt in (torch.bfloat16, torch.float32):
        e = DesmoEngine(n, m, 2, 32, 10.0, device=torch.device(DEV), snapshot_dtype=dt)
        e.set_snapshot(Uq)
        s = e.pod_analysis()
        out.append((s, e.P.clone(), e.pod_singular_values))
    assert all(torch.equal(a, b) for a, b in zip(*out))


def test_deterministic_and_ops_route():
    from desmo_b200 import ops

    X = _e2e_data("flat")
    e1, e2 = _engine(X, 32, 0), _engine(X, 32, 0)
    s1 = e1.pod_analysis()
    P1, S1 = e1.P.clone(), e1.pod_singular_values.clone()
    s1b = e1.pod_analysis()
    assert torch.equal(s1, s1b) and torch.equal(e1.P, P1) and torch.equal(e1.pod_singular_values, S1)
    s2 = e2.pod_analysis()
    assert torch.equal(s1, s2) and torch.equal(e2.P, P1) and torch.equal(e2.pod_singular_values, S1)
    e2.P.fill_(7.0)
    s3 = ops.engine_pod_analysis_via_ops(e2)
    torch.cuda.synchronize()
    assert torch.equal(s3, s1) and torch.equal(e2.P, P1)


def test_failed_call_leaves_p_untouched(monkeypatch):
    from desmo_b200 import DesmoError

    X = _e2e_data("cylinder")
    e = _engine(X, 32, 0)
    e.P.fill_(3.0)
    before = e.P.clone()
    small = e._eigh_workspace()[:-8]
    monkeypatch.setattr(e, "_eigh_workspace", lambda: small)
    with pytest.raises(DesmoError, match="workspace too small"):
        e.pod_analysis()
    torch.cuda.synchronize()
    assert torch.equal(e.P, before)


def test_workspace_report_and_argument_errors_on_device():
    L = _L()
    Cm = torch.eye(40, device=DEV)
    S, V, sigma, status, reported = _eigh(Cm, 20)
    # C = I: bisection stops within 2 u of lambda = 1, so every residual ||x - lambda x|| is |1 - lambda| <= 2 u
    assert status == 0 and reported <= 2 * U64
    assert np.all(np.abs(S - 1.0) <= 2 * U64) and np.abs(V @ V.T - np.eye(20)).max() <= 4 * U32
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    for r in (0, 41, 65):
        with pytest.raises(L.DesmoError):
            torch.ops.desmo_b200.pod_eigh(Cm, torch.zeros(40, dtype=torch.float64, device=DEV), torch.zeros(max(r, 1), 40, device=DEV),
                                          torch.zeros(max(r, 1), device=DEV), ws, 40, r)


# ------------------------------------------------------------------------------------------------ 5. training from the new modes
def test_train_r32_from_pod_analysis():
    """A DESMO with r = 32 on channel data (K = 657, GEMM path) initialised by pod_analysis() trains 3 steps with finite losses, and its
    first-step loss matches a model initialised from the fp64 SVD modes (signs aligned).  Bound: with r_j = rec_j - U,
    |L_1 - L_2| = |(||r_1||^2 - ||r_2||^2)| / (n m) <= ||rec_1 - rec_2||_F (||r_1|| + ||r_2||) / (n m), evaluated from the two
    models' measured reconstructions before the step (so from the measured distance between the modes), plus the fp32 rounding of
    each loss's sums (1e-5 relative, the gradient gate's level)."""
    from desmo_b200 import DESMO, DesmoTrainer

    X = _e2e_data("channel")
    n, m = X.shape
    Xf, Us, _ = _svd(X)
    snap = torch.as_tensor(np.ascontiguousarray(X.T), dtype=torch.float32)
    dev = torch.device(DEV)
    a = DESMO(n, m, 2, 32, 10.0, device=dev, path=3)
    a.engine.set_snapshot(snap)
    a.engine.pod_analysis()
    Pa = a.engine.P[:, :n].double().cpu().numpy()
    modes = Us[:, :32] * np.sign(np.sum(Us[:, :32] * Pa.T, axis=0))      # align the SVD's arbitrary signs with the device modes
    b = DESMO(n, m, 2, 32, 10.0, pod_modes=modes, device=dev, path=3)
    b.engine.set_snapshot(snap)
    U = snap.double().to(dev)
    rec = [x.engine.reconstruct()[:, :n].double() for x in (a, b)]
    r1, r2 = (rec[0] - U).norm().item(), (rec[1] - U).norm().item()
    bound = (rec[0] - rec[1]).norm().item() * (r1 + r2) / (n * m)
    losses = []
    for x in (a, b):
        tr = DesmoTrainer(x, use_cuda_graph=False)
        ls = []
        for _ in range(3):
            tr.step()
            torch.cuda.synchronize()
            ls.append(float(x.engine.losses[0]))
        losses.append(ls)
    assert np.isfinite(losses).all(), losses
    la, lb = losses[0][0], losses[1][0]
    assert abs(la - lb) <= bound + 1e-5 * max(la, lb), (la, lb, bound)


# ------------------------------------------------------------------------------------------------ 6. two GPUs
def test_sharded_pod_analysis_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29675", os.path.join(ROOT, "tests", "_pod_analysis_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("POD_ANALYSIS_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("POD_ANALYSIS_RESULT "):])
    assert res["V_identical_across_ranks"] and res["sigma_identical_across_ranks"], res
    # the slab Gram sums the same products in another order: the modes agree to the Davis-Kahan level of that fp32 difference
    assert res["mode_sin_vs_unsharded"] <= 1e-4, res
