"""POD by the method of snapshots against plain fp64 references, stage by stage and end to end.

A  Gram (desmo_pod_gram_ex): both kernels, fp32 and bf16 storage, edge shapes, entrywise against the Cauchy-Schwarz scale.
B  Eigensolver alone (desmo_pod_eig): fp64 eigh of the device's own C; residuals, Weyl, orthonormality, Davis-Kahan, signs.
C  Projection alone (desmo_pod_project_ex): fp64 U V^T / sigma from fp32-rounded V and sigma; every r up to DESMO_MAX_R.
D  End to end (pod_from_snapshot, torch.ops.desmo_b200.pod_*): np.linalg.svd of the fp64 data.
Every input is seeded; X = A diag(sigma) B^T with A, B from QR lets a case prescribe its spectrum."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import desmo_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEV = "cuda:0"
U32 = 2.0 ** -24          # unit roundoff of fp32 (round to nearest)
EIG_MAX_R = 14


def _lib():
    from desmo_b200 import _lib as L
    from desmo_b200 import ops  # noqa: F401  (registers torch.ops.desmo_b200.*)

    return L


def _shape(n, m, r=2, path=0):
    return _lib().make_shape(n, m, r, 2, 0, n, path)


def _upload(X, dtype=torch.float32):
    """fp64 (n, m) data -> snapshot layout U [m][ld] on the device (pad columns zero)."""
    n, m = X.shape
    ld = _shape(n, m).ld
    U = torch.zeros(m, ld, dtype=torch.float32, device=DEV)
    U[:, :n] = torch.as_tensor(np.ascontiguousarray(X.T), device=DEV).float()
    return U.to(dtype)


def _workspace(n, m, path):
    L = _lib()
    s, nbytes = _shape(n, m, 2, path), C.c_size_t(0)
    L.check(L.load().desmo_workspace_bytes(C.byref(s), C.byref(nbytes)), "desmo_workspace_bytes")
    return torch.zeros(nbytes.value, dtype=torch.uint8, device=DEV)


def _gram(U, n, path):
    m = U.shape[0]
    Cm = torch.full((m, m), float("nan"), device=DEV)
    torch.ops.desmo_b200.pod_gram(U, Cm, _workspace(n, m, path), n, n, m, 2, 2, 0, path)
    return Cm


def _eig(Cm, r):
    m = Cm.shape[0]
    V, sigma = torch.full((r, m), float("nan"), device=DEV), torch.full((r,), float("nan"), device=DEV)
    ws = torch.zeros(2 * 8 * 16 * m + 1024, dtype=torch.uint8, device=DEV)
    torch.ops.desmo_b200.pod_eig(Cm, V, sigma, ws, m, r)
    torch.cuda.synchronize()
    iters, converged = ws[:8].view(torch.int32).tolist()
    return V.double().cpu().numpy(), sigma.double().cpu().numpy(), iters, (converged, float(ws[16:24].view(torch.float64).item()))


def _spectral(n, sig, seed=0):
    """X = A diag(sig) B^T (n x m, fp64, on the host) with orthonormal A (n x m) and B (m x m) from QR of seeded Gaussians."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    m = len(sig)
    A = torch.linalg.qr(torch.randn(n, m, generator=g, device=DEV, dtype=torch.float64))[0]
    B = torch.linalg.qr(torch.randn(m, m, generator=g, device=DEV, dtype=torch.float64))[0]
    return ((A * torch.as_tensor(sig, device=DEV)) @ B.T).cpu().numpy()


def _spectrum(kind, m):
    k = np.arange(m, dtype=np.float64)
    if kind == "separated":
        return 2.0 ** (-k / 2)
    if kind == "geometric":
        return 0.97 ** k
    if kind == "power-0.5":
        return (k + 1) ** -0.5
    if kind == "power-0.15":
        return (k + 1) ** -0.15
    if kind == "pairs":           # travelling waves: sin / cos pairs of equal energy
        return np.repeat(0.8 ** np.arange((m + 1) // 2), 2)[:m]
    if kind == "rank6":           # rank below r
        return np.where(k < 6, 0.8 ** k, 0.0)
    if kind == "range1e6":        # sigma_0 / sigma_{m-1} = 1e6
        return np.logspace(0, -6, m)
    raise ValueError(kind)


SPECTRA = ["separated", "geometric", "power-0.5", "power-0.15", "pairs", "rank6", "range1e6"]


def _clusters(lam, tol):
    """Maximal runs of the descending eigenvalues lam whose neighbours are closer than tol."""
    out, cur = [], [0]
    for i in range(1, len(lam)):
        if lam[i - 1] - lam[i] < tol:
            cur.append(i)
        else:
            out.append(cur)
            cur = [i]
    out.append(cur)
    return out


# ------------------------------------------------------------------------------------------------ A. Gram
def _gram_tau(n, tensor_core):
    """Entrywise bound |C_ij - C64_ij| <= tau sqrt(C64_ii C64_jj).

    Each entry sums n products of fp32 numbers in fp32.  With the rounding errors of the sums modelled as independent and of mean
    zero (round to nearest), |error| <= lam sqrt(d) u sum_x |u_ix u_jx| with probability >= 1 - 2 exp(-lam^2 / 2) for a summation
    depth d <= n + 1 (Higham and Mary, SIAM J. Sci. Comput. 41 (2019) A2815); lam = 8 makes a false failure a 1e-14 event, and
    sum_x |u_ix u_jx| <= sqrt(C_ii C_jj) (Cauchy-Schwarz).  The tensor core truncates when it adds into its fp32 accumulator, which
    is not mean-zero: a chain of at most FLUSH * 24 = 384 MMAs between fp32 round-to-nearest flushes adds at most 2u per MMA,
    768 u in all, as a deterministic term.  The three-plane bf16 split drops products below 2^-32 relative."""
    tau = 8.0 * np.sqrt(n + 1.0) * U32
    return tau + (768.0 * U32 if tensor_core else 0.0)


def _assert_gram(Cm, C64, n, path):
    C64 = torch.as_tensor(C64, device=DEV)
    d = torch.sqrt(torch.clamp(torch.diagonal(C64), min=0.0))
    scale = d[:, None] * d[None, :]
    err = (Cm.double() - C64).abs()
    tau = _gram_tau(n, path != 1)
    bad = err > tau * scale + 1e-300
    assert torch.isfinite(Cm).all()
    assert not bad.any(), (int(bad.sum()), float((err / (scale + 1e-300)).max()), tau)


def _gram_cases():
    out = [(m, n) for m in (2, 17, 127, 128, 129, 1000, 2048, 2049) for n in (1, 63, 65, 129, 4097)]
    return out + [(1000, 1 << 20)]


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("path", [1, 0], ids=["ffma", "tcgen05"])
@pytest.mark.parametrize("m,n", _gram_cases())
def test_gram_entrywise_matches_fp64(m, n, path, dtype):
    """Every entry of C = U U^T against fp64, partial tiles (m % 128 != 0), one-point ranges, the FFMA fallback (m = 2049 on the
    tcgen05 path: more tile pairs than SMs) and, at 2^20 points, many point ranges with pacing and flushes."""
    g = torch.Generator(device=DEV).manual_seed(m * 7919 + n)
    X = torch.randn(m, n, generator=g, device=DEV, dtype=torch.float32) * torch.linspace(0.5, 2.0, m, device=DEV)[:, None]
    ld = _shape(n, m).ld
    U = torch.zeros(m, ld, dtype=torch.float32, device=DEV)
    U[:, :n] = X
    if dtype == "bf16":
        U = U.bfloat16()   # reference: the Gram of U_q in fp64
    Uq = U[:, :n].double()
    C64 = (Uq @ Uq.T).cpu().numpy()
    Cm = _gram(U, n, path)
    torch.cuda.synchronize()
    _assert_gram(Cm, C64, n, path)
    del U, Uq


def test_gram_truncation_bias_at_scale():
    """Nonnegative data at 2^20 x 1000: every product is >= 0, so the tensor core's truncating accumulation shows as a signed mean
    error.  The FFMA Gram (round to nearest) is the yardstick; DESIGN 3.4 records the measured figures."""
    n, m = 1 << 20, 1000
    g = torch.Generator(device=DEV).manual_seed(11)
    ld = _shape(n, m).ld
    U = torch.zeros(m, ld, dtype=torch.float32, device=DEV)
    U[:, :n] = torch.rand(m, n, generator=g, device=DEV)
    Uq = U[:, :n].double()
    C64 = Uq @ Uq.T
    del Uq
    bias = {}
    for path in (1, 0):
        Cm = _gram(U, n, path).double()
        bias[path] = float(((Cm - C64) / C64).mean())
        _assert_gram(Cm.float(), C64.cpu().numpy(), n, path)
    print(f"signed mean relative error: ffma {bias[1]:.3e}, tcgen05 {bias[0]:.3e}")
    # Measured on a B200: ffma -2.9e-6, tcgen05 -4.0e-6.  The truncation adds -1.1e-6 (19 u) to what round-to-nearest gives; the
    # bound leaves room for 32 u, i.e. a chain twice as long as FLUSH = 16 allows.  D's Weyl bound uses the measured ||C - C64||_2.
    assert abs(bias[0] - bias[1]) < 32 * U32, bias


def test_gram_bf16_bit_identical_to_fp32_of_rounded_at_edge_shape():
    """m = 129 (one full and one 1-row tile edge), n = 65 (a 64-point chunk plus one point): the bf16 tcgen05 Gram equals the fp32
    tcgen05 Gram of U_q.float() bit for bit."""
    n, m = 65, 129
    g = torch.Generator(device=DEV).manual_seed(5)
    U = torch.zeros(m, _shape(n, m).ld, device=DEV)
    U[:, :n] = torch.randn(m, n, generator=g, device=DEV)
    Uq = U.bfloat16()
    for path in (1, 0):
        assert torch.equal(_gram(Uq, n, path), _gram(Uq.float(), n, path)), path


@pytest.mark.parametrize("path", [1, 0], ids=["ffma", "tcgen05"])
def test_slab_grams_sum_and_slab_projections_match_columns(path):
    """Point slabs: Gram(slab 1) + Gram(slab 2) = Gram(all) to fp32 reordering; the projection of each slab with the same V and sigma
    equals the matching columns of the full projection bit for bit (a point's sum runs over t in the same order)."""
    n, m, r, cut = 9001, 300, 11, 4133
    X = _spectral(n, _spectrum("geometric", m), seed=3)
    U, U1, U2 = _upload(X), _upload(X[:cut]), _upload(X[cut:])
    Cfull, C1, C2 = _gram(U, n, path), _gram(U1, cut, path), _gram(U2, n - cut, path)
    C64 = X.astype(np.float32).astype(np.float64).T @ X.astype(np.float32).astype(np.float64)
    _assert_gram(C1 + C2, C64, n, path)
    _assert_gram(Cfull, C64, n, path)
    V, sigma, _, ok = _eig(Cfull, r)
    assert ok[0] == 1
    Vd, sd = torch.as_tensor(V, device=DEV).float(), torch.as_tensor(sigma, device=DEV).float()

    def project(Ux, nx):
        s = _shape(nx, m, r, 3)
        P = torch.full((r, s.ld), float("nan"), device=DEV)
        torch.ops.desmo_b200.pod_project(Ux, Vd, sd, P, nx, nx, m, r, 2, 0, 3)
        return P[:, :nx]

    Pf = project(U, n)
    assert torch.equal(torch.cat([project(U1, cut), project(U2, n - cut)], dim=1), Pf)


# ------------------------------------------------------------------------------------------------ B. eigensolver alone
@functools.lru_cache(maxsize=4)
def _device_gram(kind, m):
    X = _spectral(m + 7, _spectrum(kind, m), seed=m)
    Cm = _gram(_upload(X), m + 7, 0)
    C64 = Cm.double().cpu().numpy()
    lam, E = np.linalg.eigh(C64)
    return Cm, C64, lam[::-1].copy(), E[:, ::-1].copy()


def _check_eig(Cm, C64, lam, E, r):
    V, sigma, iters, converged = _eig(Cm, r)
    m = C64.shape[0]
    lam1, trace = lam[0], float(np.trace(C64))
    floor = 2.0 ** -23 * trace
    assert np.isfinite(V).all() and np.isfinite(sigma).all()
    # orthonormal to fp32 rounding: (v + d).(w + e) - v.w <= |d| + |e| + |d||e| with |d|, |e| <= u |v|
    assert np.abs(V @ V.T - np.eye(r)).max() <= 4 * U32 + 1e-12
    # sign convention: the largest-|.| entry of each V_i is positive
    assert all(V[i, np.argmax(np.abs(V[i]))] > 0 for i in range(r))
    live = sigma > 0
    # floor: sigma_i = 0 exactly for the modes at the Gram's rounding level, and only for those
    assert np.all(lam[:r][~live] <= floor * (1 + 1e-6) + 2e-8 * lam1), (lam[:r], sigma)
    assert np.all(lam[:r][live] >= floor * (1 - 1e-6) - 2e-8 * lam1), (lam[:r], sigma)
    if live.any() and not live.all():
        assert np.all(live[:int(live.sum())])     # the floored modes are the trailing ones
    res = np.zeros(r)
    theta = np.zeros(r)
    for i in np.flatnonzero(live):
        v = V[i]
        theta[i] = v @ C64 @ v / (v @ v)
        res[i] = np.linalg.norm(C64 @ v - theta[i] * v) / np.linalg.norm(v)
        # Ritz residual: 1e-8 lambda_1 of solver error plus the fp32 rounding of v, ||(C - theta) dv|| <= lambda_1 u ||v||
        assert res[i] <= 1e-8 * lam1 + U32 * lam1, (i, res[i] / lam1, iters)
        # Weyl: |sigma_i^2 - lambda_i| <= 2e-8 lambda_1 plus the fp32 rounding of sigma (2u sigma^2 + u^2 sigma^2)
        assert abs(sigma[i] ** 2 - lam[i]) <= 2e-8 * lam1 + 3 * U32 * lam[i], (i, sigma[i] ** 2, lam[i])
    # Davis-Kahan: a mode with a relative gap is within res / gap of its eigenvector; a cluster of (near-)equal eigenvalues is compared
    # as a subspace, ||(I - E E^T) V_K^T||_2 <= ||R_K||_F / gap_K (+ the fp32 rounding of V)
    nlive = int(live.sum())
    for K in _clusters(lam, 1e-6 * lam1):
        mine = [i for i in K if i < nlive]
        if not mine:
            continue
        others = np.array([j for j in range(m) if j not in K])
        if others.size == 0:
            continue
        gap = min(np.min(np.abs(theta[i] - lam[others])) for i in mine)
        bound = np.linalg.norm(res[mine]) / gap + 2 * U32 * np.sqrt(len(mine))
        if bound >= 0.5:
            continue
        EK = E[:, K]
        VK = V[mine].T / np.linalg.norm(V[mine], axis=1)
        off = VK - EK @ (EK.T @ VK)
        assert np.linalg.norm(off, 2) <= bound, (K, np.linalg.norm(off, 2), bound)
    assert converged[0] == 1, (iters, converged)
    return iters


@pytest.mark.parametrize("m", [10, 17, 200, 1000, 2100])
@pytest.mark.parametrize("kind", SPECTRA)
def test_eig_against_fp64_eigh_of_device_gram(kind, m):
    Cm, C64, lam, E = _device_gram(kind, m)
    for r in (1, 2, 4, 8, 9, 13, 14):
        if r <= m:
            _check_eig(Cm, C64, lam, E, r)


@pytest.mark.parametrize("kind", ["geometric", "pairs", "range1e6"])
@pytest.mark.parametrize("r", [1, 2, 4, 8, 9, 13, 14])
def test_eig_block_wider_than_m(kind, r):
    """m = r + 1: the block is b = min(r + 8, 16, m) = m vectors, i.e. the whole space (refused before, although well defined)."""
    m = r + 1
    X = _spectral(m + 7, _spectrum(kind, m), seed=r)
    Cm = _gram(_upload(X), m + 7, 0)
    C64 = Cm.double().cpu().numpy()
    lam, E = np.linalg.eigh(C64)
    _check_eig(Cm, C64, lam[::-1].copy(), E[:, ::-1].copy(), r)


def test_eig_refuses_r_above_limit():
    Cm = torch.eye(40, device=DEV)
    with pytest.raises(_lib().DesmoError, match="r <= 14"):
        _eig(Cm, EIG_MAX_R + 1)


# ------------------------------------------------------------------------------------------------ C. projection alone
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("n,m", [(30011, 200), (5003, 1000)])
@pytest.mark.parametrize("r", [1, 7, 8, 9, 14, 16, 32, 64])
def test_projection_every_r_against_fp64(r, n, m, dtype):
    """P_i = U^T V_i / sigma_i for every mode, including those past the first group of eight; pad columns exactly 0."""
    rng = np.random.default_rng(r * 1000 + m)
    X = rng.standard_normal((n, m))
    U = _upload(X, torch.bfloat16 if dtype == "bf16" else torch.float32)
    V = np.ascontiguousarray(np.linalg.qr(rng.standard_normal((m, r)))[0].T, dtype=np.float32)
    sigma = np.sort(rng.uniform(0.5, 50.0, r))[::-1].astype(np.float32)
    s = _shape(n, m, r, 3)
    P = torch.full((r, s.ld), float("nan"), device=DEV)
    torch.ops.desmo_b200.pod_project(U, torch.as_tensor(V, device=DEV), torch.as_tensor(sigma, device=DEV), P, n, n, m, r, 2, 0, 3)
    Pn = P.double().cpu().numpy()
    Uq = U[:, :n].double().cpu().numpy()           # what the kernel reads (U_q for bf16)
    V64, s64 = V.astype(np.float64), sigma.astype(np.float64)
    ref = (V64 @ Uq) / s64[:, None]
    # m fused multiply-adds in fp32, then one product with the rounded 1 / sigma: |error| <= (m + 2) u (|V| |U|)_ix / sigma_i
    bound = (m + 2) * U32 * (np.abs(V64) @ np.abs(Uq)) / s64[:, None]
    assert np.all(np.abs(Pn[:, :n] - ref) <= bound), [float(np.max(np.abs(Pn[i, :n] - ref[i]) / bound[i].max())) for i in range(r)]
    rel_row = np.linalg.norm(Pn[:, :n] - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert rel_row.max() < 1e-5, rel_row
    assert np.all(Pn[:, n:] == 0.0)


def test_projection_zero_sigma_gives_zero_row():
    n, m, r = 1000, 50, 10
    rng = np.random.default_rng(0)
    U = _upload(rng.standard_normal((n, m)))
    V = torch.as_tensor(np.ascontiguousarray(np.linalg.qr(rng.standard_normal((m, r)))[0].T, dtype=np.float32), device=DEV)
    sigma = torch.tensor([3.0] * 8 + [0.0, 0.0], device=DEV)
    P = torch.full((r, _shape(n, m, r, 3).ld), float("nan"), device=DEV)
    torch.ops.desmo_b200.pod_project(U, V, sigma, P, n, n, m, r, 2, 0, 3)
    assert torch.isfinite(P).all()
    assert torch.all(P[8:] == 0) and torch.all(P[:8, :n] != 0)


# ------------------------------------------------------------------------------------------------ D. end to end
def _e2e_data(kind):
    if kind == "flat":
        return _spectral(6000, _spectrum("power-0.15", 300), seed=17)
    n, m = {"cylinder": (3000, 200), "channel": (4096, 240), "aneurysm": (4000, 300)}[kind]
    return orc.synthetic_snapshots(kind, n, m, 0)


def _engine(X, r, path):
    from desmo_b200 import DesmoEngine

    n, m = X.shape
    e = DesmoEngine(n, m, 2, r, 10.0, device=torch.device(DEV), path=path)
    e.set_snapshot(torch.as_tensor(np.ascontiguousarray(X.T), dtype=torch.float32))
    return e


@pytest.mark.parametrize("r", [4, 8, 9, 12, 14])
@pytest.mark.parametrize("kind", ["cylinder", "channel", "aneurysm", "flat"])
def test_pod_from_snapshot_against_fp64_svd(kind, r):
    X = _e2e_data(kind)
    n, m = X.shape
    Xf = X.astype(np.float32).astype(np.float64)      # what U holds
    Us, S, _ = np.linalg.svd(Xf, full_matrices=False)
    lam = S ** 2
    e = _engine(X, r, 0)
    sigma = e.pod_from_snapshot().double().cpu().numpy()
    P = e.P.double().cpu().numpy()
    assert np.isfinite(P).all() and np.isfinite(sigma).all()
    assert np.all(P[:, n:] == 0)
    Cdev = e.pod_gram.double().cpu().numpy()
    dC = np.linalg.norm(Cdev - Xf.T @ Xf, 2)          # measured ||C_dev - C64||_2
    trace = float(np.trace(Cdev))
    floor = 2.0 ** -23 * trace
    live = sigma > 0
    nlive = int(live.sum())
    assert np.all(live[:nlive]) and np.all(lam[:r][~live] <= floor + dC)
    # Weyl: |sigma_i^2 - S_i^2| <= ||C_dev - C64||_2 + the solver's residual bound + fp32 rounding of sigma
    weyl = dC + 2e-8 * lam[0] + 3 * U32 * lam[:r]
    assert np.all(np.abs(sigma[live] ** 2 - lam[:r][live]) <= weyl[live]), (sigma[live] ** 2 - lam[:r][live], weyl)
    # floored modes: zero rows of P
    assert np.all(P[~live] == 0)
    # Davis-Kahan per mode / cluster: v_i is an eigenvector of C64 up to ||C_dev - C64|| + residual, and P_i = X v_i / sigma_i
    # turns an angle phi of v_i into at most (S_0 / S_i) tan(phi) in the mode
    Pn = P[:nlive, :n] / np.linalg.norm(P[:nlive, :n], axis=1, keepdims=True)
    for K in _clusters(lam, 1e-3 * lam[0]):
        mine = [i for i in K if i < nlive]
        if not mine:
            continue
        others = [j for j in range(len(lam)) if j not in K]
        gap = min(np.min(np.abs(sigma[i] ** 2 - lam[others])) for i in mine) if others else np.inf
        eps = np.sqrt(len(mine)) * (dC + 1e-8 * lam[0] + U32 * lam[0])
        if gap <= 2 * eps:
            continue
        sphi = eps / (gap - eps)
        bound = (S[0] / S[max(K)]) * sphi / np.sqrt(max(1e-30, 1 - sphi ** 2)) + 1e-5
        if bound >= 0.5:
            continue
        UK = Us[:, K]
        off = Pn[mine].T - UK @ (UK.T @ Pn[mine].T)
        assert np.linalg.norm(off, 2) <= bound, (kind, r, K, np.linalg.norm(off, 2), bound)
    # POD_analysis' diagnostics agree with the SVD's
    tot = float(np.sum(lam))
    en = lam[:r] / tot
    en_dev = e.pod_energy.numpy()
    tol_e = (weyl + abs(trace - tot)) / tot + 1e-7
    assert np.all(np.abs(en_dev[live] - en[live]) <= tol_e[live] + en[live] * 1e-6)
    assert np.allclose(e.pod_cumulative_energy.numpy(), np.cumsum(en_dev), rtol=0, atol=1e-12)
    err_ref2 = max(0.0, 1.0 - float(np.sum(en)))
    assert abs(e.pod_error ** 2 - err_ref2) <= float(np.sum(tol_e)) + 1e-6
    # the same result through the registered ops
    from desmo_b200 import ops

    P1, s1 = e.P.clone(), e.pod_from_snapshot()
    e.P.fill_(7.0)
    ops.engine_pod_via_ops(e)
    torch.cuda.synchronize()
    assert torch.equal(e.P, P1) and torch.equal(s1, torch.as_tensor(sigma, dtype=torch.float32, device=DEV))


def test_pod_rank_deficient_floor():
    """The aneurysm field has exact rank 8: at r = 12 the four null modes come back as sigma = 0 and zero rows of P, the rest
    finite -- through the engine and through the registered ops."""
    from desmo_b200 import ops

    X = _e2e_data("aneurysm")
    e = _engine(X, 12, 0)
    sigma = e.pod_from_snapshot().cpu().numpy()
    P = e.P.cpu().numpy()
    assert np.isfinite(P).all()
    assert np.all(sigma[:8] > 0) and np.all(sigma[8:] == 0), sigma
    assert np.all(P[8:] == 0) and np.all(np.linalg.norm(P[:8], axis=1) > 0.5)
    e.P.fill_(float("nan"))
    ops.engine_pod_via_ops(e)
    torch.cuda.synchronize()
    assert torch.equal(e.P.cpu(), torch.as_tensor(P))


def test_pod_r_above_limit_raises_and_leaves_p():
    from desmo_b200 import DesmoError

    X = _e2e_data("cylinder")
    e = _engine(X, EIG_MAX_R + 1, 0)
    e.P.fill_(3.0)
    before = e.P.clone()
    with pytest.raises(DesmoError, match="r <= 14"):
        e.pod_from_snapshot()
    torch.cuda.synchronize()
    assert torch.equal(e.P, before)
