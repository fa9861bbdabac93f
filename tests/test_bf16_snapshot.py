"""bf16 storage of the snapshot matrix U (DesmoEngine(snapshot_dtype=torch.bfloat16)).

Contract: U_q = bf16_rn(U) is stored; every kernel widens it exactly to fp32, so each result is BIT-IDENTICAL to the fp32-storage
path fed U_q.float() -- one step (red, dphi, losses, gradients), graph-replayed training, the split pass, point slabs, POD, the
sparsification sweeps.  The quantisation error ||U - U_q|| / ||U|| is reported in fp64."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

from oracle import desmo_oracle as orc
from tests.helpers import GOLDEN, engine_params, golden_case, load_engine, make_case, rel

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from tests.test_gpu_parity import GRAD_TOL, PATHS, _covered, _golden_pairs  # noqa: E402

DEV = "cuda:0"
BF16 = torch.bfloat16


def _pair(prm, modes, snap, path, **kw):
    """(bf16-storage engine fed snap, fp32-storage engine fed U_q.float()) with identical parameters."""
    from desmo_b200 import DesmoEngine

    if not _covered(path, prm.K, prm.r, prm.m):
        pytest.skip("shape outside this path's coverage")
    mk = lambda dt: DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device(DEV), path=path,  # noqa: E731
                                snapshot_dtype=dt, **kw)
    e16, e32 = mk(BF16), mk(torch.float32)
    load_engine(e16, prm, modes, snap)
    load_engine(e32, prm, modes, torch.from_numpy(snap).bfloat16().float().numpy())
    assert e16.U.dtype == BF16 and e32.U.dtype == torch.float32
    return e16, e32


def _assert_step_equal(a, b):
    torch.cuda.synchronize()
    assert torch.equal(a.red, b.red)
    assert torch.equal(a.dphi, b.dphi)
    assert torch.equal(a.losses, b.losses)


# ------------------------------------------------------------------------------------------------ conversion
def test_conversion_equals_torch_bfloat16_bit_for_bit(monkeypatch):
    import desmo_b200.engine as eng
    from desmo_b200 import DesmoEngine

    n, m = 1000, 37
    g = torch.Generator().manual_seed(3)
    U = torch.randn(m, n, generator=g) * torch.logspace(-30, 30, n)[None, :]
    one = 1.0 + 2.0 ** -8  # exactly halfway between two bf16 values: ties go to even
    specials = torch.tensor([one, 1.0 + 3 * 2.0 ** -8, -one, 2.0 ** -130, -(2.0 ** -140), 1.4e-45, 0.0, -0.0, float("inf"), -float("inf"),
                             3.4028235e38, -3.3e38, 1.0e38, 65504.0, 2.0 ** -126, 2.0 ** -127 * 3], dtype=torch.float32)
    U[5, :specials.numel()] = specials
    U[36, -specials.numel():] = specials
    monkeypatch.setattr(eng, "SNAPSHOT_CHUNK_BYTES", 4 * n * 5)  # 5-row chunks: 8 conversion launches, the last one ragged
    e = DesmoEngine(n, m, 2, 2, device=DEV, path=1, snapshot_dtype=BF16)
    e.set_snapshot(U)
    want = U.bfloat16()
    got = e.U[:, :n].cpu()
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
    assert int(e.U[:, n:].view(torch.int16).abs().max()) == 0  # pad columns: +0
    # fp64 and device inputs take the same rounding (fp64 is cast to fp32 first, exactly what the fp32 path stores)
    e.set_snapshot(U.double().to(DEV))
    assert torch.equal(e.U[:, :n].cpu().view(torch.int16), want.view(torch.int16))


def test_quantization_sums_match_fp64_torch():
    from desmo_b200 import DesmoEngine
    import desmo_b200.ops  # noqa: F401  (registers the ops)

    n, m = 3000, 130
    g = torch.Generator().manual_seed(5)
    U = torch.randn(m, n, generator=g) * 7.0
    e = DesmoEngine(n, m, 2, 2, device=DEV, path=1, snapshot_dtype=BF16)
    e.set_snapshot(U)
    Ud, Uq = U.double(), U.bfloat16().double()
    e2, u2 = float(((Ud - Uq) ** 2).sum()), float((Ud ** 2).sum())
    q = e._qsums.cpu().numpy()
    assert abs(q[0] - e2) <= 1e-12 * e2 and abs(q[1] - u2) <= 1e-12 * u2
    err = e.snapshot_quantization_error()
    assert abs(err - (e2 / u2) ** 0.5) <= 1e-12 * err
    assert 1e-4 < err < 1e-2  # bf16 round-to-nearest: ~2^-9 relative per element
    # reproducible: the same conversion gives the same bits of the sums
    e.set_snapshot(U)
    assert np.array_equal(e._qsums.cpu().numpy(), q)
    # the op, on rows t0.. of a bf16 U
    Ub = torch.zeros(m, e.ld, dtype=BF16, device=DEV)
    qs = torch.zeros(2, dtype=torch.float64, device=DEV)
    src = U[40:90].to(DEV)
    torch.ops.desmo_b200.snapshot_to_bf16(src, Ub, qs, 40, n, n, m, 2, 2, 0, 1)
    assert torch.equal(Ub[40:90, :n].cpu().view(torch.int16), U[40:90].bfloat16().view(torch.int16))
    assert float(Ub[:40].float().abs().max()) == 0.0 and float(Ub[90:].float().abs().max()) == 0.0
    assert abs(float(qs[1]) - float((U[40:90].double() ** 2).sum())) <= 1e-12 * float(qs[1])


# ------------------------------------------------------------------------------------------------ one step, every path
GRAD_PAIRS = _golden_pairs([os.path.basename(p)[:-4] for p in sorted(glob.glob(os.path.join(GOLDEN, "grad_*.npz")))])


@pytest.mark.parametrize("name,path", GRAD_PAIRS)
def test_step_is_bit_identical_to_fp32_storage_of_uq(name, path):
    fx, meta, modes, snap, prm = golden_case(name)
    e16, e32 = _pair(prm, modes, snap, path)
    beta, lam = meta["beta"], meta["l1_lambda"]
    g16, g32 = e16.gradients(beta=beta, l1_lambda=lam), e32.gradients(beta=beta, l1_lambda=lam)
    _assert_step_equal(e16, e32)
    for k in g32:
        assert torch.equal(g16[k], g32[k]), k
    # against the fp64 oracle evaluated on U_q, at the gates of the fp32 path
    snap_q = torch.from_numpy(snap).bfloat16().float().numpy()
    o = orc.loss_and_grads(prm, modes, snap_q, beta, lam)
    losses = e16.losses.cpu().numpy()
    assert abs(losses[0] - o.mse) <= 1e-5 * abs(o.mse)
    assert abs(losses[3] - o.total) <= 1e-5 * abs(o.total)
    for k, ref in o.grads.items():
        kk = "rows" if k == "zall" else k
        assert rel(g16[kk].cpu().numpy(), ref) < GRAD_TOL[kk], (k, rel(g16[kk].cpu().numpy(), ref))


@pytest.mark.parametrize("path", PATHS)
def test_graph_replayed_training_is_bit_identical(path):
    """20 DesmoTrainer steps (CUDA-graph replay, device scheduler): every parameter and every Adamax moment bit-equal."""
    from desmo_b200 import DesmoTrainer

    fx, meta, modes, snap, prm = golden_case("traj_chan_r4p2")
    e16, e32 = _pair(prm, modes, snap, path)
    for e in (e16, e32):
        tr = DesmoTrainer(e, lrs=meta["lrs"], beta=meta["beta"], l1_lambda=meta["l1_lambda"], patience=2, sched_every=3,
                          use_cuda_graph=True, device_scheduler=True)
        for _ in range(20):
            tr.step()
    torch.cuda.synchronize()
    for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "omega", "omega_m", "omega_u",
              "hyper", "step_dev", "losses"):
        assert torch.equal(getattr(e16, k), getattr(e32, k)), k


@pytest.mark.parametrize("path", PATHS)
def test_split_pass_equals_monolithic_bf16(path):
    from desmo_b200 import _lib

    _, modes, snap, prm = make_case("channel", 1500, 120, 4, 2)
    e, _ = _pair(prm, modes, snap, path)
    e.build_w(False)
    e.fused_residual_grad()
    torch.cuda.synchronize()
    want_red, want_dphi = e.red.clone(), e.dphi.clone()
    ecount = e.Kp * e.mld
    e.red.fill_(7.0)
    e.dphi.fill_(7.0)
    args = (C.byref(e.shape), e.U.data_ptr(), _lib.DTYPE_BF16, e.P.data_ptr(), e.phi.data_ptr(), e.omega.data_ptr(), e.W.data_ptr(),
            e.dphi.data_ptr(), e.red.data_ptr(), e.workspace.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(e.lib.desmo_fused_residual_grad_begin_ex(*args), "begin")
    torch.cuda.synchronize()
    assert torch.equal(e.red[:ecount], want_red[:ecount])
    _lib.check(e.lib.desmo_fused_residual_grad_finish_ex(*args), "finish")
    torch.cuda.synchronize()
    assert torch.equal(e.red, want_red) and torch.equal(e.dphi, want_dphi)


def test_point_slabs_sum_to_the_unsharded_bf16_step():
    from desmo_b200 import DesmoEngine

    _, modes, snap, prm = make_case("channel", 1500, 120, 4, 2)
    full, _ = _pair(prm, modes, snap, 1)
    full.build_w(False)
    full.fused_residual_grad()
    reds, dphis = [], []
    for lo, hi in ((0, 700), (700, prm.n)):
        q = prm.copy()
        q.n, q.phi = hi - lo, prm.phi[:, lo:hi].copy()
        e = DesmoEngine(hi - lo, prm.m, prm.polyorder, prm.r, device=torch.device(DEV), n_global=prm.n, path=1, snapshot_dtype=BF16)
        load_engine(e, q, modes[lo:hi], np.ascontiguousarray(snap[:, lo:hi]))
        e.build_w(False)
        e.fused_residual_grad()
        reds.append(e.red.clone())
        dphis.append(e.dphi[:, :hi - lo].clone())
    assert rel((reds[0] + reds[1]).cpu().numpy(), full.red.cpu().numpy()) < 2e-6
    assert rel(torch.cat(dphis, dim=1).cpu().numpy(), full.dphi[:, :prm.n].cpu().numpy()) < 2e-6


# ------------------------------------------------------------------------------------------------ POD, preprocessing, sweeps
@pytest.mark.parametrize("path", [1, 0], ids=["ffma-gram", "tcgen05-gram"])
def test_pod_bf16_matches_fp32_storage_and_svd(path):
    X, modes, snap, prm = make_case("cylinder", 3000, 200, 4, 2)
    e16, e32 = _pair(prm, modes, snap, path)
    s16, s32 = e16.pod_from_snapshot(), e32.pod_from_snapshot()
    torch.cuda.synchronize()
    # the tcgen05 bf16 Gram skips the fp32 kernel's MMAs whose plane-2/3 operands are exactly zero for such data
    assert torch.equal(e16.pod_gram, e32.pod_gram)
    assert torch.equal(s16, s32) and torch.equal(e16.P, e32.P)
    Xq = torch.from_numpy(snap).bfloat16().double().numpy().T  # (n, m): the data matrix the bf16 storage holds
    S = np.linalg.svd(Xq, compute_uv=False)
    assert rel(s16.cpu().numpy(), S[:4]) < 1e-4
    assert rel(e16.pod_gram.cpu().numpy(), Xq.T @ Xq) < 1e-5
    U_, S_, Vt_ = np.linalg.svd(Xq, full_matrices=False)
    P = e16.P[:, :prm.n].cpu().numpy().astype(np.float64)
    for i in range(4):
        assert abs(float(P[i] @ U_[:, i])) > 1 - 1e-4, i
    assert np.allclose(P @ P.T, np.eye(4), atol=1e-4)
    err_ref = np.linalg.norm(Xq - U_[:, :4] @ np.diag(S_[:4]) @ Vt_[:4]) / np.linalg.norm(Xq)
    assert abs(e16.pod_error - err_ref) < 1e-3 * err_ref + 1e-5
    assert rel(e16.pod_energy.numpy(), (S_ ** 2 / np.sum(S_ ** 2))[:4]) < 1e-4


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("name,cfg", [("cyl", (3, 2, True, False, 1)), ("aneu", (3, 3, True, True, 1)), ("turb", (3, 3, True, False, 2)),
                                      ("vec", (1, 1, False, False, 1))])
def test_bf16_preprocess_equals_fp32_preprocess_then_bfloat16(name, cfg, dtype):
    from desmo_b200 import DesmoEngine

    d_in, d_use, mag, scale, stride = cfg
    fx = np.load(os.path.join(GOLDEN, "preprocess.npz"))
    m, n = fx[name + "_X"].T.shape
    raw = torch.from_numpy(np.ascontiguousarray(fx[name + "_raw"].T)).to(DEV, getattr(torch, dtype))
    out = {}
    for dt in (torch.float32, BF16):
        e = DesmoEngine(n, m, 2, 2, device=DEV, path=1, snapshot_dtype=dt)
        mean = e.preprocess_snapshot(raw, d_in=d_in, d_use=d_use, magnitude=mag, scale_sqrt_m=scale, t_stride=stride)
        out[dt] = (e, mean)
    e32, e16 = out[torch.float32][0], out[BF16][0]
    assert e16.U.dtype == BF16
    assert torch.equal(e16.U.view(torch.int16), e32.U.bfloat16().view(torch.int16))  # pad columns included
    assert torch.equal(out[torch.float32][1], out[BF16][1])
    Ud, Uq = e32.U[:, :n].double(), e16.U[:, :n].double()
    err = float(torch.sqrt(((Ud - Uq) ** 2).sum() / (Ud ** 2).sum()))
    assert abs(e16.snapshot_quantization_error() - err) <= 1e-12 * err + 1e-300


@pytest.mark.parametrize("path", PATHS)
def test_sweeps_identical_between_storages(path):
    from desmo_b200 import DESMO
    from desmo_b200.sparsify import greedy_removal, threshold_sweep

    _, modes, snap, prm = make_case("channel", 700, 72, 4, 2, omega_init=10.0, perturb_rel=0.3)
    snap_q = torch.from_numpy(snap).bfloat16()
    norm2 = float((snap_q.double() ** 2).sum())
    res = []
    for dt, s in ((BF16, snap), (torch.float32, snap_q.float().numpy())):
        model = DESMO(prm.n, prm.m, 2, 4, 10.0, pod_modes=modes, device=torch.device(DEV), path=path, snapshot_dtype=dt)
        load_engine(model.engine, prm, modes, s)
        res.append((threshold_sweep(model, norm2), greedy_removal(model, norm2)))
    (ts16, gr16), (ts32, gr32) = res
    assert gr16 == gr32
    for a, b in zip(ts16, ts32):
        assert a[:3] == b[:3] and torch.equal(a[3], b[3])


# ------------------------------------------------------------------------------------------------ scale, memory, rejection
@pytest.mark.parametrize("path", PATHS)
def test_headline_size_step_is_bit_identical(path):
    from desmo_b200 import DesmoEngine

    n, m = 1 << 18, 1000
    dev = torch.device(DEV)
    g = torch.Generator(device=dev).manual_seed(0)
    P = torch.randn(4, n, device=dev, generator=g) / n ** 0.5
    rows = torch.randn(27, m, device=dev, generator=g)
    U = torch.randn(m, n, device=dev, generator=g)
    es = []
    for dt, src in ((BF16, U), (torch.float32, U.bfloat16().float())):
        e = DesmoEngine(n, m, 2, 4, omega_init=10.0, device=dev, path=path, snapshot_dtype=dt)
        e.P[:, :n] = P
        e.rows[:, :m] = rows
        e.set_snapshot(src)
        e.build_w(False)
        e.fused_residual_grad()
        es.append(e)
    _assert_step_equal(*es)


def test_set_snapshot_holds_no_fp32_copy_of_the_matrix():
    import desmo_b200.engine as eng
    from desmo_b200 import DesmoEngine

    n, m = 1 << 20, 1000
    U = torch.randn(m, n)  # 4 GB on the host
    e = DesmoEngine(n, m, 2, 4, device=DEV, path=0, snapshot_dtype=BF16)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.max_memory_allocated()
    e.set_snapshot(U)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown <= 2 * m * e.ld + eng.SNAPSHOT_CHUNK_BYTES + (2 << 20), grown
    assert torch.equal(e.U[-3:, :n].cpu().view(torch.int16), U[-3:].bfloat16().view(torch.int16))


def test_other_dtypes_are_rejected():
    import desmo_b200.ops as ops
    from desmo_b200 import DesmoEngine, _lib

    with pytest.raises(_lib.DesmoError):
        DesmoEngine(300, 40, 2, 2, device=DEV, snapshot_dtype=torch.float16)
    _, modes, snap, prm = make_case("aneurysm", 1000, 100, 4, 2, omega_init=10.0)
    e16, _ = _pair(prm, modes, snap, 0)
    sa = ops._shape_args(e16)
    for dt in (torch.float16, torch.float64):
        e16.U = torch.zeros(e16.m, e16.ld, dtype=dt, device=DEV)
        for call in (e16.residual_norm2, e16.train_step, e16.pod_from_snapshot):
            with pytest.raises(_lib.DesmoError):
                call()
        with pytest.raises(_lib.DesmoError):
            torch.ops.desmo_b200.fused_residual_grad(e16.U, e16.P, e16.phi, e16.omega, e16.W, e16.dphi, e16.red, e16.workspace, *sa)
        with pytest.raises(_lib.DesmoError):
            torch.ops.desmo_b200.pod_gram(e16.U, torch.zeros(e16.m, e16.m, device=DEV), e16.workspace, *sa)
        with pytest.raises(_lib.DesmoError):
            torch.ops.desmo_b200.pod_project(e16.U, torch.zeros(e16.r, e16.m, device=DEV), torch.ones(e16.r, device=DEV), e16.P, *sa)
        raw = torch.zeros(e16.m, e16.n, device=DEV)
        with pytest.raises(_lib.DesmoError):
            torch.ops.desmo_b200.preprocess(raw, e16.U, None, e16.m, 1, 1, 1, 0, *sa)
    # the C ABI rejects an unknown u_dtype by itself
    rc = e16.lib.desmo_fused_residual_grad_ex(C.byref(e16.shape), e16.U.data_ptr(), 7, e16.P.data_ptr(), e16.phi.data_ptr(),
                                              e16.omega.data_ptr(), e16.W.data_ptr(), e16.dphi.data_ptr(), e16.red.data_ptr(),
                                              e16.workspace.data_ptr(), 0)
    assert rc == 1 and b"u_dtype" in e16.lib.desmo_last_error()


def test_module_surface_takes_snapshot_dtype():
    from desmo_b200 import DESMO, DESMOFourier

    _, modes, snap, prm = make_case("channel", 300, 150, 4, 2, omega_init=10.0)
    m = DESMO(prm.n, prm.m, 2, 4, 10.0, pod_modes=modes, device=torch.device(DEV), snapshot_dtype=BF16)
    loss = m.mse_loss(torch.from_numpy(snap))
    assert m.engine.U.dtype == BF16 and torch.isfinite(loss)
    f = DESMOFourier(prm.n, prm.m, 2, 4, 10.0, 3, pod_modes=modes, device=torch.device(DEV), snapshot_dtype=BF16)
    assert f.engine.snapshot_dtype == BF16
    assert engine_params(m.engine)["phi"].shape == (4, prm.n)
