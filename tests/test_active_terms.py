"""Training on an active set of library terms (DesmoEngine.set_active_terms, desmo_*_active): gradients against the masked fp64
oracle on every path, agreement across paths, a masked trajectory, bit-identities (all-active set, clearing the set, bf16 storage,
graph replay, checkpoint / resume, the ops route), host-side rejection of bad masks, sequential thresholding and a 2-GPU slab run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import desmo_oracle as orc
from tests import _active_oracle as ao
from tests.helpers import engine_params, load_engine, make_case, rel

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRAD_TOL = {"gates": 1e-5, "rows": 1e-5, "coefs": 1e-5, "periods": 5e-5, "phi": 5e-5, "omega": 5e-5}
BETA, LAM = 1e-3, 1e-4


def _engine(prm, modes, snap, path, snapshot_dtype=torch.float32):
    from desmo_b200 import DesmoEngine

    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    e = DesmoEngine(prm.n, prm.m, prm.polyorder, prm.r, nF=prm.nF or None, device=torch.device("cuda:0"), path=path,
                    snapshot_dtype=snapshot_dtype)
    load_engine(e, prm, modes, snap)
    return e


def _masks(T, r, K, seed=0):
    rng = np.random.default_rng(seed)
    deg_top = np.zeros(K, bool)
    from math import comb
    p = next(q for q in range(8) if sum(comb(r + d - 1, d) for d in range(q + 1)) == T)
    deg_top[T - comb(r + p - 1, p):T] = True
    out = {}
    for name, frac in (("rand50", 0.5), ("rand10", 0.1)):
        m = rng.random(K) < frac
        m[rng.integers(K)] = True
        out[name] = m
    out["single"] = np.arange(K) == rng.integers(1, K)
    out["const"] = np.arange(K) == 0
    out["no_top_degree"] = ~deg_top
    triples = np.ones(K, bool)
    for i in range(0, r, 2):  # whole sin / cos / tanh triples of every other mode
        triples[[T + i, T + r + i, T + 2 * r + i]] = False
    out["no_triples"] = triples
    out["trig_only"] = np.arange(K) >= T
    return out


CASES = [  # (id, kind, n, m, r, p, nF, paths)
    ("r2p2", "cylinder", 700, 90, 2, 2, None, (2,)),
    ("r4p2", "channel", 2048, 256, 4, 2, None, (1, 2, 3)),
    ("r4p3", "cylinder", 3961, 201, 4, 3, None, (1, 3)),
    ("r8p2", "cylinder", 1500, 150, 8, 2, None, (1, 3)),
    ("r32p2", "channel", 2048, 200, 32, 2, None, (3,)),
    ("fr2p2", "cylinder", 700, 90, 2, 2, 4, (1, 2, 3)),
    ("fr4p3", "cylinder", 900, 120, 4, 3, 3, (1, 3)),
    # m < 128: one time slab on the FFMA path, whose multi-slab launches add into D with float atomics (not bit-reproducible)
    ("r4p2s", "channel", 2048, 60, 4, 2, None, ()),
    ("r4p3s", "cylinder", 3961, 60, 4, 3, None, ()),
]
MASK_NAMES = ["rand50", "rand10", "single", "const", "no_top_degree", "no_triples", "trig_only"]


def _case(cid):
    c = next(c for c in CASES if c[0] == cid)
    _, modes, snap, prm = make_case(c[1], c[2], c[3], c[4], c[5], c[6], omega_init=2.0, perturb_rel=0.2)
    return c, modes, snap, prm


def _f64(prm):
    q = prm.copy()
    for k, v in q.__dict__.items():
        if isinstance(v, np.ndarray):
            setattr(q, k, v.astype(np.float64))
    return q


def _check_against_oracle(e, prm, modes, snap, mask):
    out = ao.loss_and_grads(_f64(prm), modes, snap.astype(np.float64), BETA, LAM, active=mask)
    fms = ao.frozen_masks(prm, mask)
    g = e.gradients(beta=BETA, l1_lambda=LAM)
    losses = e.losses.cpu().numpy()
    assert abs(losses[0] - out.mse) <= 1e-5 * abs(out.mse)
    assert abs(losses[2] - out.l1) <= 1e-5 * abs(out.l1)
    assert abs(losses[3] - out.total) <= 1e-5 * abs(out.total)
    for k, ref in out.grads.items():
        kk = "rows" if k == "zall" else k
        got = g[kk].cpu().numpy()
        if k in fms:
            assert np.all(got[~fms[k]] == 0.0), k  # frozen: exactly zero
            got, ref = got[fms[k]], ref[fms[k]]
        scale = np.linalg.norm(ref)
        if k == "periods":
            # d period sums cancelling terms over t: its fp32 error is relative to the scale of the whole library's period
            # gradient (what the unmasked golden gate measures), not to one surviving term's
            full = ao.loss_and_grads(_f64(prm), modes, snap.astype(np.float64), BETA, LAM).grads["periods"]
            scale = max(scale, np.linalg.norm(full))
        err = np.linalg.norm(np.asarray(got, np.float64) - ref) / max(scale, 1e-300)
        assert err < GRAD_TOL[kk], (k, err)
    return g


@pytest.mark.parametrize("cid,path,mname", [(c[0], p, mn) for c in CASES for p in c[7] for mn in MASK_NAMES])
def test_gradients_match_masked_oracle(cid, path, mname):
    c, modes, snap, prm = _case(cid)
    mask = _masks(prm.T, prm.r, prm.K)[mname]
    e = _engine(prm, modes, snap, path)
    e.set_active_terms(mask)
    assert e.path_used == path
    _check_against_oracle(e, prm, modes, snap, mask)


@pytest.mark.parametrize("cid,path", [("r4p2", 2), ("r4p3", 3), ("r32p2", 3), ("fr2p2", 3)])
def test_gradients_bf16_storage(cid, path):
    """bf16 storage against the oracle on U_q, the snapshot rounded to bf16."""
    c, modes, snap, prm = _case(cid)
    snap_q = torch.from_numpy(snap).bfloat16().float().numpy()
    mask = _masks(prm.T, prm.r, prm.K)["rand50"]
    e = _engine(prm, modes, snap_q, path, snapshot_dtype=torch.bfloat16)
    e.set_active_terms(mask)
    _check_against_oracle(e, prm, modes, snap_q, mask)


@pytest.mark.parametrize("cid", ["r4p3", "r8p2"])
def test_paths_agree(cid):
    """Masked FFMA path (full library, zero W rows) and masked GEMM path (compacted columns)."""
    c, modes, snap, prm = _case(cid)
    for mname in ("rand50", "no_triples", "trig_only"):
        mask = _masks(prm.T, prm.r, prm.K)[mname]
        gs = []
        for path in (1, 3):
            e = _engine(prm, modes, snap, path)
            e.set_active_terms(mask)
            gs.append((e.gradients(beta=BETA, l1_lambda=LAM), e.losses.cpu().numpy()))
        (g1, l1), (g3, l3) = gs
        assert np.all(np.abs(l1 - l3) <= 1e-5 * np.abs(l1) + 1e-12), (l1, l3)
        for k in g1:
            assert rel(g3[k].cpu().numpy(), g1[k].cpu().numpy()) < GRAD_TOL[k], (mname, k)


def _frozen_state(e, mask):
    m = torch.from_numpy(~mask).to(e.device)
    T, r = e.T, e.r
    q = torch.arange(3 * r, device=e.device)
    om = m[T + (q % 3) * r + q // 3]
    out = {k: getattr(e, k)[m].clone() for k in ("gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u")}
    out.update({k: getattr(e, k)[om].clone() for k in ("omega", "omega_m", "omega_u")})
    return out


@pytest.mark.parametrize("path", [1, 3])
def test_trajectory_matches_masked_oracle(path):
    """20 ordinary steps, then 200 on an active set, at the 1000-step goldens' omega_init = 10, lr_omega = 1e-2 setting."""
    from desmo_b200 import DesmoTrainer

    _, modes, snap, prm = make_case("cylinder", 180, 60, 4, 3, omega_init=10.0, perturb_seed=43, perturb_rel=0.02)
    lrs = (1e-2, 1e-3, 1e-2, 1e-2, 1e-2)
    mask = _masks(prm.T, prm.r, prm.K, seed=3)["rand50"]
    e = _engine(prm, modes, snap, path)
    tr = DesmoTrainer(e, lrs=lrs, beta=BETA, l1_lambda=LAM, patience=5, sched_every=10, use_cuda_graph=False)
    ref = prm.copy()
    _, opt, sch = ao.train(ref, modes, snap, 20, BETA, LAM, patience=5, sched_every=10, lrs=lrs)
    for _ in range(20):
        tr.step()
    e.set_active_terms(mask)
    before = _frozen_state(e, mask)
    ao.train(ref, modes, snap, 200, BETA, LAM, patience=5, sched_every=10, lrs=lrs, active=mask, opt=opt, sch=sch)
    for _ in range(200):
        tr.step()
    torch.cuda.synchronize()
    after = _frozen_state(e, mask)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    got = engine_params(e)
    fms = ao.frozen_masks(prm, mask)
    for k in ("gates", "phi", "omega", "zall"):
        a, b = got[k], getattr(ref, k)
        if k in fms:
            a, b = a[fms[k]], b[fms[k]]
        assert rel(a, b) < 1e-3, (k, rel(a, b))


@pytest.mark.parametrize("cid,path", [("r4p2s", 1), ("r4p2", 2), ("r4p2", 3), ("r8p2", 3), ("fr2p2", 3)])
def test_all_active_set_is_bit_identical_to_no_set(cid, path):
    c, modes, snap, prm = _case(cid)
    ea, eb = _engine(prm, modes, snap, path), _engine(prm, modes, snap, path)
    eb.set_active_terms(np.ones(prm.K, bool))
    for _ in range(20):
        ea.train_step()
        eb.train_step()
    torch.cuda.synchronize()
    for k in ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "omega", "omega_u", "losses", "coefs", "periods"):
        if getattr(ea, k) is not None:
            assert torch.equal(getattr(ea, k), getattr(eb, k)), k


STATE = ("phi", "phi_m", "phi_u", "gates", "gates_m", "gates_u", "rows", "rows_m", "rows_u", "omega", "omega_m", "omega_u", "coefs",
         "coefs_m", "coefs_u", "periods", "periods_m", "periods_u", "step_dev")


@pytest.mark.parametrize("path", [1, 3])
def test_clearing_the_set_resumes_ordinary_training(path):
    c, modes, snap, prm = _case("r4p3s")
    ea, eb = _engine(prm, modes, snap, path), _engine(prm, modes, snap, path)
    ea.set_active_terms(_masks(prm.T, prm.r, prm.K)["rand50"])
    for _ in range(5):
        ea.train_step()
    for k in STATE:
        if getattr(ea, k) is not None:
            getattr(eb, k).copy_(getattr(ea, k))
    ea.set_active_terms(None)
    assert ea.active_terms is None
    ea.train_step()
    eb.train_step()
    torch.cuda.synchronize()
    for k in STATE + ("losses",):
        if getattr(ea, k) is not None:
            assert torch.equal(getattr(ea, k), getattr(eb, k)), k


@pytest.mark.parametrize("cid,path", [("r4p2", 2), ("r4p3s", 1), ("r4p3", 3)])
def test_bf16_storage_equals_fp32_storage_of_uq(cid, path):
    c, modes, snap, prm = _case(cid)
    snap_q = torch.from_numpy(snap).bfloat16()
    mask = _masks(prm.T, prm.r, prm.K)["rand50"]
    e16 = _engine(prm, modes, None, path, snapshot_dtype=torch.bfloat16)
    e32 = _engine(prm, modes, None, path)
    e16.set_snapshot(snap_q)
    e32.set_snapshot(snap_q.float())
    for e in (e16, e32):
        e.set_active_terms(mask)
        for _ in range(5):
            e.train_step()
    torch.cuda.synchronize()
    for k in STATE + ("losses",):
        if getattr(e16, k) is not None:
            assert torch.equal(getattr(e16, k), getattr(e32, k)), k


@pytest.mark.parametrize("path", [2, 3])
def test_graph_replay_equals_eager(path):
    from desmo_b200 import DesmoTrainer

    c, modes, snap, prm = _case("r4p2")
    mask = _masks(prm.T, prm.r, prm.K)["rand50"]
    es = []
    for graph in (False, True):
        e = _engine(prm, modes, snap, path)
        e.set_active_terms(mask)
        tr = DesmoTrainer(e, beta=BETA, l1_lambda=LAM, patience=2, sched_every=3, use_cuda_graph=graph)
        for _ in range(20):
            tr.step()
        es.append(e)
    torch.cuda.synchronize()
    for k in STATE + ("losses", "hyper"):
        if getattr(es[0], k) is not None:
            assert torch.equal(getattr(es[0], k), getattr(es[1], k)), k


def test_graph_is_recaptured_when_the_set_changes():
    from desmo_b200 import DesmoTrainer

    c, modes, snap, prm = _case("r4p3")
    masks = _masks(prm.T, prm.r, prm.K)
    es = []
    for graph in (False, True):
        e = _engine(prm, modes, snap, 3)
        tr = DesmoTrainer(e, beta=BETA, l1_lambda=LAM, sched_every=10 ** 6, use_cuda_graph=graph)
        for mk in ("rand50", None, "rand10"):
            e.set_active_terms(None if mk is None else masks[mk] & (masks["rand50"] if mk == "rand10" else True))
            for _ in range(4):
                tr.step()
        es.append(e)
    torch.cuda.synchronize()
    for k in STATE:
        if getattr(es[0], k) is not None:
            assert torch.equal(getattr(es[0], k), getattr(es[1], k)), k


def test_checkpoint_resume_is_exact():
    from desmo_b200 import DESMO, DesmoTrainer

    c, modes, snap, prm = _case("r4p3")
    mask = _masks(prm.T, prm.r, prm.K)["rand50"]

    def fresh():
        model = DESMO(prm.n, prm.m, prm.polyorder, prm.r, device=torch.device("cuda:0"), path=3)
        load_engine(model.engine, prm, modes, snap)
        return model, DesmoTrainer(model, beta=BETA, l1_lambda=LAM, patience=2, sched_every=5, use_cuda_graph=False)

    ma, ta = fresh()
    ma.set_active_terms(torch.from_numpy(mask))
    for _ in range(10):
        ta.step()
    sd = ta.state_dict()
    assert torch.equal(sd["active_terms"], torch.from_numpy(mask))
    assert all(float(sd["model"][f"{n}.{i}"]) == 0.0 for b, n in enumerate(("sin_coef_list", "cos_coef_list", "tanh_coef_list"))
               for i in range(prm.r) if not mask[prm.T + b * prm.r + i])
    for _ in range(10):
        ta.step()
    mb, tb = fresh()
    tb.load_state_dict(sd)
    assert torch.equal(mb.engine.active_terms, torch.from_numpy(mask))
    for _ in range(10):
        tb.step()
    torch.cuda.synchronize()
    for k in STATE:
        if getattr(ma.engine, k) is not None:
            assert torch.equal(getattr(ma.engine, k), getattr(mb.engine, k)), k


@pytest.mark.parametrize("cid,path", [("r4p2", 2), ("r8p2", 3)])
def test_ops_route_equals_engine(cid, path):
    from desmo_b200 import ops

    c, modes, snap, prm = _case(cid)
    mask = _masks(prm.T, prm.r, prm.K)["rand50"]
    ea, eb = _engine(prm, modes, snap, path), _engine(prm, modes, snap, path)
    for e in (ea, eb):
        e.set_active_terms(mask)
    for _ in range(5):
        ea.train_step()
        ops.engine_step_via_ops(eb)
    torch.cuda.synchronize()
    for k in STATE + ("losses",):
        if getattr(ea, k) is not None:
            assert torch.equal(getattr(ea, k), getattr(eb, k)), k


def test_ops_prepare_and_grads_route():
    """The table made by the active_terms_prepare op drives assemble_grads_active like the engine's gradients()."""
    from desmo_b200 import ops  # noqa: F401

    c, modes, snap, prm = _case("r4p3")
    mask = _masks(prm.T, prm.r, prm.K)["no_triples"]
    e = _engine(prm, modes, snap, 3)
    e.set_active_terms(mask)
    g = e.gradients(beta=BETA, l1_lambda=LAM)
    idx = torch.from_numpy(np.flatnonzero(mask).astype(np.int32))
    table = torch.full_like(e._active, 7)
    sa = (e.n, e.n_global, e.m, e.r, e.polyorder, e.nF, e.shape.path)
    torch.ops.desmo_b200.active_terms_prepare(idx, table, *sa)
    assert torch.equal(table, e._active)
    step = e.step_dev.clone()
    torch.ops.desmo_b200.build_w_active(e.gates, e.rows, e.coefs, e.periods, e.W, step, e.workspace, table, *sa)
    torch.ops.desmo_b200.fused_residual_grad_active(e.U, e.P, e.phi, e.omega, e.W, e.dphi, e.red, e.workspace, table, idx.numel(), *sa)
    f32 = dict(dtype=torch.float32, device=e.device)
    d = {"gates": torch.zeros(e.K, **f32), "rows": torch.zeros(e.K, e.mld, **f32), "omega": torch.zeros(3 * e.r, **f32)}
    dphi = e.dphi.clone()
    hyper = e.hyper.clone()
    hyper[5], hyper[6] = BETA, LAM
    torch.ops.desmo_b200.assemble_grads_active(e.red, dphi, e.P, e.phi, e.gates, e.rows, None, None, hyper, d["gates"], d["rows"], None,
                                               None, d["omega"], torch.zeros(4, **f32), e.workspace, table, *sa)
    torch.cuda.synchronize()
    assert torch.equal(d["gates"], g["gates"]) and torch.equal(d["omega"], g["omega"])
    assert torch.equal(d["rows"][:, :e.m], g["rows"]) and torch.equal(dphi[:, :e.n], g["phi"])


def test_bad_masks_raise_before_anything_is_written():
    from desmo_b200._lib import DesmoError

    c, modes, snap, prm = _case("r4p3")
    e = _engine(prm, modes, snap, 3)
    good = _masks(prm.T, prm.r, prm.K)["rand50"]
    e.set_active_terms(good)
    gates, table = e.gates.clone(), e._active.clone()
    for bad in (np.ones(prm.K - 1, bool), np.ones(prm.K, np.int64), torch.ones(prm.K), np.zeros(prm.K, bool)):
        with pytest.raises(DesmoError):
            e.set_active_terms(bad)
        assert torch.equal(e.gates, gates) and torch.equal(e._active, table)
        assert torch.equal(e.active_terms, torch.from_numpy(good))


def test_sequential_thresholding_matches_oracle_loop():
    from desmo_b200 import DesmoTrainer
    from desmo_b200.sparsify import sequential_thresholding

    _, modes, snap, prm = make_case("cylinder", 700, 90, 4, 2, omega_init=2.0, perturb_rel=0.3)
    prm.gates[::3] *= 1e-3  # a third of the terms far weaker than the rest: a wide gap in the norms
    lrs, every, rounds, epochs = (1e-2, 1e-3, 1e-2, 1e-2, 1e-2), 10, 2, 30
    p64 = _f64(prm)
    norms = np.sort(orc.term_norms(p64))
    # a threshold in the widest gap between adjacent norms (away from both ends), asserted wide so rounding cannot move a term
    ratios = norms[4:-4] / np.maximum(norms[3:-5], 1e-300)
    j = int(np.argmax(ratios)) + 3
    assert ratios[j - 3] > 1.5, ratios
    thr = float(np.sqrt(norms[j] * norms[j + 1]))
    e = _engine(prm, modes, snap, 3)
    tr = DesmoTrainer(e, lrs=lrs, beta=BETA, l1_lambda=LAM, patience=5, sched_every=every, use_cuda_graph=False)
    got = sequential_thresholding(tr, thr, rounds, epochs)
    ref, cur = prm.copy(), np.ones(prm.K, bool)
    opt = sch = None
    total = float(np.sum(snap.astype(np.float64) ** 2))
    want = []
    for _ in range(rounds):
        q = _f64(ref)
        q.gates = q.gates * cur
        nrm = orc.term_norms(q)
        cur = cur & (nrm >= thr) & (q.gates != 0)
        if opt is None:
            opt = orc.Adamax(ref, lrs)
            sch = orc.ReduceLROnPlateau(opt, 5)
        ao.train(ref, modes, snap, epochs, BETA, LAM, patience=5, sched_every=every, lrs=lrs, active=cur, opt=opt, sch=sch)
        o = ao.loss_and_grads(_f64(ref), modes, snap.astype(np.float64), 0.0, 0.0, want_grads=False, active=cur)
        want.append((int(cur.sum()), (o.mse * prm.n * prm.m / total) ** 0.5))
    assert [w[0] for w in got] == [w[0] for w in want], (got, want)
    assert torch.equal(e.active_terms, torch.from_numpy(cur))
    for (_, a), (_, b) in zip(got, want):
        assert abs(a - b) <= 1e-3 * b, (got, want)


def test_sharded_masked_step_matches_unsharded():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one node")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29677", os.path.join(ROOT, "tests", "_active_terms_worker.py")]
    pr = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    line = [ln for ln in pr.stdout.splitlines() if ln.startswith("ACTIVE_RESULT ")]
    assert line, pr.stdout[-3000:]
    res = json.loads(line[-1][len("ACTIVE_RESULT "):])
    assert res["rel_vs_unsharded"] < 1e-4, res
    assert res["identical_across_ranks"] and res["mismatch_raised"], res
