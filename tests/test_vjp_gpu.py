"""copra_b200_lmpc_vjp (K8) on the GPU: against the dense numpy adjoint reference, against central differences of the GPU
forward, its edge cases, the sharded form and torch.autograd."""
import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import vjp_reference as vr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = capi.Engine(0)
    yield e
    e.close()


def _cotangents(B, s, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(B, s["nU"])), rng.normal(size=(B, s["X"]))


def _dot(g, inst_delta, b):
    """<VJP of instance b, delta> over every input of `inst_delta`"""
    val = 0.0
    for (kind, i), d in inst_delta.items():
        grad = g["x0"][b] if kind == "x0" else g[kind][i][b]
        val += float(grad @ d)
    return val


def _batch_vectors(bp, key, B):
    kind, i = key
    v = np.asarray(bp["x0"] if kind == "x0" else (bp["costs"] if kind == "p" else bp["constraints"])[i][kind], float)
    return np.broadcast_to(v, (B,) + v.shape[-1:]).copy() if v.ndim == 1 else v.copy()


REF = [("c2", lambda: wl.c2(batch=96), "gi_small"), ("c3", lambda: wl.c3(batch=64), "gi_thin"),
       ("c3_walk", lambda: wl.c3_walk(batch=64), "gi_thin"), ("c5", lambda: wl.c5(batch=8), None), ("c1", lambda: wl.c1(), "gi_cluster"),
       ("c2_floor", lambda: vr.c2_floor(96), "gi_small")]


@pytest.mark.parametrize("name,make,solver", REF, ids=[r[0] for r in REF])
def test_vjp_matches_reference(eng, name, make, solver):
    bp = make()
    out = eng.lmpc_run(bp)
    assert (out["status"] == 0).all()
    if solver:
        assert solver in eng.last_solver(), eng.last_solver()
    B = bp["batch"]
    dc, dt = _cotangents(B, out["sizes"], 5)
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    rng = np.random.default_rng(9)
    nonzero = set()
    for b in sorted({0, B // 2, B - 1}):
        inst = wl.instance(bp, b)
        o = vr.solve(inst)
        assert set(o["iact"].tolist()) == set(int(k) for k in out["iact"][b] if k > 0)
        adj = vr.adjoint(o, dc[b], dt[b])
        # one direction per input, so that every gradient is checked on its own
        for key in vr.vector_keys(inst):
            delta = vr.random_direction(inst, rng, [key])
            ref = vr.directional(inst, adj, delta)
            got = _dot(g, delta, b)
            assert abs(got - ref) <= 1e-8 * max(abs(ref), 1.0), (name, b, key, got, ref)
            if abs(ref) > 1e-6:
                nonzero.add(key)
    if name == "c2_floor":  # the lower trajectory-bound rows (quirk Q1) and the full-size control bound are active somewhere
        assert ("lower", 0) in nonzero and ("upper", 1) in nonzero, nonzero


@pytest.mark.parametrize("make", [lambda: wl.c3(batch=256), lambda: wl.c3_walk(batch=256)], ids=["c3", "c3_walk"])
def test_vjp_matches_gpu_central_differences(eng, make):
    bp = make()
    B = bp["batch"]
    base = eng.lmpc_run(bp)
    dc, dt = _cotangents(B, base["sizes"], 3)
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    act = [set(int(k) for k in base["iact"][b] if k > 0) for b in range(B)]
    rng = np.random.default_rng(4)
    checked = 0
    for key in [("x0", None), ("p", 0), ("f", 0)]:
        v = _batch_vectors(bp, key, B)
        delta = rng.normal(size=v.shape)
        grad = g["x0"] if key[0] == "x0" else g[key[0]][key[1]]
        pred = (grad * delta).sum(axis=1)
        done = np.zeros(B, bool)
        for h in (1e-3, 1e-4, 1e-5):
            ends = []
            for sgn in (1.0, -1.0):
                q = dict(bp)
                q["costs"] = [dict(c) for c in bp["costs"]]
                q["constraints"] = [dict(c) for c in bp["constraints"]]
                if key[0] == "x0":
                    q["x0"] = v + sgn * h * delta
                else:
                    (q["costs"] if key[0] == "p" else q["constraints"])[key[1]][key[0]] = v + sgn * h * delta
                ends.append(eng.lmpc_run(q))
            for b in range(B):
                if done[b] or any(set(int(k) for k in e["iact"][b] if k > 0) != act[b] for e in ends):
                    continue
                fd = ((ends[0]["control"][b] - ends[1]["control"][b]) @ dc[b] +
                      (ends[0]["trajectory"][b] - ends[1]["trajectory"][b]) @ dt[b]) / (2 * h)
                scale = max(abs(pred[b]), abs(fd), 1.0)
                assert abs(fd - pred[b]) <= 1e-7 * scale, (key, b, fd, pred[b], h)
                done[b] = True
                checked += 1
    assert checked >= B


def test_failed_instance_gets_zeros(eng):
    bp = wl.c3(batch=64)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(64, out["sizes"], 1)
    g0 = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    bad = dict(bp)
    bad["constraints"] = [dict(bp["constraints"][0])]
    f = np.asarray(bp["constraints"][0]["f"]).copy()
    f[5] = -0.1  # an empty ZMP box: infeasible
    bad["constraints"][0]["f"] = f
    out2 = eng.lmpc_run(bad)
    assert out2["status"][5] != 0 and (np.delete(out2["status"], 5) == 0).all()
    g1 = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    for k in ("x0",):
        assert not g1[k][5].any()
        np.testing.assert_allclose(np.delete(g1[k], 5, 0), np.delete(g0[k], 5, 0), rtol=1e-12, atol=1e-12)
    assert not g1["p"][0][5].any() and not g1["f"][0][5].any()
    np.testing.assert_allclose(np.delete(g1["f"][0], 5, 0), np.delete(g0["f"][0], 5, 0), rtol=1e-12, atol=1e-12)


def test_vjp_is_repeatable_and_leaves_the_build_alone(eng):
    bp = wl.c3_walk(batch=128)
    nxt = wl.c3_walk(batch=128, tick=1)
    # without a VJP
    ref_run = eng.lmpc_run(bp)
    ref_rt = eng.lmpc_retarget(nxt)
    ref_rs = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, ref_run["sizes"])
    # with VJPs in between
    run = eng.lmpc_run(bp)
    dc, dt = _cotangents(128, run["sizes"], 2)
    a = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    b = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    for k in ("x0",):
        assert np.array_equal(a[k], b[k])
    for k in ("p", "f"):
        for x, y in zip(a[k], b[k]):
            assert (x is None and y is None) or np.array_equal(x, y)
    rt = eng.lmpc_retarget(nxt)
    eng.lmpc_vjp(dcontrol=dc)
    rs = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, run["sizes"])
    for k in ("control", "trajectory", "iact", "iters"):
        assert np.array_equal(rt[k], ref_rt[k]) and np.array_equal(rs[k], ref_rs[k])
    # warm-started resolve
    eng.set_warm_start(True)
    try:
        eng.lmpc_run(bp)
        w_ref = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, run["sizes"])
        eng.lmpc_run(bp)
        eng.lmpc_vjp(dcontrol=dc)
        w = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, run["sizes"])
        assert np.array_equal(w["control"], w_ref["control"]) and np.array_equal(w["iters"], w_ref["iters"])
    finally:
        eng.set_warm_start(False)


def test_dtrajectory_equals_its_control_term(eng):
    bp = wl.c3(batch=32)
    out = eng.lmpc_run(bp)
    _, dt = _cotangents(32, out["sizes"], 6)
    from oracle import copra_numpy as cn
    Phi, Psi, _ = cn.condense(bp["A"], bp["B"], bp["d"], bp["N"])
    g_t = eng.lmpc_vjp(dtrajectory=dt)
    g_c = eng.lmpc_vjp(dcontrol=dt @ Psi)
    np.testing.assert_allclose(g_t["x0"], g_c["x0"] + dt @ Phi, rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(g_t["f"][0], g_c["f"][0], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("shards", [2, 4])
def test_sharded_vjp_is_bitwise_single_device(eng, shards):
    bp = wl.c3_walk(batch=250)  # 250 / 4: a ragged last shard
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(250, out["sizes"], 8)
    ref = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    m = capi.MultiEngine([0] * shards)
    try:
        m.lmpc_run(bp, out["sizes"])
        got = m.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    finally:
        m.close()
    assert np.array_equal(got["x0"], ref["x0"])
    for k in ("p", "f"):
        for x, y in zip(got[k], ref[k]):
            assert (x is None and y is None) or np.array_equal(x, y)


def test_autograd_matches_engine_and_detects_stale_backward(eng):
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    bp = wl.c3_walk(batch=16)
    dev = torch.device("cuda:0")
    x0 = torch.tensor(np.asarray(bp["x0"]), device=dev, requires_grad=True)
    p0 = torch.tensor(_batch_vectors(bp, ("p", 0), 16), device=dev, requires_grad=True)
    f0 = torch.tensor(_batch_vectors(bp, ("f", 0), 16), device=dev, requires_grad=True)
    ctrl, traj = ag.lmpc(eng, bp, x0, p=[p0], f=[f0])
    dc = torch.randn_like(ctrl)
    dt = torch.randn_like(traj)
    gx, gp, gf = torch.autograd.grad((ctrl * dc).sum() + (traj * dt).sum(), (x0, p0, f0), retain_graph=True)
    ref = eng.lmpc_vjp(dcontrol=dc.cpu().numpy(), dtrajectory=dt.cpu().numpy())
    assert np.array_equal(gx.cpu().numpy(), ref["x0"])
    assert np.array_equal(gp.cpu().numpy(), ref["p"][0])
    assert np.array_equal(gf.cpu().numpy(), ref["f"][0])
    eng.lmpc_run(wl.c2(batch=4))
    with pytest.raises(RuntimeError):
        torch.autograd.grad((ctrl * dc).sum(), (x0,))


def _vjp_rc(eng):
    """the raw return code of copra_b200_lmpc_vjp on the engine's last solve (no gradient requested)"""
    import ctypes as C
    return eng.lib.copra_b200_lmpc_vjp(eng.h, None, None, capi.HOST, C.byref(capi.VjpOut()))


def test_vjp_error_codes():
    eng = capi.Engine(0)
    try:
        assert _vjp_rc(eng) == -5  # no solve yet
        eng.lmpc_run(wl.c4(batch=4))
        assert _vjp_rc(eng) == -4  # initial-state mode
        eng.lmpc_run(wl.spanned(wl.c3_walk(batch=4)))
        assert _vjp_rc(eng) == -4  # full-size cost and row constraint
        bp = wl.c1()
        tb = bp["constraints"][0]
        X = bp["nx"] * (bp["N"] + 1)
        bp["constraints"][0] = dict(tb, lower=np.tile(tb["lower"], bp["N"] + 1), upper=np.tile(tb["upper"], bp["N"] + 1))
        eng.lmpc_run(bp)
        assert capi.HostBatch(bp).problem.cstrs[0].full_size == 1 and bp["constraints"][0]["lower"].shape == (X,)
        assert _vjp_rc(eng) == -4  # full-size trajectory bound
        eng.lmpc_run(vr.c2_floor(4))
        assert _vjp_rc(eng) == 0  # a full-size control bound is fine
        eng.solve_qp_batch(np.eye(2)[None], np.ones((1, 2)), None, None, None, None, np.full((1, 2), -1.0), np.full((1, 2), 1.0))
        assert _vjp_rc(eng) == -5  # a raw QP batch replaced the active sets
        big = wl.c2(batch=65536)
        eng.lmpc_run(big, want=("status",))
        assert _vjp_rc(eng) == -5  # only the last chunk of a > 65535 run is resident
    finally:
        eng.close()


def test_multi_engine_takes_host_arrays_only(eng):
    torch = pytest.importorskip("torch")
    bp = wl.c3(batch=8)
    m = capi.MultiEngine([0, 0])
    try:
        m.lmpc_run(bp, eng.sizes(capi.HostBatch(bp)))
        with pytest.raises(capi.CopraB200Error):
            m.lmpc_vjp(dcontrol=torch.zeros((8, 320), dtype=torch.float64, device="cuda:0"))
    finally:
        m.close()


def test_cpp_batched_lmpc_vjp():
    """BatchedLMPC::vjp against central differences of per-instance copra::LMPC solves, and its errors"""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([os.path.join(root, "tests", "cpp", "test_vjp")], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
