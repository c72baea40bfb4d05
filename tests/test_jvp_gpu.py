"""copra_b200_lmpc_jvp / copra_b200_lmpc_feedback_gain (K9) on the GPU: against the dense numpy forward reference, the adjoint
identity with the VJP (K8), the gain against an identity JVP, the VJP and a re-solve, its edge cases, the sharded form,
forward-mode torch.autograd and the C++ facade."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import jvp_reference as jr
from tests import vjp_reference as vr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = capi.Engine(0)
    yield e
    e.close()


def _batch_vector(bp, key, B):
    """the (batch, len) values of one vector input (a shared vector broadcast)"""
    kind, i = key
    v = np.asarray(bp["x0"] if kind == "x0" else (bp["costs"] if kind == "p" else bp["constraints"])[i][kind], float)
    return np.broadcast_to(v, (B,) + v.shape[-1:]).copy() if v.ndim == 1 else v.copy()


def _tangent_args(tangents):
    """{key: (batch, k, len)} -> lmpc_jvp keyword arguments"""
    args = dict(x0=None, p={}, f={}, lower={}, upper={})
    for (kind, i), t in tangents.items():
        if kind == "x0":
            args["x0"] = t
        else:
            args[kind][i] = t
    for kind in ("p", "f", "lower", "upper"):
        d = args[kind]
        args[kind] = [d.get(i) for i in range(max(d) + 1)] if d else None
    return args


def _random_tangents(bp, keys, B, k, rng, direction=None):
    """(batch, k, len) tangents for `keys`: random where the input is finite; with `direction`, key j only moves along
    direction[j] (one input kind per direction)"""
    out = {}
    for j, key in enumerate(keys):
        v = _batch_vector(bp, key, B)
        t = np.where(np.isfinite(v)[:, None, :], rng.normal(size=(B, k, v.shape[1])), 0.0)
        if direction is not None:
            mask = np.zeros((1, k, 1))
            mask[0, direction[j], 0] = 1.0
            t = t * mask
        out[key] = t
    return out


REF = [("c2", lambda: wl.c2(batch=96), "gi_small"), ("c3", lambda: wl.c3(batch=64), "gi_thin"),
       ("c3_walk", lambda: wl.c3_walk(batch=64), "gi_thin"), ("c5", lambda: wl.c5(batch=8), None), ("c1", lambda: wl.c1(), "gi_cluster"),
       ("c2_floor", lambda: vr.c2_floor(96), "gi_small")]


@pytest.mark.parametrize("name,make,solver", REF, ids=[r[0] for r in REF])
def test_jvp_matches_reference(eng, name, make, solver):
    bp = make()
    out = eng.lmpc_run(bp)
    assert (out["status"] == 0).all()
    if solver:
        assert solver in eng.last_solver(), eng.last_solver()
    B = bp["batch"]
    keys = vr.vector_keys(wl.instance(bp, 0))
    # one input kind per direction: direction j moves input keys[j] alone, so every kind is checked on its own
    tang = _random_tangents(bp, keys, B, len(keys), np.random.default_rng(21), direction=list(range(len(keys))))
    du, dx = eng.lmpc_jvp(**_tangent_args(tang))
    assert du.shape == (B, len(keys), out["sizes"]["nU"]) and dx.shape == (B, len(keys), out["sizes"]["X"])
    moved = set()
    for b in sorted({0, B // 2, B - 1}):
        inst = wl.instance(bp, b)
        o = vr.solve(inst)
        assert set(o["iact"].tolist()) == set(int(k) for k in out["iact"][b] if k > 0)
        for j, key in enumerate(keys):
            ref_u, ref_x = jr.tangent(inst, o, {key: tang[key][b, j]})
            for got, ref in ((du[b, j], ref_u), (dx[b, j], ref_x)):
                err = np.abs(got - ref).max()
                assert err <= 1e-8 * max(np.abs(ref).max(), 1.0), (name, b, key, err, np.abs(ref).max())
            if np.abs(ref_u).max() > 1e-6:
                moved.add(key)
    if name == "c2_floor":  # the lower trajectory-bound rows (quirk Q1) and the full-size control bound are active somewhere
        assert ("lower", 0) in moved and ("upper", 1) in moved, moved


ADJ = [("c3", lambda: wl.c3(batch=256)), ("c3_walk", lambda: wl.c3_walk(batch=256)), ("c2", lambda: wl.c2(batch=1024))]


@pytest.mark.parametrize("name,make", ADJ, ids=[a[0] for a in ADJ])
def test_jvp_is_the_adjoint_of_the_vjp(eng, name, make):
    # sum_b <gbar_b, JVP_b(thetadot)> == sum_b <VJP_b(gbar), thetadot> with random tangents on every input kind at once
    bp = make()
    out = eng.lmpc_run(bp)
    B = bp["batch"]
    rng = np.random.default_rng(22)
    dc, dt = rng.normal(size=(B, out["sizes"]["nU"])), rng.normal(size=(B, out["sizes"]["X"]))
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    keys = vr.vector_keys(wl.instance(bp, 0))
    tang = _random_tangents(bp, keys, B, 1, rng)
    du, dx = eng.lmpc_jvp(**_tangent_args(tang))
    lhs = float((dc * du[:, 0]).sum() + (dt * dx[:, 0]).sum())
    rhs = 0.0
    for (kind, i), t in tang.items():
        grad = g["x0"] if kind == "x0" else g[kind][i]
        rhs += float((grad * t[:, 0]).sum())
    scale = float(np.abs(dc * du[:, 0]).sum() + np.abs(dt * dx[:, 0]).sum())
    assert abs(lhs - rhs) <= 1e-10 * max(abs(lhs), abs(rhs), scale), (name, lhs, rhs, scale)


@pytest.mark.parametrize("make", [lambda: wl.c3(batch=64), lambda: vr.c2_floor(128)], ids=["c3", "c2_floor"])
def test_gain_is_the_identity_jvp_and_matches_the_vjp(eng, make):
    bp = make()
    out = eng.lmpc_run(bp)
    B, nx, nu, N = bp["batch"], bp["nx"], bp["nu"], bp["N"]
    nU, X = out["sizes"]["nU"], out["sizes"]["X"]
    Ku, Kx = eng.lmpc_feedback_gain(steps=N)
    assert Ku.shape == (B, nU, nx) and Kx.shape == (B, X, nx)
    du, dx = eng.lmpc_jvp(x0=np.broadcast_to(np.eye(nx), (B, nx, nx)).copy())
    np.testing.assert_allclose(Ku, du.transpose(0, 2, 1), rtol=1e-12, atol=1e-12 * np.abs(du).max())
    np.testing.assert_allclose(Kx, dx.transpose(0, 2, 1), rtol=1e-12, atol=1e-12 * np.abs(dx).max())
    # the first nx rows of Kx are dx0/dx0
    np.testing.assert_allclose(Kx[:, :nx], np.broadcast_to(np.eye(nx), (B, nx, nx)), rtol=0, atol=1e-15)
    # steps = 1: the first nu rows, bitwise
    K1u, K1x = eng.lmpc_feedback_gain(steps=1)
    assert K1u.shape == (B, nu, nx) and K1x.shape == (B, 2 * nx, nx)
    assert np.array_equal(K1u, Ku[:, :nu]) and np.array_equal(K1x, Kx[:, :2 * nx])
    # row k of Ku is the VJP of the unit cotangent e_k with respect to x0
    for k in range(nu):
        e = np.zeros((B, nU))
        e[:, k] = 1.0
        gx = eng.lmpc_vjp(dcontrol=e, want=("x0",))["x0"]
        np.testing.assert_allclose(K1u[:, k], gx, rtol=1e-10, atol=1e-10 * max(1.0, np.abs(gx).max()))


@pytest.mark.parametrize("make", [lambda: wl.c3(batch=256), lambda: wl.c3_walk(batch=256)], ids=["c3", "c3_walk"])
def test_gain_predicts_a_resolve(eng, make):
    bp = make()
    B, nx = bp["batch"], bp["nx"]
    base = eng.lmpc_run(bp)
    Ku, Kx = eng.lmpc_feedback_gain(steps=bp["N"])
    rng = np.random.default_rng(23)
    delta = rng.normal(size=(B, nx))
    x0 = _batch_vector(bp, ("x0", None), B)
    eps = 1e-4 * max(1.0, np.abs(x0).max())
    moved = eng.lmpc_resolve(x0 + eps * delta, base["sizes"])
    checked = 0
    for b in range(B):
        if base["status"][b] or moved["status"][b]:
            continue
        if set(int(k) for k in base["iact"][b] if k > 0) != set(int(k) for k in moved["iact"][b] if k > 0):
            continue  # the affine law holds on one active set only
        for out, K in (("control", Ku), ("trajectory", Kx)):
            pred = base[out][b] + eps * K[b] @ delta[b]
            err = np.abs(moved[out][b] - pred).max()
            assert err <= 1e-9 * max(1.0, np.abs(moved[out][b]).max()), (b, out, err)
        checked += 1
    assert checked >= B // 2, checked


def test_failed_instance_repeatability_and_build_untouched(eng):
    bp = wl.c3(batch=64)
    eng.lmpc_run(bp)
    Ku0, Kx0 = eng.lmpc_feedback_gain(steps=2)
    bad = dict(bp)
    bad["constraints"] = [dict(bp["constraints"][0])]
    f = np.asarray(bp["constraints"][0]["f"]).copy()
    f[5] = -0.1  # an empty ZMP box: infeasible
    bad["constraints"][0]["f"] = f
    out = eng.lmpc_run(bad)
    assert out["status"][5] != 0 and (np.delete(out["status"], 5) == 0).all()
    Ku1, Kx1 = eng.lmpc_feedback_gain(steps=2)
    assert not Ku1[5].any() and not Kx1[5].any()
    for a, b in ((Ku1, Ku0), (Kx1, Kx0)):
        np.testing.assert_allclose(np.delete(a, 5, 0), np.delete(b, 5, 0), rtol=1e-12, atol=1e-12 * np.abs(b).max())
    tang = _random_tangents(bad, vr.vector_keys(wl.instance(bad, 0)), 64, 3, np.random.default_rng(24))
    du, dx = eng.lmpc_jvp(**_tangent_args(tang))
    assert not du[5].any() and not dx[5].any()
    # two calls are bitwise equal
    du2, dx2 = eng.lmpc_jvp(**_tangent_args(tang))
    Ku2, Kx2 = eng.lmpc_feedback_gain(steps=2)
    assert np.array_equal(du, du2) and np.array_equal(dx, dx2)
    assert np.array_equal(Ku1, Ku2) and np.array_equal(Kx1, Kx2)

    # retarget, resolve and a warm-started resolve after a JVP and a gain give bitwise what they give without
    walk, nxt = wl.c3_walk(batch=128), wl.c3_walk(batch=128, tick=1)
    ref_run = eng.lmpc_run(walk)
    ref_rt = eng.lmpc_retarget(nxt)
    ref_rs = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, ref_run["sizes"])
    run = eng.lmpc_run(walk)
    tw = _random_tangents(walk, [("x0", None), ("p", 0), ("f", 0)], 128, 2, np.random.default_rng(25))
    eng.lmpc_jvp(**_tangent_args(tw))
    eng.lmpc_feedback_gain(steps=3)
    rt = eng.lmpc_retarget(nxt)
    eng.lmpc_feedback_gain(steps=1)
    eng.lmpc_jvp(**_tangent_args(tw))
    rs = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, run["sizes"])
    for k in ("control", "trajectory", "iact", "iters"):
        assert np.array_equal(rt[k], ref_rt[k]) and np.array_equal(rs[k], ref_rs[k])
    eng.set_warm_start(True)
    try:
        eng.lmpc_run(walk)
        w_ref = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, run["sizes"])
        eng.lmpc_run(walk)
        eng.lmpc_feedback_gain(steps=1)
        eng.lmpc_jvp(**_tangent_args(tw))
        w = eng.lmpc_resolve(np.asarray(nxt["x0"]) * 0.5, run["sizes"])
        assert np.array_equal(w["control"], w_ref["control"]) and np.array_equal(w["iters"], w_ref["iters"])
    finally:
        eng.set_warm_start(False)


@pytest.mark.parametrize("shards", [2, 4])
def test_sharded_jvp_and_gain_are_bitwise_single_device(eng, shards):
    bp = wl.c3_walk(batch=250)  # 250 / 4: a ragged last shard
    out = eng.lmpc_run(bp)
    tang = _random_tangents(bp, vr.vector_keys(wl.instance(bp, 0)), 250, 3, np.random.default_rng(26))
    ref = eng.lmpc_jvp(**_tangent_args(tang))
    ref_gain = eng.lmpc_feedback_gain(steps=4)
    m = capi.MultiEngine([0] * shards)
    try:
        m.lmpc_run(bp, out["sizes"])
        got = m.lmpc_jvp(**_tangent_args(tang))
        got_gain = m.lmpc_feedback_gain(steps=4)
    finally:
        m.close()
    for a, b in zip(got + got_gain, ref + ref_gain):
        assert np.array_equal(a, b)


def test_forward_ad_matches_engine_and_backward_still_works(eng):
    torch = pytest.importorskip("torch")
    import torch.autograd.forward_ad as fwAD
    from copra_b200 import autograd as ag
    bp = wl.c3_walk(batch=16)
    dev = torch.device("cuda:0")
    x0 = torch.tensor(np.asarray(bp["x0"]), device=dev, requires_grad=True)
    p0 = torch.tensor(_batch_vector(bp, ("p", 0), 16), device=dev, requires_grad=True)
    f0 = torch.tensor(_batch_vector(bp, ("f", 0), 16), device=dev, requires_grad=True)
    g = torch.Generator(device=dev).manual_seed(3)
    tx, tp, tf = (torch.randn(t.shape, dtype=torch.float64, device=dev, generator=g) for t in (x0, p0, f0))
    with fwAD.dual_level():
        ctrl, traj = ag.lmpc(eng, bp, fwAD.make_dual(x0, tx), p=[fwAD.make_dual(p0, tp)], f=[fwAD.make_dual(f0, tf)])
        dctrl, dtraj = fwAD.unpack_dual(ctrl).tangent, fwAD.unpack_dual(traj).tangent
        ref_u, ref_x = eng.lmpc_jvp(x0=tx[:, None], p=[tp[:, None], None], f=[tf[:, None]])
        assert torch.equal(dctrl, ref_u[:, 0]) and torch.equal(dtraj, ref_x[:, 0])
        # reverse mode on the same graph, as before
        dc = torch.randn(ctrl.shape, dtype=torch.float64, device=dev, generator=g)
        gx, gf = torch.autograd.grad((ctrl * dc).sum(), (x0, f0))
    ref = eng.lmpc_vjp(dcontrol=dc.cpu().numpy())
    assert np.array_equal(gx.cpu().numpy(), ref["x0"]) and np.array_equal(gf.cpu().numpy(), ref["f"][0])


def _jvp_rc(eng, ndir=1, null=False):
    t = capi.JvpIn()
    t.ndir = ndir
    return eng.lib.copra_b200_lmpc_jvp(eng.h, None if null else C.byref(t), capi.HOST, None, None)


def _gain_rc(eng, steps=1):
    return eng.lib.copra_b200_lmpc_feedback_gain(eng.h, steps, None, None, capi.HOST)


def test_jvp_error_codes():
    eng = capi.Engine(0)
    try:
        assert _jvp_rc(eng) == -5 and _gain_rc(eng) == -5  # no solve yet
        eng.lmpc_run(wl.c4(batch=4))
        assert _jvp_rc(eng) == -4 and _gain_rc(eng) == -4  # initial-state mode
        eng.lmpc_run(wl.spanned(wl.c3_walk(batch=4)))
        assert _jvp_rc(eng) == -4 and _gain_rc(eng) == -4  # full-size cost and row constraint
        bp = wl.c1()
        tb = bp["constraints"][0]
        bp["constraints"][0] = dict(tb, lower=np.tile(tb["lower"], bp["N"] + 1), upper=np.tile(tb["upper"], bp["N"] + 1))
        eng.lmpc_run(bp)
        assert capi.HostBatch(bp).problem.cstrs[0].full_size == 1
        assert _jvp_rc(eng) == -4 and _gain_rc(eng) == -4  # full-size trajectory bound
        floor = vr.c2_floor(4)
        eng.lmpc_run(floor)
        assert _jvp_rc(eng) == 0 and _gain_rc(eng) == 0  # a full-size control bound is fine
        assert _jvp_rc(eng, ndir=0) == -1 and _jvp_rc(eng, null=True) == -1
        assert _gain_rc(eng, 0) == -1 and _gain_rc(eng, floor["N"] + 1) == -1 and _gain_rc(eng, floor["N"]) == 0
        eng.solve_qp_batch(np.eye(2)[None], np.ones((1, 2)), None, None, None, None, np.full((1, 2), -1.0), np.full((1, 2), 1.0))
        assert _jvp_rc(eng) == -5 and _gain_rc(eng) == -5  # a raw QP batch replaced the active sets
        eng.lmpc_run(wl.c2(batch=65536), want=("status",))
        assert _jvp_rc(eng) == -5 and _gain_rc(eng) == -5  # only the last chunk of a > 65535 run is resident
    finally:
        eng.close()


def test_multi_engine_takes_host_arrays_only(eng):
    torch = pytest.importorskip("torch")
    bp = wl.c3(batch=8)
    m = capi.MultiEngine([0, 0])
    try:
        m.lmpc_run(bp, eng.sizes(capi.HostBatch(bp)))
        with pytest.raises(capi.CopraB200Error):
            m.lmpc_jvp(x0=torch.zeros((8, 1, 6), dtype=torch.float64, device="cuda:0"))
        with pytest.raises(capi.CopraB200Error) as e:
            m.lmpc_feedback_gain(steps=0)
        assert e.value.code == -1
    finally:
        m.close()


def test_cpp_batched_lmpc_jvp():
    """BatchedLMPC::feedbackGain and ::jvp against central differences of per-instance copra::LMPC solves, and their errors"""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([os.path.join(root, "tests", "cpp", "test_jvp")], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
