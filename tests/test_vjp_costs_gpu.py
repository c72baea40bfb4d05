"""copra_b200_lmpc_vjp_costs (K8 + k8_cost_grad) on the GPU: the gradients with respect to the cost weights and matrices
against the numpy closed forms of tests/vjp_cost_reference.py on every solver path the VJP runs after, after a retarget and
a resolve, its edge cases, bitwise stability of the vector gradients, the sharded form and torch.autograd."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import vjp_cost_reference as cr
from tests import vjp_reference as vr

pytestmark = pytest.mark.gpu

ALL = capi.VJP_WANT + capi.VJP_COST_WANT


@pytest.fixture(scope="module")
def eng():
    e = capi.Engine(0)
    yield e
    e.close()


def _cotangents(B, s, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(B, s["nU"])), rng.normal(size=(B, s["X"]))


def _check_against_reference(bp, out, g, dc, dt, samples, tag):
    B = bp["batch"]
    for b in samples:
        inst = wl.instance(bp, b)
        o = vr.solve(inst)
        assert set(o["iact"].tolist()) == set(int(k) for k in out["iact"][b] if k > 0), (tag, b)
        ref = cr.closed_form(inst, o, vr.adjoint(o, dc[b], dt[b]))
        for (kind, i), r in ref.items():
            got = g[kind][i][b]
            assert got.shape == r.shape, (tag, kind, i, got.shape, r.shape)
            err = np.abs(got - r).max()
            assert err <= 1e-7 * max(np.abs(r).max(), 1.0), (tag, b, kind, i, err, np.abs(r).max())
    # matrices a cost does not have come back as None
    for i, (_, has_m, has_n) in enumerate(capi.cost_shapes(bp)):
        assert (g["M"][i] is None) != has_m and (g["N"][i] is None) != has_n
        assert g["w"][i].shape[0] == B


def _c1_batch():
    bp = wl.c1()
    bp["batch"] = 4
    bp["x0"] = np.array([[0.0, -5.0], [0.1, -4.0], [-0.1, -6.0], [0.0, -3.0]])
    return bp


def _c2_per_instance_weights():
    bp = wl.c2(batch=64, N=110)
    rng = np.random.default_rng(2)
    bp["costs"][0] = dict(bp["costs"][0], w=np.array([10.0, 10000.0]) * rng.uniform(0.5, 2.0, size=(64, 2)))
    return bp


REF = [("c2", lambda: wl.c2(batch=96), "gi_small"), ("c3", lambda: wl.c3(batch=64), "gi_thin"),
       ("c2_n110_per_instance_w", _c2_per_instance_weights, "gi_thin"), ("c1_batch", _c1_batch, None),
       ("c2_mixed", lambda: cr.mixed(96), "gi_small"), ("c2_floor", lambda: vr.c2_floor(96), "gi_small")]


@pytest.mark.parametrize("name,make,solver", REF, ids=[r[0] for r in REF])
def test_cost_gradients_match_reference(eng, name, make, solver):
    bp = make()
    out = eng.lmpc_run(bp)
    assert (out["status"] == 0).all()
    if solver:
        assert solver in eng.last_solver(), eng.last_solver()
    if name == "c2_n110_per_instance_w":
        assert not eng.hessian_is_shared()
    if name == "c3":
        assert eng.hessian_is_shared()
    B = bp["batch"]
    dc, dt = _cotangents(B, out["sizes"], 5)
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    _check_against_reference(bp, out, g, dc, dt, sorted({0, B // 2, B - 1}), name)


def test_after_retarget_and_resolve(eng):
    bp = wl.c3_walk(batch=64)
    nxt = wl.c3_walk(batch=64, tick=3)
    run = eng.lmpc_run(bp)
    out = eng.lmpc_retarget(nxt)
    assert (out["status"] == 0).all() and "gi_thin" in eng.last_solver()
    dc, dt = _cotangents(64, run["sizes"], 7)
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    _check_against_reference(nxt, out, g, dc, dt, [0, 33, 63], "c3_walk retarget")
    # a receding-horizon resolve with new initial states on the same build
    c3 = wl.c3(batch=64)
    run = eng.lmpc_run(c3)
    x0 = np.asarray(c3["x0"]) * 0.5
    out = eng.lmpc_resolve(x0, run["sizes"])
    assert (out["status"] == 0).all()
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    _check_against_reference(dict(c3, x0=x0), out, g, dc, dt, [1, 40], "c3 resolve")


def test_failed_instance_gets_zeros(eng):
    bp = wl.c3(batch=64)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(64, out["sizes"], 1)
    g0 = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    bad = dict(bp)
    bad["constraints"] = [dict(bp["constraints"][0])]
    f = np.asarray(bp["constraints"][0]["f"]).copy()
    f[5] = -0.1  # an empty ZMP box: infeasible
    bad["constraints"][0]["f"] = f
    out2 = eng.lmpc_run(bad)
    assert out2["status"][5] != 0 and (np.delete(out2["status"], 5) == 0).all()
    g1 = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    for kind in capi.VJP_COST_WANT:
        for a, b in zip(g1[kind], g0[kind]):
            if a is None:
                continue
            assert not a[5].any()
            np.testing.assert_allclose(np.delete(a, 5, 0), np.delete(b, 5, 0), rtol=1e-12, atol=1e-12)


def _same(a, b):
    for k in set(a) | set(b):
        x, y = a[k], b[k]
        if isinstance(x, list):
            assert len(x) == len(y)
            for u, v in zip(x, y):
                assert (u is None and v is None) or np.array_equal(u, v), k
        else:
            assert (x is None and y is None) or np.array_equal(x, y), k


def test_vector_gradients_are_bitwise_unchanged_and_calls_repeat(eng):
    for bp in (wl.c3_walk(batch=128), cr.mixed(64)):
        out = eng.lmpc_run(bp)
        dc, dt = _cotangents(bp["batch"], out["sizes"], 2)
        plain = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
        a = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
        b = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
        _same({k: a[k] for k in capi.VJP_WANT}, plain)
        _same(a, b)
        # dcontrol alone, and only some of the cost gradients
        only = eng.lmpc_vjp(dcontrol=dc, want=("w", "M"))
        assert only["x0"] is None and only["N"] == [None] * len(bp["costs"])


def test_shared_weights_give_the_per_instance_gradients(eng):
    bp = wl.c3(batch=64)
    per = dict(bp)
    per["costs"] = [dict(c) for c in bp["costs"]]
    per["costs"][0]["w"] = np.tile(np.asarray(bp["costs"][0]["w"]), (64, 1))
    per["costs"][1]["N"] = np.tile(np.asarray(bp["costs"][1]["N"]), (64, 1, 1))
    out = eng.lmpc_run(bp)
    assert eng.hessian_is_shared()
    dc, dt = _cotangents(64, out["sizes"], 3)
    g_shared = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    eng.lmpc_run(per)
    assert not eng.hessian_is_shared()
    g_per = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    for kind in capi.VJP_COST_WANT:
        for a, b in zip(g_shared[kind], g_per[kind]):
            if a is not None:
                np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-9 * np.abs(b).max())


@pytest.mark.parametrize("shards", [2, 4])
def test_sharded_is_bitwise_single_device(eng, shards):
    bp = cr.mixed(250)  # 250 / 4: a ragged last shard
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(250, out["sizes"], 8)
    ref = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    m = capi.MultiEngine([0] * shards)
    try:
        m.lmpc_run(bp, out["sizes"])
        got = m.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    finally:
        m.close()
    _same(got, ref)


def test_error_codes(eng):
    out = eng.lmpc_run(wl.c2(batch=4))
    assert (out["status"] == 0).all()
    buf = np.zeros(64)
    ptrs = (C.c_void_p * 2)(buf.ctypes.data, None)
    co = capi.VjpCostOut()
    co.M = C.cast(ptrs, C.POINTER(C.c_void_p))
    assert eng.lib.copra_b200_lmpc_vjp_costs(eng.h, None, None, capi.HOST, None, C.byref(co)) == 0  # TargetCost's M
    ptrs[0], ptrs[1] = None, buf.ctypes.data
    assert eng.lib.copra_b200_lmpc_vjp_costs(eng.h, None, None, capi.HOST, None, C.byref(co)) == -1  # ControlCost: no M
    co2 = capi.VjpCostOut()
    co2.N = C.cast((C.c_void_p * 2)(buf.ctypes.data, None), C.POINTER(C.c_void_p))
    assert eng.lib.copra_b200_lmpc_vjp_costs(eng.h, None, None, capi.HOST, None, C.byref(co2)) == -1  # TargetCost: no N
    eng.lmpc_run(wl.c4(batch=4))
    assert eng.lib.copra_b200_lmpc_vjp_costs(eng.h, None, None, capi.HOST, None, C.byref(capi.VjpCostOut())) == -4


def test_autograd_matches_engine_and_reference(eng):
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    bp = cr.mixed(16)
    dev = torch.device("cuda:0")
    B = bp["batch"]
    x0 = torch.tensor(np.asarray(bp["x0"]), device=dev)
    c0, c2 = bp["costs"][0], bp["costs"][2]
    w0 = torch.tensor(np.tile(np.asarray(c0["w"]), (B, 1)), device=dev, requires_grad=True)  # batched
    M0 = torch.tensor(np.asarray(c0["M"]), device=dev, requires_grad=True)                    # shared
    w2 = torch.tensor(np.asarray(c2["w"]), device=dev, requires_grad=True)                    # shared
    M2 = torch.tensor(np.tile(np.asarray(c2["M"]), (B, 1, 1)), device=dev, requires_grad=True)  # batched
    N2 = torch.tensor(np.asarray(c2["N"]), device=dev, requires_grad=True)                    # shared
    ctrl, traj = ag.lmpc(eng, bp, x0, w=[w0, None, w2], M=[M0, None, M2], N=[None, None, N2])
    g = torch.Generator(device=dev).manual_seed(3)
    dc = torch.randn(ctrl.shape, dtype=torch.float64, device=dev, generator=g)
    dt = torch.randn(traj.shape, dtype=torch.float64, device=dev, generator=g)
    grads = torch.autograd.grad((ctrl * dc).sum() + (traj * dt).sum(), (w0, M0, w2, M2, N2), retain_graph=True)
    ref = eng.lmpc_vjp(dcontrol=dc.cpu().numpy(), dtrajectory=dt.cpu().numpy(), want=ALL)
    assert np.array_equal(grads[0].cpu().numpy(), ref["w"][0])
    assert np.array_equal(grads[3].cpu().numpy(), ref["M"][2])
    for got, r in ((grads[1], ref["M"][0]), (grads[2], ref["w"][2]), (grads[4], ref["N"][2])):
        np.testing.assert_allclose(got.cpu().numpy(), r.sum(0), rtol=1e-12, atol=1e-12 * np.abs(r).sum())
    # against the numpy closed forms on one instance (the tensors hold bp's values)
    inst = wl.instance(bp, 5)
    o = vr.solve(inst)
    cf = cr.closed_form(inst, o, vr.adjoint(o, dc[5].cpu().numpy(), dt[5].cpu().numpy()))
    np.testing.assert_allclose(grads[0][5].cpu().numpy(), cf[("w", 0)], rtol=1e-7, atol=1e-7 * np.abs(cf[("w", 0)]).max())
    np.testing.assert_allclose(grads[3][5].cpu().numpy(), cf[("M", 2)], rtol=1e-7, atol=1e-7 * np.abs(cf[("M", 2)]).max())
    # forward mode along a cost matrix is refused, not answered wrongly
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        wd = fwAD.make_dual(w2.detach(), torch.ones_like(w2))
        with pytest.raises(NotImplementedError):
            ag.lmpc(eng, bp, x0, w=[None, None, wd])


def _cpp_problem():
    """the problem tests/cpp/test_vjp_costs.cpp builds: a double integrator with a tracking, an effort and a mixed cost"""
    T, N, B = 0.05, 20, 4
    b = np.arange(B)
    return dict(nx=2, nu=1, N=N, batch=B, initial_state=False, A=np.array([[1.0, T], [0.0, 1.0]]),
                B=np.array([[0.5 * T * T], [T]]), d=np.zeros(2), x0=np.stack([0.1 * b, -0.2 + 0.05 * b], axis=1),
                costs=[dict(kind="trajectory", M=np.eye(2), p=np.stack([np.sin(b), np.zeros(B)], axis=1), w=np.array([10.0, 1.0])),
                       dict(kind="control", N=np.eye(1), p=np.zeros(1), w=np.array([1e-2])),
                       dict(kind="mixed", M=np.array([[0.5, 1.0]]), N=np.array([[0.1]]), p=np.array([0.2]), w=np.array([2.0]))],
                constraints=[dict(kind="control_bound", lower=np.array([-2.0]), upper=np.array([3.0]))])


def test_cpp_batched_lmpc_vjp_costs(tmp_path):
    """BatchedLMPC::vjp with cost outputs (tests/cpp/test_vjp_costs.cpp) against the numpy closed forms, and its errors"""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dump = str(tmp_path / "grads.txt")
    r = subprocess.run([os.path.join(root, "tests", "cpp", "test_vjp_costs"), dump], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    got = np.loadtxt(dump).reshape(4, -1)  # per instance: dw0 (2), dM0 (2 x 2, column-major), dw1, dN1, dw2, dM2 (1 x 2), dN2
    bp = _cpp_problem()
    nU = bp["N"]
    dc = np.sin(0.7 * np.arange(4 * nU) + 1.0).reshape(4, nU)
    for b in range(4):
        inst = wl.instance(bp, b)
        o = vr.solve(inst)
        cf = cr.closed_form(inst, o, vr.adjoint(o, dc[b]))
        ref = np.concatenate([cf[("w", 0)], cf[("M", 0)].T.ravel(), cf[("w", 1)], cf[("N", 1)].T.ravel(), cf[("w", 2)],
                              cf[("M", 2)].T.ravel(), cf[("N", 2)].T.ravel()])
        np.testing.assert_allclose(got[b], ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())
