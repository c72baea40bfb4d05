"""copra_b200_lmpc_vjp_model (K8 with the forward solve as a second right-hand side + k8_model_grad) on the GPU: the gradients
with respect to A, B, d, E and G against the numpy closed forms of tests/vjp_model_reference.py on every solver path the VJP
runs after, after a retarget and a resolve, against central differences of the GPU forward, its edge cases, bitwise
stability of the vector and cost gradients, the sharded form, the C++ facade and torch.autograd."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import vjp_cost_reference as cr
from tests import vjp_model_reference as mr
from tests import vjp_reference as vr

pytestmark = pytest.mark.gpu

ALL = capi.VJP_WANT + capi.VJP_MODEL_WANT
EVERYTHING = ALL + capi.VJP_COST_WANT


@pytest.fixture(scope="module")
def eng():
    e = capi.Engine(0)
    yield e
    e.close()


def _cotangents(B, s, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(B, s["nU"])), rng.normal(size=(B, s["X"]))


def _got(g, key, b):
    kind, j = key
    return g[kind][b] if kind in mr.SYSTEM else g[kind][j][b]


def _check_against_reference(bp, out, g, dc, dt, samples, tag):
    for b in samples:
        inst = wl.instance(bp, b)
        o = vr.solve(inst)
        assert set(o["iact"].tolist()) == set(int(k) for k in out["iact"][b] if k > 0), (tag, b)
        ref, _ = mr.closed_form(inst, o, vr.adjoint(o, dc[b], dt[b]), dt[b])
        for key, r in ref.items():
            got = _got(g, key, b)
            assert got.shape == r.shape, (tag, key, got.shape, r.shape)
            err = np.abs(got - r).max()
            assert err <= 1e-8 * max(np.abs(r).max(), 1.0), (tag, b, key, err, np.abs(r).max())
    for j, (_, has_e, has_g) in enumerate(capi.cstr_shapes(bp)):
        assert (g["E"][j] is None) != has_e and (g["G"][j] is None) != has_g


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
       ("c2_n110_per_instance_w", _c2_per_instance_weights, "gi_thin"), ("c3_cluster", lambda: wl.c3(batch=4), "cluster"),
       ("c5_tight", lambda: mr.c5_tight(64), None), ("c1_batch", _c1_batch, None),
       ("c2_mixed", lambda: cr.mixed(96), "gi_small"), ("c2_floor", lambda: vr.c2_floor(96), "gi_small"),
       ("c3_g", lambda: mr.c3_g(64), None), ("c2_two_inputs", lambda: mr.c2_two_inputs(64), None)]


@pytest.mark.parametrize("name,make,solver", REF, ids=[r[0] for r in REF])
def test_model_gradients_match_reference(eng, name, make, solver):
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
    _check_against_reference(bp, out, g, dc, dt, sorted({0, 1, B // 2, B - 1}), name)


def test_after_retarget_and_resolve(eng):
    bp = wl.c3_walk(batch=64)
    nxt = wl.c3_walk(batch=64, tick=3)
    run = eng.lmpc_run(bp)
    out = eng.lmpc_retarget(nxt)
    assert (out["status"] == 0).all() and "gi_thin" in eng.last_solver()
    dc, dt = _cotangents(64, run["sizes"], 7)
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    _check_against_reference(nxt, out, g, dc, dt, [0, 33, 63], "c3_walk retarget")
    c3 = wl.c3(batch=64)
    run = eng.lmpc_run(c3)
    x0 = np.asarray(c3["x0"]) * 0.5
    out = eng.lmpc_resolve(x0, run["sizes"])
    assert (out["status"] == 0).all()
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    _check_against_reference(dict(c3, x0=x0), out, g, dc, dt, [1, 40], "c3 resolve")


def test_central_differences_of_the_gpu_forward(eng):
    """<gradient, delta> against central differences of the GPU solutions along random A, B, d, E and G directions, on the
    instances whose active set does not change across the step"""
    bp = mr.c3_g(64)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(64, out["sizes"], 12)
    g = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    rng = np.random.default_rng(13)
    act = [set(int(k) for k in r if k > 0) for r in out["iact"]]
    checked = 0
    for key in [(k, 0) for k in ("A", "B", "d", "E", "G")]:
        kind = key[0]
        src = bp if kind in mr.SYSTEM else bp["constraints"][0]
        theta = np.broadcast_to(np.asarray(src[kind], float), (64,) + np.asarray(mr.get_matrix(wl.instance(bp, 0), key)).shape)
        delta = rng.normal(size=theta.shape) * np.maximum(np.abs(theta), 1e-2 * max(np.abs(theta).max(), 1.0))
        h = 1e-6
        loss, same = [], np.ones(64, bool)
        for s in (1.0, -1.0):
            pb = dict(bp, constraints=[dict(c) for c in bp["constraints"]])
            (pb if kind in mr.SYSTEM else pb["constraints"][0])[kind] = theta + s * h * delta
            o = eng.lmpc_run(pb)
            same &= (o["status"] == 0) & np.array([set(int(k) for k in r if k > 0) == a for r, a in zip(o["iact"], act)])
            loss.append((o["control"] * dc).sum(1) + (o["trajectory"] * dt).sum(1))
        fd = (loss[0] - loss[1]) / (2.0 * h)
        got = g[kind] if kind in mr.SYSTEM else g[kind][0]
        pred = (got * delta).reshape(64, -1).sum(1)
        mag = np.maximum(np.abs((got * delta).reshape(64, -1)).sum(1), 1e-12)
        assert same.sum() >= 32, key
        assert (np.abs(fd - pred)[same] <= 1e-4 * mag[same]).all(), (key, np.max(np.abs(fd - pred)[same] / mag[same]))
        checked += int(same.sum())
    assert checked >= 160


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
    for kind in capi.VJP_MODEL_WANT:
        for a, b in (zip(g1[kind], g0[kind]) if kind in ("E", "G") else [(g1[kind], g0[kind])]):
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


def test_vector_and_cost_gradients_are_bitwise_unchanged_and_calls_repeat(eng):
    for bp in (wl.c3_walk(batch=128), cr.mixed(64), mr.c2_two_inputs(64)):
        out = eng.lmpc_run(bp)
        dc, dt = _cotangents(bp["batch"], out["sizes"], 2)
        plain = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=capi.VJP_WANT + capi.VJP_COST_WANT)
        a = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=EVERYTHING)
        b = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=EVERYTHING)
        _same({k: a[k] for k in plain}, plain)
        _same(a, b)
        only = eng.lmpc_vjp(dcontrol=dc, want=("d",))
        assert only["x0"] is None and only["A"] is None and only["E"] == [None] * len(bp["constraints"])
        np.testing.assert_allclose(only["d"], eng.lmpc_vjp(dcontrol=dc, want=("d", "x0"))["d"], rtol=0, atol=0)


def test_launch_count_without_model_gradients(eng):
    """model = NULL runs the launches it ran before; model gradients add one k8_model_grad per chunk"""
    bp = wl.c3(batch=64)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(64, out["sizes"], 6)
    counts = {}
    for name, want in (("plain", capi.VJP_WANT), ("costs", capi.VJP_WANT + capi.VJP_COST_WANT), ("model", ALL)):
        before = eng.launch_count()
        eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=want)
        counts[name] = eng.launch_count() - before
    o = capi.VjpOut()
    before = eng.launch_count()
    assert eng.lib.copra_b200_lmpc_vjp_model(eng.h, None, None, capi.HOST, C.byref(o), None, None) == 0
    assert eng.launch_count() - before == counts["plain"]
    assert counts["costs"] == counts["plain"] + 1 and counts["model"] == counts["plain"] + 1, counts


def test_shared_model_gives_the_per_instance_gradients(eng):
    bp = wl.c3(batch=64)
    per = dict(bp, A=np.tile(np.asarray(bp["A"]), (64, 1, 1)), B=np.tile(np.asarray(bp["B"]), (64, 1, 1)))
    out = eng.lmpc_run(bp)
    assert eng.hessian_is_shared()
    dc, dt = _cotangents(64, out["sizes"], 3)
    g_shared = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    eng.lmpc_run(per)
    assert not eng.hessian_is_shared()
    g_per = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=ALL)
    for kind in capi.VJP_MODEL_WANT:
        for a, b in (zip(g_shared[kind], g_per[kind]) if kind in ("E", "G") else [(g_shared[kind], g_per[kind])]):
            if a is not None:
                np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-9 * np.abs(b).max())


@pytest.mark.parametrize("shards", [2, 4])
def test_sharded_is_bitwise_single_device(eng, shards):
    bp = mr.c2_two_inputs(250)  # 250 / 4: a ragged last shard
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(250, out["sizes"], 8)
    ref = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=EVERYTHING)
    m = capi.MultiEngine([0] * shards)
    try:
        m.lmpc_run(bp, out["sizes"])
        got = m.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=EVERYTHING)
    finally:
        m.close()
    _same(got, ref)


def test_error_codes(eng):
    out = eng.lmpc_run(wl.c5(batch=4))
    assert (out["status"] == 0).all()
    buf = np.zeros(4 * 8 * 12)

    def call(kind, j):
        ptrs = (C.c_void_p * 2)(*[buf.ctypes.data if i == j else None for i in range(2)])
        mo = capi.VjpModelOut()
        setattr(mo, kind, C.cast(ptrs, C.POINTER(C.c_void_p)))
        return eng.lib.copra_b200_lmpc_vjp_model(eng.h, None, None, capi.HOST, None, None, C.byref(mo))
    assert call("E", 0) == 0    # the TrajectoryConstraint's E
    assert call("G", 0) == -1   # a TrajectoryConstraint has no G
    assert call("E", 1) == -1   # nor has a bound an E
    assert call("G", 1) == -1
    eng.lmpc_run(mr.c2_two_inputs(4))
    buf2 = np.zeros(4 * 2)
    mo = capi.VjpModelOut()
    mo.E = C.cast((C.c_void_p * 4)(None, None, buf2.ctypes.data, None), C.POINTER(C.c_void_p))
    assert eng.lib.copra_b200_lmpc_vjp_model(eng.h, None, None, capi.HOST, None, None, C.byref(mo)) == -1  # CONTROL: no E
    eng.lmpc_run(wl.c4(batch=4))
    assert eng.lib.copra_b200_lmpc_vjp_model(eng.h, None, None, capi.HOST, None, None, C.byref(capi.VjpModelOut())) == -4


def test_autograd_matches_engine_and_reference(eng):
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    bp = mr.c3_g(16)
    dev = torch.device("cuda:0")
    B = bp["batch"]
    x0 = torch.tensor(np.asarray(bp["x0"]), device=dev)
    A = torch.tensor(np.asarray(bp["A"]), device=dev, requires_grad=True)                         # shared
    Bm = torch.tensor(np.tile(np.asarray(bp["B"]), (B, 1, 1)), device=dev, requires_grad=True)     # batched
    d = torch.tensor(np.asarray(bp["d"]), device=dev, requires_grad=True)                         # shared
    E = torch.tensor(np.asarray(bp["constraints"][0]["E"]), device=dev, requires_grad=True)       # batched (C3's E is)
    G = torch.tensor(np.asarray(bp["constraints"][0]["G"]), device=dev, requires_grad=True)       # shared
    ctrl, traj = ag.lmpc(eng, bp, x0, A=A, B=Bm, d=d, E=[E], G=[G])
    gen = torch.Generator(device=dev).manual_seed(3)
    dc = torch.randn(ctrl.shape, dtype=torch.float64, device=dev, generator=gen)
    dt = torch.randn(traj.shape, dtype=torch.float64, device=dev, generator=gen)
    grads = torch.autograd.grad((ctrl * dc).sum() + (traj * dt).sum(), (A, Bm, d, E, G), retain_graph=True)
    ref = eng.lmpc_vjp(dcontrol=dc.cpu().numpy(), dtrajectory=dt.cpu().numpy(), want=ALL)
    assert np.array_equal(grads[1].cpu().numpy(), ref["B"])
    assert np.array_equal(grads[3].cpu().numpy(), ref["E"][0])
    for got, r in ((grads[0], ref["A"]), (grads[2], ref["d"]), (grads[4], ref["G"][0])):
        np.testing.assert_allclose(got.cpu().numpy(), r.sum(0), rtol=1e-12, atol=1e-12 * np.abs(r).sum())
    inst = wl.instance(bp, 5)
    o = vr.solve(inst)
    dt5 = dt[5].cpu().numpy()
    cf, _ = mr.closed_form(inst, o, vr.adjoint(o, dc[5].cpu().numpy(), dt5), dt5)
    np.testing.assert_allclose(grads[1][5].cpu().numpy(), cf[("B", 0)], rtol=1e-8, atol=1e-8 * np.abs(cf[("B", 0)]).max())
    np.testing.assert_allclose(grads[3][5].cpu().numpy(), cf[("E", 0)], rtol=1e-8, atol=1e-8 * np.abs(cf[("E", 0)]).max())
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        Ad = fwAD.make_dual(A.detach(), torch.ones_like(A))
        with pytest.raises(NotImplementedError):
            ag.lmpc(eng, bp, x0, A=Ad)


def test_cpp_batched_lmpc_vjp_model():
    """BatchedLMPC::vjp with model outputs (tests/cpp/test_vjp_model.cpp) against central differences of copra::LMPC"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([os.path.join(root, "tests", "cpp", "test_vjp_model")], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
