"""copra_b200_lmpc_vjp_initial_state / copra_b200_lmpc_jvp_initial_state (K8 / K9 in initial-state mode) on the GPU: against
the dense numpy reference on every solver route an initial-state build takes, central differences of the GPU forward, LMPC
mode on the same problem, the adjoint identity, failed instances, repeatability, HOST / DEVICE, sharding, launch counts,
the error codes and torch.autograd."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import initial_state_sens_reference as ir
from tests.golden import make_golden as mg

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = capi.Engine(0)
    yield e
    e.close()


def c4(B=6, N=12, **kw):
    return wl.c4(batch=B, N=N, T=0.12 if N <= 20 else 0.03, **kw)


def single(inst):
    """a one-instance batch problem of an instance dict"""
    return dict(inst, batch=1, name="single")


def golden():
    return dict(mg.small_cases())["all_kinds_initial_state"]


def variant():
    """the golden initial-state fixture with an active finite lower position line on its trajectory bound (quirk Q1)"""
    v = golden()
    v["constraints"] = [dict(c) for c in v["constraints"]]
    v["x0lb"] = np.array([0.0, -1.5])
    v["constraints"][4] = dict(v["constraints"][4], lower=np.array([0.15, -np.inf]))
    return v


def _engine_grad(g, key, b):
    kind, i = key
    return g[kind][b] if i is None else g[kind][i][b]


def _cotangents(out, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=out["control"].shape), rng.normal(size=out["trajectory"].shape)


def _check_vjp(bp, out, g, dc, dt, instances, tol=1e-8):
    for b in instances:
        inst = wl.instance(bp, b)
        ref = ir.vjp(inst, dc[b], dt[b])
        scale = max(1.0, max(float(np.abs(v).max()) for v in ref.values() if np.size(v)))
        for key, r in ref.items():
            got = _engine_grad(g, key, b)
            assert np.abs(got - r).max() <= tol * scale, (key, b, got, r)


def _tangents(bp, B, k, rng):
    """{key: (batch, k, len)} random tangents of every input of the build (R included), 0 on infinite entries"""
    inst = wl.instance(bp, 0)
    out = {}
    for key in ir.vector_keys(inst):
        v = ir.get(inst, key)
        out[key] = np.where(np.isfinite(v)[None, None, :], rng.normal(size=(B, k, v.size)), 0.0)
    if bp.get("R") is not None:
        out[("R", None)] = rng.normal(size=(B, k, bp["nx"], bp["nx"]))
    return out


def _jvp_args(tangents):
    args = dict(p={}, f={}, lower={}, upper={})
    for (kind, i), t in tangents.items():
        if i is None:
            args[kind] = t
        else:
            args[kind][i] = t
    for kind in ("p", "f", "lower", "upper"):
        d = args[kind]
        args[kind] = [d.get(i) for i in range(max(d) + 1)] if d else None
    return args


def _check_jvp(bp, du, dx, tang, instances, d=0, tol=1e-8):
    for b in instances:
        inst = wl.instance(bp, b)
        ru, rx = ir.jvp(inst, {k: t[b, d].reshape(np.shape(ir.get(inst, k))) for k, t in tang.items()})
        scale = max(1.0, float(np.abs(ru).max()), float(np.abs(rx).max()))
        assert np.abs(du[b, d] - ru).max() <= tol * scale
        assert np.abs(dx[b, d] - rx).max() <= tol * scale


ROUTES = [("c4_small_v1", lambda: c4(), 1, "gi_small"), ("c4_small_v2", lambda: c4(), 2, "gi_small"),
          ("c4_small_v3", lambda: c4(), 3, "gi_small"), ("c4_n100_general", lambda: c4(B=4, N=100), 0, None),
          ("golden", lambda: single(golden()), 0, "gi_small"), ("variant", lambda: single(variant()), 0, "gi_small")]


@pytest.mark.parametrize("name,make,small_variant,solver", ROUTES, ids=[r[0] for r in ROUTES])
def test_matches_reference_on_every_route(name, make, small_variant, solver):
    bp = make()
    e = capi.Engine(0, small_variant=small_variant)
    try:
        out = e.lmpc_run(bp)
        assert (out["status"] == 0).all()
        if solver:
            assert solver in e.last_solver(), e.last_solver()
        else:
            assert "gi_small" not in e.last_solver() and "thin" not in e.last_solver(), e.last_solver()
        B = bp["batch"]
        dc, dt = _cotangents(out, 1)
        g = e.initial_state_vjp(dcontrol=dc, dtrajectory=dt)
        _check_vjp(bp, out, g, dc, dt, sorted({0, B - 1}))
        tang = _tangents(bp, B, 2, np.random.default_rng(2))
        du, dx = e.initial_state_jvp(**_jvp_args(tang))
        _check_jvp(bp, du, dx, tang, sorted({0, B - 1}), d=1)
        # the adjoint identity, on every instance
        lhs = sum(np.sum(_engine_grad(g, k, slice(None)).reshape(B, -1) * t[:, 0].reshape(B, -1), axis=1) for k, t in tang.items())
        rhs = np.sum(dc * du[:, 0], axis=1) + np.sum(dt * dx[:, 0], axis=1)
        np.testing.assert_allclose(lhs, rhs, rtol=1e-10, atol=1e-12 * np.abs(rhs).max())
    finally:
        e.close()


def test_matches_central_differences_of_the_gpu_forward(eng):
    bp = c4(B=4)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(out, 4)
    g = eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt)
    rng = np.random.default_rng(9)
    for key, h in ((("r", None), 1e-4), (("x0ub", None), 1e-4), (("p", 0), 1e-4), (("upper", 0), 1e-4), (("R", None), 1e-5)):
        kind, i = key
        base = np.asarray(bp[kind] if i is None else bp["costs" if kind == "p" else "constraints"][i][kind], float)
        full = np.broadcast_to(base, (4,) + base.shape[-(2 if kind == "R" else 1):]).copy()
        d = rng.normal(size=full.shape)
        loss = []
        for s in (h, -h):
            q = dict(bp, costs=[dict(c) for c in bp["costs"]], constraints=[dict(c) for c in bp["constraints"]])
            (q if i is None else q["costs" if kind == "p" else "constraints"][i])[kind] = full + s * d
            o = eng.lmpc_run(q)
            loss.append(np.sum(dc * o["control"], axis=1) + np.sum(dt * o["trajectory"], axis=1))
        fd = (loss[0] - loss[1]) / (2 * h)
        an = np.sum((_engine_grad(g, key, slice(None)) * d).reshape(4, -1), axis=1)
        np.testing.assert_allclose(an, fd, rtol=1e-6, atol=1e-6)


def test_pinned_bounds_match_lmpc_mode(eng):
    """default x0 bounds and R = I: x0* = x0, and the initial-state gradients with respect to x0 and the vectors equal those
    of copra_b200_lmpc_vjp on the same problem in LMPC mode; the JVP along the identity on x0 equals the feedback gain"""
    bp = c4(B=6)
    B, nx, N = bp["batch"], bp["nx"], bp["N"]
    ist = dict(bp, R=np.eye(nx), r=None, x0lb=None, x0ub=None)
    lm = {k: v for k, v in bp.items() if k not in ("R", "r", "x0lb", "x0ub")}
    lm["initial_state"] = False
    o_is = eng.lmpc_run(ist)
    dc, dt = _cotangents(o_is, 6)
    g_is = eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt)
    tx0 = np.broadcast_to(np.eye(nx)[None], (B, nx, nx)).copy()
    du, dx = eng.initial_state_jvp(x0=tx0)
    o_lm = eng.lmpc_run(lm)
    assert (o_is["status"] == 0).all() and (o_lm["status"] == 0).all()
    np.testing.assert_allclose(o_is["control"], o_lm["control"], rtol=0, atol=1e-8 * np.abs(o_lm["control"]).max())
    g_lm = eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)
    for key in ("x0", "p", "lower", "upper"):
        a, b = g_is[key], g_lm[key]
        for x, y in (zip(a, b) if isinstance(a, list) else [(a, b)]):
            if y is None:
                continue
            np.testing.assert_allclose(x, y, rtol=0, atol=1e-8 * max(1.0, np.abs(y).max()))
    ku, kx = eng.lmpc_feedback_gain(steps=N)
    np.testing.assert_allclose(du.transpose(0, 2, 1), ku, rtol=0, atol=1e-8 * max(1.0, np.abs(ku).max()))
    np.testing.assert_allclose(dx.transpose(0, 2, 1), kx, rtol=0, atol=1e-8 * max(1.0, np.abs(kx).max()))


def test_failed_instances_get_zeros(eng):
    bp = c4(B=4)
    x0lb, x0ub = np.array(bp["x0lb"]), np.array(bp["x0ub"])
    x0lb[1] = x0ub[1] + 1.0  # an empty x0 box
    R = np.broadcast_to(np.eye(2), (4, 2, 2)).copy()
    R[2] = -1e3 * np.eye(2)  # Q_tl not positive definite
    bp = dict(bp, x0lb=x0lb, R=R)
    out = eng.lmpc_run(bp)
    assert out["status"][1] != 0 and out["status"][2] == 2 and out["status"][0] == 0 and out["status"][3] == 0
    dc, dt = _cotangents(out, 8)
    g = eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt)
    tang = _tangents(bp, 4, 1, np.random.default_rng(8))
    du, dx = eng.initial_state_jvp(**_jvp_args(tang))
    for b in (1, 2):
        for k in ("x0", "R", "r", "x0lb", "x0ub"):
            assert not np.any(g[k][b])
        assert not np.any(g["p"][0][b]) and not np.any(g["upper"][0][b])
        assert not np.any(du[b]) and not np.any(dx[b])
    _check_vjp(bp, out, g, dc, dt, [0, 3])


def test_bitwise_repeatable_host_device_and_sharded(eng):
    torch = pytest.importorskip("torch")
    bp = c4(B=37)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(out, 10)
    tang = _tangents(bp, 37, 3, np.random.default_rng(10))
    g1 = eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt)
    g2 = eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt)
    j1 = eng.initial_state_jvp(**_jvp_args(tang))
    j2 = eng.initial_state_jvp(**_jvp_args(tang))
    gd = eng.initial_state_vjp(dcontrol=torch.from_numpy(dc).cuda(), dtrajectory=torch.from_numpy(dt).cuda())
    tt = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in tang.items()}
    jd = eng.initial_state_jvp(**_jvp_args(tt))

    def flat(g):
        return {k: (np.asarray(v.cpu() if hasattr(v, "cpu") else v) if not isinstance(v, list)
                    else [None if a is None else np.asarray(a.cpu() if hasattr(a, "cpu") else a) for a in v])
                for k, v in g.items()}

    def same(a, b):
        for k in a:
            x, y = a[k], b[k]
            for u, w in (zip(x, y) if isinstance(x, list) else [(x, y)]):
                assert (u is None and w is None) or np.array_equal(u, w), k
    same(flat(g1), flat(g2))
    same(flat(g1), flat(gd))
    for a, b, c in zip(j1, j2, jd):
        assert np.array_equal(a, b) and np.array_equal(a, c.cpu().numpy())
    for shards in (2, 4):
        m = capi.MultiEngine([0] * shards)
        try:
            m.lmpc_run(bp, eng.sizes(capi.HostBatch(bp)))
            same(flat(g1), flat(m.initial_state_vjp(dcontrol=dc, dtrajectory=dt)))
            for a, b in zip(j1, m.initial_state_jvp(**_jvp_args(tang))):
                assert np.array_equal(a, b)
        finally:
            m.close()


def test_launch_counts(eng):
    """the first call factors the build's per-instance Hessians (one gt_factor launch kept until the next build); after it the
    VJP with or without the R / r / x0 bound outputs and a JVP run the same launches"""
    bp = c4(B=8)
    out = eng.lmpc_run(bp)
    dc, dt = _cotangents(out, 12)
    tang = _tangents(bp, 8, 2, np.random.default_rng(12))
    counts = []
    for call in (lambda: eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt, want=("x0", "p")),
                 lambda: eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt, want=("x0", "p")),
                 lambda: eng.initial_state_vjp(dcontrol=dc, dtrajectory=dt),
                 lambda: eng.initial_state_jvp(**_jvp_args(tang))):
        n0 = eng.launch_count()
        call()
        counts.append(eng.launch_count() - n0)
    assert counts[0] == counts[1] + 1
    assert counts[1] == counts[2] == counts[3]


def _vjp_rc(e, init=None):
    return e.lib.copra_b200_lmpc_vjp_initial_state(e.h, None, None, capi.HOST, None, init and C.byref(init))


def _jvp_rc(e, ndir=1, init=None, null_in=False):
    t = capi.JvpIn()
    t.ndir = ndir
    return e.lib.copra_b200_lmpc_jvp_initial_state(e.h, None if null_in else C.byref(t), init and C.byref(init), capi.HOST,
                                                   None, None)


def test_error_codes():
    e = capi.Engine(0)
    try:
        assert _vjp_rc(e) == -5 and _jvp_rc(e) == -5  # nothing solved
        e.lmpc_run(wl.c2(batch=4))
        assert _vjp_rc(e) == -4 and _jvp_rc(e) == -4  # LMPC mode
        assert "copra_b200_lmpc_vjp" in e.lib.copra_b200_last_error(e.h).decode()
        bp = c4(B=4)
        e.lmpc_run(dict(bp, R=None, r=None))
        assert _vjp_rc(e) == 0 and _jvp_rc(e) == 0
        for key in ("R", "r"):
            o, t = capi.VjpInitialOut(), capi.JvpInitialIn()
            buf = np.zeros(4 * 4 * 2)
            setattr(o, key, buf.ctypes.data)
            setattr(t, key, buf.ctypes.data)
            assert _vjp_rc(e, o) == -1 and _jvp_rc(e, init=t) == -1  # not given to the build
        e.lmpc_run(dict(bp, x0lb=None, x0ub=None))
        for key in ("x0lb", "x0ub"):
            o = capi.VjpInitialOut()
            buf = np.zeros(4 * 2)
            setattr(o, key, buf.ctypes.data)
            assert _vjp_rc(e, o) == -1
        assert _jvp_rc(e, ndir=0) == -1 and _jvp_rc(e, null_in=True) == -1
        # full-size cost
        full = c4(B=4)
        full["costs"] = [dict(full["costs"][0]), dict(full["costs"][1], N=np.eye(12), p=np.zeros(12), w=np.full(12, 1e-2))]
        e.lmpc_run(full)
        assert _vjp_rc(e) == -4 and _jvp_rc(e) == -4
        # a raw QP batch since the solve
        e.lmpc_run(bp)
        n = 4
        e.solve_qp_batch(np.eye(n)[None], np.ones((1, n)), None, None, None, None, np.full((1, n), -10.0), np.full((1, n), 10.0))
        assert _vjp_rc(e) == -5 and _jvp_rc(e) == -5
    finally:
        e.close()


def test_lmpc_entry_points_unchanged_on_initial_state_builds(eng):
    eng.lmpc_run(c4(B=4))
    assert eng.lib.copra_b200_lmpc_vjp(eng.h, None, None, capi.HOST, C.byref(capi.VjpOut())) == -4
    assert eng.lib.copra_b200_lmpc_feedback_gain(eng.h, 1, None, None, capi.HOST) == -4


def test_torch_autograd():
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    from torch.autograd import forward_ad as fwAD
    e = capi.Engine(0)
    try:
        bp = c4(B=5)
        dev = torch.device("cuda", 0)
        B, nx = bp["batch"], bp["nx"]
        x0 = torch.tensor(np.asarray(bp["x0"]), device=dev)
        R = torch.tensor(np.eye(nx) * 1.5, device=dev, requires_grad=True)  # shared
        r = torch.tensor(np.asarray(bp["r"]), device=dev, requires_grad=True)
        lb = torch.tensor(np.asarray(bp["x0lb"]), device=dev, requires_grad=True)
        ub = torch.tensor(np.asarray(bp["x0ub"]), device=dev, requires_grad=True)
        p0 = torch.tensor(np.asarray(bp["costs"][0]["p"]), device=dev, requires_grad=True)
        ctrl, traj = ag.initial_state_lmpc(e, bp, x0, R=R, r=r, x0lb=lb, x0ub=ub, p=[p0])
        dc, dt = torch.randn_like(ctrl), torch.randn_like(traj)
        (dc * ctrl).sum().add((dt * traj).sum()).backward()
        # the engine on the same build, with R tiled per instance: a shared R's gradient is the batch sum
        q = dict(bp, R=np.broadcast_to(np.eye(nx) * 1.5, (B, nx, nx)).copy())
        e.lmpc_run(q)
        g = e.initial_state_vjp(dcontrol=dc.cpu().numpy(), dtrajectory=dt.cpu().numpy())
        np.testing.assert_allclose(R.grad.cpu().numpy(), g["R"].sum(0), rtol=1e-10, atol=1e-12)
        for t, k in ((r, "r"), (lb, "x0lb"), (ub, "x0ub")):
            np.testing.assert_allclose(t.grad.cpu().numpy(), g[k], rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(p0.grad.cpu().numpy(), g["p"][0], rtol=1e-10, atol=1e-12)
        # forward mode against initial_state_jvp
        tr = torch.randn_like(r)
        tR = torch.randn(nx, nx, dtype=torch.float64, device=dev)
        with fwAD.dual_level():
            c2, t2 = ag.initial_state_lmpc(e, bp, x0, R=fwAD.make_dual(R.detach(), tR), r=fwAD.make_dual(r.detach(), tr),
                                           x0lb=lb.detach(), x0ub=ub.detach(), p=[p0.detach()])
            jc, jt = fwAD.unpack_dual(c2).tangent, fwAD.unpack_dual(t2).tangent
        du, dx = e.initial_state_jvp(R=tR.expand(B, nx, nx).unsqueeze(1).cpu().numpy(), r=tr.unsqueeze(1).cpu().numpy())
        np.testing.assert_allclose(jc.cpu().numpy(), du[:, 0], rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(jt.cpu().numpy(), dx[:, 0], rtol=1e-12, atol=1e-14)
    finally:
        e.close()
