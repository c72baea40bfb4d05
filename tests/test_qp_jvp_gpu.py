"""copra_b200_qp_jvp / copra_b200_qp_jacobian (Engine.qp_jvp, Engine.qp_jacobian) on the GPU: every raw-QP solver route
against the dense reference of tests/qp_jvp_reference.py, adjointness with the GPU's own qp_vjp, finite differences of the
GPU forward, the Jacobians, direction independence, failed instances, chunking, determinism, HOST / DEVICE memory, stride-0
tangents, launch counts, isolation from a resident LMPC build and from qp_vjp, and error codes."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import qp_jvp_reference as jr
from tests import qp_vjp_reference as qr
from tests.test_qp_vjp_gpu import _downloaded, random_batch, stack
from tests.util import active_set

pytestmark = pytest.mark.gpu

KEYS = qr.KEYS
WRT = ("c", "beq", "bineq", "lb", "ub")


def tangents(ps, k, seed, keys=KEYS):
    """k random directions per instance over `keys`: {key: (batch, k, *shape)} (0 on infinite bounds; Q not symmetrised, the
    engine reads its symmetric part)"""
    rng = np.random.default_rng(seed)
    out = {}
    for key in keys:
        if not ps[0][key].size:
            continue
        t = rng.normal(size=(len(ps), k) + ps[0][key].shape)
        if key in ("lb", "ub"):
            t = np.where(np.stack([np.isfinite(p[key]) for p in ps])[:, None], t, 0.0)
        out[key] = t
    return out


def one(t, b, d):
    return {key: v[b, d] for key, v in t.items()}


def check_reference(engine, ps, solver, tol=1e-8, k=2):
    """each direction's xdot within `tol` of the reference, relative to the direction's largest entry"""
    r = engine.solve_qp_batch(*stack(ps))
    assert engine.last_solver() == solver
    t = tangents(ps, k, 3)
    got = engine.qp_jvp(**t)
    assert got.shape == (len(ps), k, ps[0]["Q"].shape[0])
    worst = 0.0
    for b, p in enumerate(ps):
        o = qr.solve(p)
        assert r["status"][b] == o["fail"] == 0
        assert active_set(r["iact"][b], r["nact"][b]) == active_set(o["iact"]), b
        for d in range(k):
            ref = jr.jvp(o, one(t, b, d))
            e = float(np.abs(got[b, d] - ref).max() / max(np.abs(ref).max(), 1e-300))
            worst = max(worst, e)
            assert e <= tol, (solver, b, d, e)
    print(solver, ps[0]["Q"].shape[0], "worst rel err %.2e" % worst)


@pytest.mark.parametrize("variant", [1, 2, 3])
def test_gi_small_matches_reference(variant):
    eng = capi.Engine(0, small_variant=variant)
    try:
        for n, meq, m in ((10, 2, 12), (24, 0, 30), (40, 3, 50)):
            check_reference(eng, random_batch(300 + n + variant, n, meq, m, 4), "gi_small_kernel")
    finally:
        eng.close()


@pytest.mark.parametrize("n,meq,m", [(65, 4, 40), (100, 0, 120), (160, 3, 64)])
def test_general_kernel_matches_reference(engine, n, meq, m):
    check_reference(engine, random_batch(400 + n, n, meq, m, 3), "gi_batch_kernel")


def test_cluster_kernel_matches_reference(engine):
    check_reference(engine, random_batch(503, 203, 5, 150, 2), "gi_cluster_kernel")


def test_c5_downloaded_qp_through_the_general_kernel(engine):
    check_reference(engine, [_downloaded(engine, wl.c5(batch=1))], "gi_batch_kernel", k=1)


def test_adjoint_of_the_gpu_vjp(engine):
    """<w, xdot_d> = sum_k <g_k, t_k,d> with g the GPU's qp_vjp of w, all eight tangents at once, k = 3"""
    ps = random_batch(31, 18, 2, 20, 5)
    engine.solve_qp_batch(*stack(ps))
    t = tangents(ps, 3, 32)
    xd = engine.qp_jvp(**t)
    w = np.random.default_rng(33).normal(size=(5, 18))
    g = engine.qp_vjp(w)
    for b in range(5):
        for d in range(3):
            lhs = float(w[b] @ xd[b, d])
            rhs = float(sum(np.sum(g[key][b] * t[key][b, d]) for key in t))
            assert abs(lhs - rhs) <= 1e-10 * max(1.0, abs(lhs), abs(rhs)), (b, d, lhs, rhs)


def test_gpu_forward_differences(engine):
    """central differences of the GPU forward along a random direction of each input agree with the GPU JVP"""
    ps = random_batch(34, 12, 2, 14, 4)
    args = stack(ps)
    r0 = engine.solve_qp_batch(*args)
    t = tangents(ps, 1, 35)
    t["Q"] = 0.5 * (t["Q"] + np.swapaxes(t["Q"], -1, -2))  # the solver reads Q as symmetric: move it along symmetric directions
    for i, key in enumerate(KEYS):
        engine.solve_qp_batch(*args)
        xd = engine.qp_jvp(**{key: t[key]})[:, 0]
        h = 1e-4 if key in ("c", "beq", "bineq", "lb", "ub") else 1e-6
        ends = []
        for s in (1.0, -1.0):
            a = list(args)
            a[i] = args[i] + s * h * t[key][:, 0]
            r = engine.solve_qp_batch(*a)
            assert np.array_equal(r["iact"], r0["iact"]) and np.array_equal(r["nact"], r0["nact"])
            ends.append(r["x"])
        fd = (ends[0] - ends[1]) / (2 * h)
        assert np.abs(xd - fd).max() <= 1e-6 * max(1.0, np.abs(fd).max()), (key, np.abs(xd - fd).max())


def test_jacobians(engine):
    """each Jacobian is qp_jvp along the identity columns (bitwise) and matches the reference; dx/dc is symmetric; the
    columns of inactive rows are exactly zero"""
    ps = random_batch(36, 16, 2, 22, 3)
    engine.solve_qp_batch(*stack(ps))
    n = 16
    for wrt in WRT:
        J = engine.qp_jacobian(wrt)
        ln = ps[0][wrt].shape[0]
        assert J.shape == (3, n, ln)
        xd = engine.qp_jvp(**{wrt: np.eye(ln)})
        assert np.array_equal(J, xd.transpose(0, 2, 1)), wrt
        for b, p in enumerate(ps):
            o = qr.solve(p)
            ref = jr.jacobian(o, wrt)
            assert np.abs(J[b] - ref).max() <= 1e-8 * max(np.abs(ref).max(), 1e-300), (wrt, b)
            if wrt == "c":
                assert np.abs(J[b] - J[b].T).max() <= 1e-12 * np.abs(J[b]).max(), b
            else:
                assert not np.delete(J[b], jr.active_rows(o, wrt), axis=1).any(), (wrt, b)


def test_directions_are_independent(engine):
    """direction d of a k = 5 call equals a k = 1 call along it"""
    ps = random_batch(37, 20, 2, 25, 4)
    engine.solve_qp_batch(*stack(ps))
    t = tangents(ps, 5, 38)
    all5 = engine.qp_jvp(**t)
    for d in range(5):
        single = engine.qp_jvp(**{key: v[:, d:d + 1] for key, v in t.items()})[:, 0]
        assert np.allclose(all5[:, d], single, rtol=0, atol=1e-12 * max(1.0, np.abs(single).max())), d


def test_failed_instances_get_zeros():
    """an infeasible (status 1) and a non-convex (status 2) instance inside a batch: zeros, the others unaffected"""
    good = random_batch(9, 2, 0, 2, 2)
    bad1 = qr.problem(np.eye(2), np.zeros(2), Aineq=np.array([[1.0, 0.0], [-1.0, 0.0]]), bineq=np.array([-1.0, -1.0]))
    bad2 = qr.problem(np.array([[1.0, 2.0], [2.0, 1.0]]), np.zeros(2), Aineq=np.zeros((2, 2)), bineq=np.ones(2),
                      lb=np.full(2, -1.0), ub=np.full(2, 1.0))
    for p in good:
        p["lb"], p["ub"] = np.full(2, -10.0), np.full(2, 10.0)
    batch = [good[0], bad1, bad2, good[1]]
    t = tangents(batch, 2, 39)
    eng = capi.Engine(0)
    try:
        r = eng.solve_qp_batch(*stack(batch))
        assert list(r["status"]) == [0, 1, 2, 0]
        xd = eng.qp_jvp(**t)
        J = eng.qp_jacobian("c")
        eng.solve_qp_batch(*stack(good))
        ref = eng.qp_jvp(**{key: v[[0, 3]] for key, v in t.items()})
        Jref = eng.qp_jacobian("c")
    finally:
        eng.close()
    assert not xd[1:3].any() and not J[1:3].any()
    assert np.allclose(xd[[0, 3]], ref, rtol=1e-12, atol=1e-14)
    assert np.allclose(J[[0, 3]], Jref, rtol=1e-12, atol=1e-14)


def test_chunks_match_a_small_batch():
    """a batch whose KKT workspace spans several chunks (per-instance Q, so the factor is made per chunk) gives, bitwise, the
    JVP of the same instances solved as a small batch"""
    n, B = 64, 12000
    rng = np.random.default_rng(12)
    L = rng.normal(size=(n, n))
    Q0 = L @ L.T / n + 0.5 * np.eye(n)
    Q = np.broadcast_to(Q0, (B, n, n)) + np.eye(n) * rng.uniform(0.0, 1.0, size=(B, 1, 1))
    c = rng.normal(size=(B, n))
    Aineq = rng.normal(size=(48, n))
    bineq = rng.uniform(0.0, 0.5, size=(B, 48))
    lb, ub = np.full((B, n), -0.2), np.full((B, n), 0.2)
    tc, tb = rng.normal(size=(B, 1, n)), rng.normal(size=(B, 1, 48))
    eng = capi.Engine(0)
    try:
        r = eng.solve_qp_batch(Q, c, None, None, Aineq, bineq, lb, ub)
        assert (r["status"] == 0).all()
        n0 = eng.launch_count()
        xd = eng.qp_jvp(c=tc, bineq=tb)
        launches = eng.launch_count() - n0
        idx = [0, 1, B // 2, B - 1]
        eng.solve_qp_batch(Q[idx], c[idx], None, None, Aineq, bineq[idx], lb[idx], ub[idx])
        small = eng.qp_jvp(c=tc[idx], bineq=tb[idx])
    finally:
        eng.close()
    # per chunk: factor of Q, qp_tangent, Y GEMM, Gram GEMM, sens_gram, Gram factor, sens_solve, V GEMM, qp_output
    assert launches >= 2 * 9 and launches % 9 == 0, launches
    assert np.array_equal(xd[idx], small)


def test_host_device_and_repeated_calls_are_bitwise_equal(engine):
    torch = pytest.importorskip("torch")
    ps = random_batch(40, 30, 3, 40, 6)
    args = stack(ps)
    t = tangents(ps, 3, 41)
    engine.solve_qp_batch(*args)
    a, b = engine.qp_jvp(**t), engine.qp_jvp(**t)
    Ja = engine.qp_jacobian("bineq")
    dev = torch.device("cuda:0")
    engine.solve_qp_batch(*[None if x is None else torch.tensor(x, device=dev) for x in args])
    d = engine.qp_jvp(**{key: torch.tensor(v, device=dev) for key, v in t.items()})
    Jd = engine.qp_jacobian("bineq", device=dev)
    assert isinstance(d, torch.Tensor) and isinstance(Jd, torch.Tensor)
    assert np.array_equal(a, b)
    assert np.array_equal(a, d.cpu().numpy())
    assert np.array_equal(Ja, Jd.cpu().numpy())


def test_stride0_tangent_matches_its_tiled_copy(engine):
    ps = random_batch(42, 16, 1, 20, 5)
    engine.solve_qp_batch(*stack(ps))
    t = tangents(ps[:1], 2, 43)
    shared = {key: v[0] for key, v in t.items()}
    tiled = {key: np.repeat(v, 5, axis=0) for key, v in t.items()}
    assert np.array_equal(engine.qp_jvp(**shared), engine.qp_jvp(**tiled))


def test_launch_counts(engine):
    """one chunk: 9 launches without Aeq / Aineq tangents (factor of Q, qp_tangent, Y GEMM, Gram GEMM, sens_gram, Gram factor,
    sens_solve, V GEMM, qp_output), 18 with them (the same nine of the lambda pass, qp_lambda_gather and qp_lambda_store at the
    ends, first); the k = 1 JVP along c alone is bitwise the same either way it is asked for"""
    ps = random_batch(44, 20, 2, 25, 5)
    engine.solve_qp_batch(*stack(ps))
    t = tangents(ps, 2, 45)
    counts = []
    for kw in ({key: t[key] for key in ("Q", "c", "beq", "bineq", "lb", "ub")}, t, {"Aineq": t["Aineq"]}):
        n0 = engine.launch_count()
        engine.qp_jvp(**kw)
        counts.append(engine.launch_count() - n0)
    n0 = engine.launch_count()
    engine.qp_jacobian("c")
    counts.append(engine.launch_count() - n0)
    assert counts == [9, 18, 18, 9], counts


def _lmpc_sequence(bp, with_qp_jvp):
    eng = capi.Engine(0)
    try:
        out = eng.lmpc_run(bp)
        ps = random_batch(16, 12, 1, 10, 3)
        eng.solve_qp_batch(*stack(ps))
        if with_qp_jvp:
            eng.qp_jvp(**tangents(ps, 2, 46))
        B = bp["batch"]
        x0 = np.asarray(bp["x0"], float) * 0.9 if np.ndim(bp["x0"]) == 2 else np.tile(np.asarray(bp["x0"], float) * 0.9, (B, 1))
        r = eng.lmpc_resolve(x0, out["sizes"])
        g = eng.lmpc_vjp(dcontrol=np.ones((B, out["sizes"]["nU"])))
        return r, g
    finally:
        eng.close()


@pytest.mark.parametrize("name", ["C2", "C3"])
def test_isolation_from_the_lmpc_build(name):
    """lmpc_run, solve_qp_batch, qp_jvp, lmpc_resolve, lmpc_vjp: bitwise the results of the same sequence without qp_jvp"""
    bp = wl.c2(batch=8) if name == "C2" else wl.c3(batch=8)
    r0, g0 = _lmpc_sequence(bp, False)
    r1, g1 = _lmpc_sequence(bp, True)
    for k in r0:
        assert np.array_equal(r0[k], r1[k]), k
    assert np.array_equal(g0["x0"], g1["x0"])
    for k in ("p", "f", "lower", "upper"):
        for a, b in zip(g0[k], g1[k]):
            assert (a is None and b is None) or np.array_equal(a, b), k


def test_qp_vjp_after_qp_jvp_is_unchanged(engine):
    ps = random_batch(47, 14, 2, 16, 4)
    dx = np.random.default_rng(48).normal(size=(4, 14))
    engine.solve_qp_batch(*stack(ps))
    g0 = engine.qp_vjp(dx)
    engine.solve_qp_batch(*stack(ps))
    engine.qp_jvp(**tangents(ps, 3, 49))
    engine.qp_jacobian("c")
    g1 = engine.qp_vjp(dx)
    for k in KEYS:
        assert np.array_equal(g0[k], g1[k]), k


def _jvp_rc(eng, ndir=1, dx=True, **given):
    t = capi.QpJvpIn()
    t.ndir = ndir
    buf = np.zeros(1 << 16)
    for k, stride in given.items():
        a = getattr(t, k)
        a.ptr, a.stride = buf.ctypes.data, stride
    out = np.zeros(1 << 16)
    return eng.lib.copra_b200_qp_jvp(eng.h, C.byref(t), capi.HOST, out.ctypes.data if dx else None)


def test_error_codes():
    eng = capi.Engine(0)
    J = np.zeros(1 << 12)
    try:
        assert _jvp_rc(eng, c=0) == -5  # no solve yet
        assert eng.lib.copra_b200_qp_jacobian(eng.h, 0, J.ctypes.data, capi.HOST) == -5
        ps = random_batch(17, 6, 0, 0, 2)
        eng.solve_qp_batch(*stack(ps))
        assert _jvp_rc(eng, c=0) == 0 and _jvp_rc(eng, ndir=3, c=18, lb=0) == 0
        assert _jvp_rc(eng, dx=False, c=0) == 0  # NULL dx
        assert eng.lib.copra_b200_qp_jvp(eng.h, None, capi.HOST, J.ctypes.data) == -1  # NULL in
        assert _jvp_rc(eng, ndir=0, c=0) == -1
        assert _jvp_rc(eng, c=-6) == -1
        for k in ("Aeq", "beq", "Aineq", "bineq"):
            assert _jvp_rc(eng, **{k: 0}) == -1, k  # meq = m = 0
        for wrt in (1, 2, 5, -1):
            assert eng.lib.copra_b200_qp_jacobian(eng.h, wrt, J.ctypes.data, capi.HOST) == -1, wrt
        for wrt in (0, 3, 4):
            assert eng.lib.copra_b200_qp_jacobian(eng.h, wrt, J.ctypes.data, capi.HOST) == 0, wrt
        assert eng.lib.copra_b200_qp_jacobian(eng.h, 0, None, capi.HOST) == 0  # NULL J
        bp = wl.c2(batch=2)
        eng.lmpc_run(bp)
        assert _jvp_rc(eng, c=0) == -5  # an LMPC run since
        assert eng.lib.copra_b200_qp_jacobian(eng.h, 0, J.ctypes.data, capi.HOST) == -5
    finally:
        eng.close()
