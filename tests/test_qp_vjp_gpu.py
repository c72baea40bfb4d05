"""copra_b200_qp_vjp (Engine.qp_vjp, copra_b200.autograd.qp) on the GPU: every raw-QP solver route against the dense
reference of tests/qp_vjp_reference.py, finite differences of the GPU forward, failed instances, chunking, determinism,
HOST / DEVICE memory, the launches of the k = 1 call, stride-0 inputs, isolation from a resident LMPC build, error codes and
torch.autograd."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import qp_vjp_reference as qr
from tests.util import active_set

pytestmark = pytest.mark.gpu

KEYS = qr.KEYS


def stack(ps):
    """a list of qr.problem dicts -> solve_qp_batch arguments (every input per instance; None for absent rows)"""
    meq, m = ps[0]["Aeq"].shape[0], ps[0]["Aineq"].shape[0]
    args = [np.stack([p[k] for p in ps]) for k in KEYS]
    if meq == 0:
        args[2] = args[3] = None
    if m == 0:
        args[4] = args[5] = None
    return args


def random_batch(seed, n, meq, m, B):
    rng = np.random.default_rng(seed)
    return [qr.random_qp(rng, n, meq, m) for _ in range(B)]


def check_reference(engine, ps, solver, tol=1e-8):
    """each gradient within `tol` of the reference, relative to its largest entry or, when that is at roundoff level (an
    instance with n active rows has v = 0, hence dc = dQ = 0 up to roundoff), to 1e-6 of the instance's largest gradient"""
    r = engine.solve_qp_batch(*stack(ps))
    assert engine.last_solver() == solver
    n = ps[0]["Q"].shape[0]
    dx = np.random.default_rng(3).normal(size=(len(ps), n))
    g = engine.qp_vjp(dx)
    worst = 0.0
    for b, p in enumerate(ps):
        o = qr.solve(p)
        assert r["status"][b] == o["fail"] == 0
        assert active_set(r["iact"][b], r["nact"][b]) == active_set(o["iact"]), b
        ref = qr.closed_form(o, dx[b])
        top = max(np.abs(ref[k]).max() if ref[k].size else 0.0 for k in KEYS)
        for k in KEYS:
            if not ref[k].size:
                continue
            e = float(np.abs(g[k][b] - ref[k]).max() / max(np.abs(ref[k]).max(), 1e-6 * top))
            worst = max(worst, e)
            assert e <= tol, (solver, b, k, e)
    print(solver, n, "worst rel err %.2e" % worst)


@pytest.mark.parametrize("variant", [1, 2, 3])
def test_gi_small_matches_reference(variant):
    eng = capi.Engine(0, small_variant=variant)
    try:
        for n, meq, m in ((10, 2, 12), (24, 0, 30), (40, 3, 50)):
            check_reference(eng, random_batch(100 + n + variant, n, meq, m, 4), "gi_small_kernel")
    finally:
        eng.close()


@pytest.mark.parametrize("n,meq,m", [(65, 4, 40), (100, 0, 120), (160, 3, 64)])
def test_general_kernel_matches_reference(engine, n, meq, m):
    check_reference(engine, random_batch(200 + n, n, meq, m, 3), "gi_batch_kernel")


def test_cluster_kernel_matches_reference(engine):
    check_reference(engine, random_batch(203, 203, 5, 150, 2), "gi_cluster_kernel")


def _downloaded(engine, bp):
    hb = capi.HostBatch(bp)
    engine.lmpc_run(hb)
    st = {k: engine.download(hb, k)[0] for k in ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")}
    return qr.problem(st["Q"], st["c"], st["Aeq"] if st["Aeq"].size else None, st["beq"] if st["beq"].size else None,
                      st["Aineq"], st["bineq"], st["lb"], st["ub"])


def test_c5_downloaded_qp_through_the_general_kernel(engine):
    check_reference(engine, [_downloaded(engine, wl.c5(batch=1))], "gi_batch_kernel")


def test_gpu_forward_differences(engine):
    """central differences of the GPU forward along a random direction of each input agree with the GPU VJP"""
    ps = random_batch(7, 12, 2, 14, 4)
    args = stack(ps)
    rng = np.random.default_rng(8)
    dx = rng.normal(size=(4, 12))
    r0 = engine.solve_qp_batch(*args)
    g = engine.qp_vjp(dx)
    for i, k in enumerate(KEYS):
        d = rng.normal(size=args[i].shape)
        if k == "Q":
            d = 0.5 * (d + np.swapaxes(d, 1, 2))
        if k in ("lb", "ub"):
            d = np.where(np.isfinite(args[i]), d, 0.0)
        h = 1e-4 if k in ("c", "beq", "bineq", "lb", "ub") else 1e-6
        ends = []
        for s in (1.0, -1.0):
            a = list(args)
            a[i] = args[i] + s * h * d
            r = engine.solve_qp_batch(*a)
            assert np.array_equal(r["iact"], r0["iact"]) and np.array_equal(r["nact"], r0["nact"])
            ends.append(np.sum(dx * r["x"]))
        fd = (ends[0] - ends[1]) / (2 * h)
        got = float(np.sum(g[k] * d))
        assert abs(got - fd) <= 1e-6 * max(1.0, abs(fd)), (k, got, fd)


def test_failed_instances_get_zeros():
    """an infeasible (status 1) and a non-convex (status 2) instance inside a batch: zeros, the others unaffected"""
    good = random_batch(9, 2, 0, 2, 2)
    bad1 = qr.problem(np.eye(2), np.zeros(2), Aineq=np.array([[1.0, 0.0], [-1.0, 0.0]]), bineq=np.array([-1.0, -1.0]))
    bad2 = qr.problem(np.array([[1.0, 2.0], [2.0, 1.0]]), np.zeros(2), Aineq=np.zeros((2, 2)), bineq=np.ones(2),
                      lb=np.full(2, -1.0), ub=np.full(2, 1.0))
    for p in good:
        p["lb"], p["ub"] = np.full(2, -10.0), np.full(2, 10.0)
    eng = capi.Engine(0)
    try:
        dx = np.random.default_rng(2).normal(size=(4, 2))
        r = eng.solve_qp_batch(*stack([good[0], bad1, bad2, good[1]]))
        assert list(r["status"]) == [0, 1, 2, 0]
        g = eng.qp_vjp(dx)
        eng.solve_qp_batch(*stack(good))
        ref = eng.qp_vjp(dx[[0, 3]])
    finally:
        eng.close()
    for k in KEYS:
        assert not g[k][1:3].any(), k
        assert np.allclose(g[k][[0, 3]], ref[k], rtol=1e-12, atol=1e-14), k


def test_two_chunks_match_a_small_batch():
    """a batch whose KKT workspace spans several chunks (per-instance Q, so the factor is made per chunk) gives, bitwise, the
    gradients of the same instances solved as a small batch"""
    n, B = 64, 12000
    rng = np.random.default_rng(12)
    L = rng.normal(size=(n, n))
    Q0 = L @ L.T / n + 0.5 * np.eye(n)
    Q = np.broadcast_to(Q0, (B, n, n)) + np.eye(n) * rng.uniform(0.0, 1.0, size=(B, 1, 1))
    c = rng.normal(size=(B, n))
    Aineq = rng.normal(size=(48, n))
    bineq = rng.uniform(0.0, 0.5, size=(B, 48))
    lb, ub = np.full((B, n), -0.2), np.full((B, n), 0.2)
    dx = rng.normal(size=(B, n))
    eng = capi.Engine(0)
    try:
        r = eng.solve_qp_batch(Q, c, None, None, Aineq, bineq, lb, ub)
        assert (r["status"] == 0).all()
        n0 = eng.launch_count()
        g = eng.qp_vjp(dx)
        launches = eng.launch_count() - n0
        idx = [0, 1, B // 2, B - 1]
        eng.solve_qp_batch(Q[idx], c[idx], None, None, Aineq, bineq[idx], lb[idx], ub[idx])
        small = eng.qp_vjp(dx[idx])
    finally:
        eng.close()
    # per chunk: factor of Q, gather, Y GEMM, Gram GEMM, sens_gram, Gram factor, sens_solve, V GEMM, qp_grad
    assert launches >= 2 * 9 and launches % 9 == 0, launches
    for k in KEYS:
        assert np.array_equal(g[k][idx], small[k]), k


def test_repeated_host_and_device_calls_are_bitwise_equal(engine):
    torch = pytest.importorskip("torch")
    ps = random_batch(13, 30, 3, 40, 6)
    args = stack(ps)
    dx = np.random.default_rng(4).normal(size=(6, 30))
    engine.solve_qp_batch(*args)
    a, b = engine.qp_vjp(dx), engine.qp_vjp(dx)
    dev = torch.device("cuda:0")
    t = [None if x is None else torch.tensor(x, device=dev) for x in args]
    rd = engine.solve_qp_batch(*t)
    assert isinstance(rd["x"], torch.Tensor)
    d = engine.qp_vjp(torch.tensor(dx, device=dev))
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(a[k], d[k].cpu().numpy()), k


def test_without_row_matrices_k1_is_bitwise_and_launches_nothing_extra(engine):
    ps = random_batch(14, 20, 2, 25, 5)
    engine.solve_qp_batch(*stack(ps))
    dx = np.random.default_rng(5).normal(size=(5, 20))
    n0 = engine.launch_count()
    full = engine.qp_vjp(dx)
    n1 = engine.launch_count()
    part = engine.qp_vjp(dx, want=("Q", "c", "beq", "bineq", "lb", "ub"))
    n2 = engine.launch_count()
    assert part["Aeq"] is None and part["Aineq"] is None
    for k in ("Q", "c", "beq", "bineq", "lb", "ub"):
        assert np.array_equal(full[k], part[k]), k
    # one chunk: factor of Q, gather, Y GEMM, Gram GEMM, sens_gram, Gram factor, sens_solve, V GEMM, qp_grad
    assert n1 - n0 == n2 - n1 == 9


def test_stride0_q_matches_tiled_q(engine):
    ps = random_batch(15, 16, 1, 20, 5)
    for p in ps[1:]:
        p["Q"] = ps[0]["Q"]
    args = stack(ps)
    dx = np.random.default_rng(6).normal(size=(5, 16))
    engine.solve_qp_batch(*args)
    tiled = engine.qp_vjp(dx)
    shared = list(args)
    shared[0] = ps[0]["Q"]
    engine.solve_qp_batch(*shared)
    one = engine.qp_vjp(dx)
    for k in KEYS:
        assert one[k].shape == tiled[k].shape
        assert np.allclose(one[k], tiled[k], rtol=1e-12, atol=1e-12 * max(1.0, np.abs(tiled[k]).max())), k


def _lmpc_sequence(bp, with_qp_vjp):
    eng = capi.Engine(0)
    try:
        out = eng.lmpc_run(bp)
        ps = random_batch(16, 12, 1, 10, 3)
        eng.solve_qp_batch(*stack(ps))
        if with_qp_vjp:
            eng.qp_vjp(np.ones((3, 12)))
        B = bp["batch"]
        x0 = np.asarray(bp["x0"], float) * 0.9 if np.ndim(bp["x0"]) == 2 else np.tile(np.asarray(bp["x0"], float) * 0.9, (B, 1))
        r = eng.lmpc_resolve(x0, out["sizes"])
        g = eng.lmpc_vjp(dcontrol=np.ones((B, out["sizes"]["nU"])))
        return r, g
    finally:
        eng.close()


@pytest.mark.parametrize("name", ["C2", "C3"])
def test_isolation_from_the_lmpc_build(name):
    """lmpc_run, solve_qp_batch, qp_vjp, lmpc_resolve, lmpc_vjp: bitwise the results of the same sequence without qp_vjp
    (the resident build's factors and caches are not the raw-QP VJP's workspace)"""
    bp = wl.c2(batch=8) if name == "C2" else wl.c3(batch=8)
    r0, g0 = _lmpc_sequence(bp, False)
    r1, g1 = _lmpc_sequence(bp, True)
    for k in r0:
        assert np.array_equal(r0[k], r1[k]), k
    assert np.array_equal(g0["x0"], g1["x0"])
    for k in ("p", "f", "lower", "upper"):
        for a, b in zip(g0[k], g1[k]):
            assert (a is None and b is None) or np.array_equal(a, b), k


def _qp_rc(eng, dx=True, **want):
    o = capi.QpVjpOut()
    bufs = {k: np.zeros(4096) for k in want}
    for k, a in bufs.items():
        setattr(o, k, a.ctypes.data)
    d = np.zeros(4096)
    return eng.lib.copra_b200_qp_vjp(eng.h, d.ctypes.data if dx else None, capi.HOST, C.byref(o))


def test_error_codes():
    eng = capi.Engine(0)
    try:
        assert _qp_rc(eng, c=1) == -5  # no solve yet
        ps = random_batch(17, 6, 0, 0, 2)
        eng.solve_qp_batch(*stack(ps))
        assert _qp_rc(eng, c=1) == 0 and _qp_rc(eng) == 0
        assert eng.lib.copra_b200_qp_vjp(eng.h, np.zeros(12).ctypes.data, capi.HOST, None) == 0  # NULL out
        assert _qp_rc(eng, dx=False, c=1) == -1
        for k in ("Aeq", "beq", "Aineq", "bineq"):
            assert _qp_rc(eng, **{k: 1}) == -1, k  # meq = m = 0
        out = capi.VjpOut()
        assert eng.lib.copra_b200_lmpc_vjp(eng.h, None, None, capi.HOST, C.byref(out)) == -5  # a raw QP batch, not an LMPC
        bp = wl.c2(batch=2)
        eng.lmpc_run(bp)
        assert _qp_rc(eng, c=1) == -5  # an LMPC run since
        eng.solve_qp_batch(*stack(ps))
        assert _qp_rc(eng, c=1) == 0
        eng.lmpc_retarget(bp)
        assert _qp_rc(eng, c=1) == -5  # a retarget since
    finally:
        eng.close()


def test_torch_autograd_matches_qp_vjp(engine):
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(18)
    B, n = 5, 14
    ps = random_batch(18, n, 2, 16, B)
    for p in ps:  # Q, Aineq and ub shared by the batch, x = 0 feasible for every instance
        p["Q"], p["Aineq"], p["ub"] = ps[0]["Q"], ps[0]["Aineq"], np.full(n, 0.8)
        p["beq"], p["bineq"] = np.zeros(2), rng.uniform(0.1, 1.0, size=16)
        p["lb"] = -rng.uniform(0.5, 1.5, size=n)
    t = {k: torch.tensor(np.stack([p[k] for p in ps]), device=dev, requires_grad=True) for k in KEYS}
    for k in ("Q", "Aineq", "ub"):  # shared by the batch: stride 0, the gradient sums the instances'
        t[k] = torch.tensor(ps[0][k], device=dev, requires_grad=True)
    w = torch.tensor(np.random.default_rng(7).normal(size=(B, 14)), device=dev)
    x, status = ag.qp(engine, **t)
    assert not status.requires_grad and (status == 0).all()
    (w * x).sum().backward()
    ref = engine.qp_vjp(w)
    for k in KEYS:
        want = ref[k].sum(0) if k in ("Q", "Aineq", "ub") else ref[k]
        assert torch.equal(t[k].grad, want), k
    # a stale backward
    x, _ = ag.qp(engine, **{k: v.detach().requires_grad_() for k, v in t.items()})
    engine.solve_qp_batch(*stack(ps))
    with pytest.raises(RuntimeError, match="another solve ran"):
        x.sum().backward()
    # forward mode
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        c = fwAD.make_dual(t["c"].detach(), torch.ones_like(t["c"]))
        with pytest.raises(NotImplementedError):
            ag.qp(engine, t["Q"].detach(), c)
