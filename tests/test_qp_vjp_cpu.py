"""The raw-QP VJP reference (tests/qp_vjp_reference.py) against finite differences, and the host-side plumbing of
Engine.qp_vjp / copra_b200.autograd.qp (no GPU needed)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from oracle import pyoracle as po
from tests import qp_vjp_reference as qr
from tests import vjp_model_reference as mr
from tests.util import exact_active_set_solution

HERE = os.path.dirname(os.path.abspath(__file__))


def ka1():
    ka = json.load(open(os.path.join(HERE, "golden", "ka_problem.json")))
    return qr.problem(ka["Q"], ka["c"], ka["Aeq"], ka["beq"], ka["Aineq"], ka["bineq"], ka["XL"], ka["XU"])


def c2_qp():
    """instance 0 of C2 as the oracle assembles it (the QP the engine's download returns)"""
    b = po.lmpc(wl.instance(wl.c2(batch=1), 0), solve=False)
    return qr.problem(b["Q"], b["c"], b["Aeq"], b["beq"], b["Aineq"], b["bineq"], b["lb"], b["ub"])


def random_qps():
    rng = np.random.default_rng(11)
    return [qr.random_qp(rng, n, meq, m) for n, meq, m in ((6, 1, 4), (10, 2, 12), (14, 0, 20), (20, 3, 15), (25, 4, 30))]


def _cases():
    return [("random%d" % i, p) for i, p in enumerate(random_qps())] + [("KA-1", ka1()), ("C2", c2_qp())]


def _kinds(o):
    n, meq, m = o["Q"].shape[0], o["Aeq"].shape[0], o["Aineq"].shape[0]
    out = set()
    for k in np.asarray(o["iact"], int) - 1:
        out.add("eq" if k < meq else "ineq" if k < meq + m else "upper" if k < meq + m + n else "lower")
    return out


def test_random_qps_cover_every_row_kind():
    kinds, inf = set(), set()
    for p in random_qps():
        o = qr.solve(p)
        assert o["fail"] == 0
        kinds |= _kinds(o)
        inf |= {"-inf" for v in p["lb"] if v == -np.inf} | {"+inf" for v in p["ub"] if v == np.inf}
    assert kinds == {"eq", "ineq", "upper", "lower"} and inf == {"-inf", "+inf"}


@pytest.mark.parametrize("name,p", _cases(), ids=[c[0] for c in _cases()])
def test_closed_form_matches_exact_active_set_differences(name, p):
    """central differences of the exact solution on the oracle's final active set along a random direction of each input
    (Q symmetric).  x is affine in c and beta, so a long step is exact there; it is smooth in Q and the rows, where the
    difference is O(h^2) (C2's Hessian carries the 1e-6 I regulariser: x moves ~1e7 times faster with it, so a shorter step)"""
    rng = np.random.default_rng(5)
    o = qr.solve(p)
    assert o["fail"] == 0
    n = p["Q"].shape[0]
    for _ in range(3):
        dx = rng.normal(size=n)
        g = qr.closed_form(o, dx)
        d = qr.random_direction(p, rng)
        for k in qr.KEYS:
            if d[k].size == 0:
                continue
            h = 1e-4 if k in ("c", "beq", "bineq", "lb", "ub") else 1e-8 if name == "C2" else 1e-6
            ends = [dx @ exact_active_set_solution(dict(qr.moved(p, {k: d[k]}, s * h), iact=o["iact"])) for s in (1.0, -1.0)]
            fd = (ends[0] - ends[1]) / (2 * h)
            assert abs(qr.dot(g, {k: d[k]}) - fd) <= 1e-6 * max(1.0, abs(fd)), (name, k, qr.dot(g, {k: d[k]}), fd)


@pytest.mark.parametrize("name,p", _cases(), ids=[c[0] for c in _cases()])
def test_closed_form_matches_oracle_differences(name, p):
    """central differences of the oracle's own solutions, where the step keeps the active set and the oracle resolves it"""
    rng = np.random.default_rng(6)
    o = qr.solve(p)
    n = p["Q"].shape[0]
    dx = rng.normal(size=n)
    g = qr.closed_form(o, dx)
    checked = 0
    for _ in range(4):
        d = qr.random_direction(p, rng)
        h = 1e-9 if name == "C2" else 1e-5
        sol = [qr.solve(qr.moved(p, d, s * h)) for s in (1.0, -1.0)]
        if any(s["fail"] != 0 or set(s["iact"]) != set(o["iact"]) for s in sol):
            continue
        fd = (dx @ sol[0]["x"] - dx @ sol[1]["x"]) / (2 * h)
        assert abs(qr.dot(g, d) - fd) <= 1e-5 * max(1.0, abs(fd)), (name, qr.dot(g, d), fd)
        checked += 1
    assert checked >= 2


@pytest.mark.parametrize("name,p", _cases(), ids=[c[0] for c in _cases()])
def test_forward_multipliers_agree_with_the_oracle(name, p):
    """lambda (natural orientation) against the oracle's lagr: quadprog reports a lower row as -x <= -lb, so its multiplier
    has the other sign; an equality's sign depends on the orientation quadprog gave the row, so its magnitude is compared"""
    o = qr.solve(p)
    n, meq, m = o["Q"].shape[0], o["Aeq"].shape[0], o["Aineq"].shape[0]
    lam = qr.multipliers(o)
    assert np.allclose(lam, mr.forward_multipliers(o), rtol=0, atol=1e-8 * max(1.0, np.abs(lam).max()))
    lagr = np.asarray(o["lagr"], float)
    scale = max(1.0, np.abs(lagr).max())
    for k in np.asarray(o["iact"], int) - 1:
        want = -lam[k] if k >= meq + m + n else lam[k]
        if k < meq:
            want, got = abs(want), abs(lagr[k])
        else:
            got = lagr[k]
        assert abs(want - got) <= 1e-8 * scale, (name, k, lam[k], lagr[k])
    inactive = np.setdiff1d(np.arange(lagr.size), np.asarray(o["iact"], int) - 1)
    assert np.all(lam[inactive] == 0.0) and np.all(lagr[inactive] == 0.0)


def test_closed_form_shapes_and_symmetry():
    p = random_qps()[3]
    o = qr.solve(p)
    g = qr.closed_form(o, np.ones(p["Q"].shape[0]))
    for k in qr.KEYS:
        assert g[k].shape == p[k].shape, k
    assert np.array_equal(g["Q"], g["Q"].T)
    act = set(np.asarray(o["iact"], int) - 1)
    meq = p["Aeq"].shape[0]
    for j in range(p["Aineq"].shape[0]):
        if meq + j not in act:
            assert not g["Aineq"][j].any() and g["bineq"][j] == 0.0


def test_qp_vjp_refuses_without_a_solve():
    lib = capi.load()
    assert "copra_b200_qp_vjp" in capi.EXPORTS
    out = capi.QpVjpOut()
    assert lib.copra_b200_qp_vjp(None, None, capi.HOST, C.byref(out)) == -1
    eng = capi.Engine.__new__(capi.Engine)  # no device handle: only the host-side bookkeeping
    eng._last_qp = None
    with pytest.raises(capi.CopraB200Error) as e:
        eng.qp_vjp(np.zeros((1, 2)))
    assert e.value.code == -5


class _FakeEngine:
    """the two calls copra_b200.autograd.qp makes, on CPU tensors: x = 1, and gradient b (the instance number) everywhere"""
    def __init__(self):
        self.solve_count = 0

    def solve_qp_batch(self, *args):
        import torch
        self.solve_count += 1
        kw = {k: a for k, a in zip(qr.KEYS, args) if a is not None}
        self.inputs = kw
        B = max([a.shape[0] for k, a in kw.items() if a.dim() > capi.QP_BASE_NDIM[k]] or [1])
        return dict(x=torch.ones((B, kw["Q"].shape[-1]), dtype=torch.float64), status=torch.zeros(B, dtype=torch.int32))

    def qp_vjp(self, dx, want):
        import torch
        B, n = dx.shape
        self.want = want
        shapes = dict(Q=(n, n), c=(n,), Aeq=(2, n), beq=(2,), Aineq=(3, n), bineq=(3,), lb=(n,), ub=(n,))
        return {k: torch.arange(B, dtype=torch.float64).reshape((B,) + (1,) * len(s)).expand((B,) + s).clone()
                if k in want else None for k, s in shapes.items()}


def test_autograd_qp_plumbing():
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    eng = _FakeEngine()
    Q = torch.eye(3, dtype=torch.float64, requires_grad=True)          # shared: the sum over the batch
    c = torch.zeros((4, 3), dtype=torch.float64, requires_grad=True)   # batched: per instance
    Aeq = torch.zeros((2, 3), dtype=torch.float64)                     # no gradient wanted
    beq = torch.zeros((4, 2), dtype=torch.float64, requires_grad=True)
    x, status = ag.qp(eng, Q, c, Aeq=Aeq, beq=beq)
    assert not status.requires_grad
    assert torch.equal(eng.inputs["lb"], torch.full((3,), -torch.inf, dtype=torch.float64))
    assert torch.equal(eng.inputs["ub"], torch.full((3,), torch.inf, dtype=torch.float64))
    x.sum().backward()
    assert eng.want == ("Q", "c", "beq")
    assert torch.equal(Q.grad, torch.full((3, 3), 6.0, dtype=torch.float64))
    assert torch.equal(c.grad, torch.arange(4, dtype=torch.float64)[:, None].expand(4, 3))
    assert torch.equal(beq.grad, torch.arange(4, dtype=torch.float64)[:, None].expand(4, 2))
    # a stale backward
    x, _ = ag.qp(eng, Q, c)
    eng.solve_count += 1
    with pytest.raises(RuntimeError, match="another solve ran"):
        x.sum().backward()
    # forward mode
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        with pytest.raises(NotImplementedError):
            ag.qp(eng, Q.detach(), fwAD.make_dual(c.detach(), torch.ones_like(c)))
        x, _ = ag.qp(eng, Q.detach(), fwAD.make_dual(c.detach(), torch.zeros_like(c)))
        assert not fwAD.unpack_dual(x).tangent.any()
