"""The raw-QP JVP reference (tests/qp_jvp_reference.py) against finite differences of the oracle and as the adjoint of the VJP
reference, and the host-side plumbing of Engine.qp_jvp / Engine.qp_jacobian (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi
from tests import qp_jvp_reference as jr
from tests import qp_vjp_reference as qr
from tests.test_qp_vjp_cpu import _cases
from tests.util import exact_active_set_solution

KEYS = qr.KEYS


def _direction(p, rng, keys=KEYS):
    d = qr.random_direction(p, rng)
    return {k: d[k] for k in keys if d[k].size}


@pytest.mark.parametrize("name,p", _cases(), ids=[c[0] for c in _cases()])
def test_reference_matches_exact_active_set_differences(name, p):
    """central differences of the exact solution on the oracle's final active set along a random direction of each input
    (the steps of test_qp_vjp_cpu: x is affine in c and beta, smooth in Q and the rows; C2 carries the 1e-6 I regulariser)"""
    rng = np.random.default_rng(21)
    o = qr.solve(p)
    assert o["fail"] == 0
    for k in KEYS:
        d = _direction(p, rng, (k,))
        if not d:
            continue
        h = 1e-4 if k in ("c", "beq", "bineq", "lb", "ub") else 1e-8 if name == "C2" else 1e-6
        ends = [exact_active_set_solution(dict(qr.moved(p, d, s * h), iact=o["iact"])) for s in (1.0, -1.0)]
        fd = (ends[0] - ends[1]) / (2 * h)
        got = jr.jvp(o, d)
        assert np.abs(got - fd).max() <= 1e-6 * max(1.0, np.abs(fd).max()), (name, k, np.abs(got - fd).max())


@pytest.mark.parametrize("name,p", _cases(), ids=[c[0] for c in _cases()])
def test_reference_matches_oracle_differences(name, p):
    """central differences of the oracle's own solutions along random directions of every input at once, where the step keeps
    the active set"""
    rng = np.random.default_rng(22)
    o = qr.solve(p)
    checked = 0
    for _ in range(4):
        d = _direction(p, rng)
        h = 1e-9 if name == "C2" else 1e-5
        sol = [qr.solve(qr.moved(p, d, s * h)) for s in (1.0, -1.0)]
        if any(s["fail"] != 0 or set(s["iact"]) != set(o["iact"]) for s in sol):
            continue
        fd = (np.asarray(sol[0]["x"]) - np.asarray(sol[1]["x"])) / (2 * h)
        got = jr.jvp(o, d)
        assert np.abs(got - fd).max() <= 1e-5 * max(1.0, np.abs(fd).max()), (name, np.abs(got - fd).max())
        checked += 1
    assert checked >= 2


@pytest.mark.parametrize("name,p", _cases(), ids=[c[0] for c in _cases()])
def test_reference_is_the_adjoint_of_the_vjp_reference(name, p):
    """<w, J t> = sum_k <g_k, t_k> with g the VJP reference's gradients of L = w'x, for a tangent on every input"""
    rng = np.random.default_rng(23)
    o = qr.solve(p)
    n = p["Q"].shape[0]
    for _ in range(3):
        w = rng.normal(size=n)
        t = _direction(p, rng)
        lhs = float(w @ jr.jvp(o, t))
        rhs = qr.dot(qr.closed_form(o, w), t)
        assert abs(lhs - rhs) <= 1e-10 * max(1.0, abs(lhs), abs(rhs)), (name, lhs, rhs)


def test_reference_jacobians():
    """dx/dc is symmetric; the columns of inactive rows are zero; dx/dbeta of an active bound row moves that variable by 1"""
    p = qr.random_qp(np.random.default_rng(24), 12, 2, 14)
    o = qr.solve(p)
    Jc = jr.jacobian(o, "c")
    assert np.allclose(Jc, Jc.T, rtol=0, atol=1e-12 * np.abs(Jc).max())
    n = p["Q"].shape[0]
    for wrt in ("beq", "bineq", "lb", "ub"):
        J = jr.jacobian(o, wrt)
        act = jr.active_rows(o, wrt)
        assert J.shape == (n, p[wrt].shape[0])
        assert not np.delete(J, act, axis=1).any(), wrt
        if wrt in ("lb", "ub"):
            for v in act:
                assert abs(J[v, v] - 1.0) <= 1e-12, (wrt, v, J[v, v])


def test_abi_symbols_and_null_handle():
    lib = capi.load()
    assert "copra_b200_qp_jvp" in capi.EXPORTS and "copra_b200_qp_jacobian" in capi.EXPORTS
    t = capi.QpJvpIn()
    t.ndir = 1
    assert lib.copra_b200_qp_jvp(None, C.byref(t), capi.HOST, None) == -1
    assert lib.copra_b200_qp_jacobian(None, 0, None, capi.HOST) == -1


def _hostside_engine(last_qp):
    eng = capi.Engine.__new__(capi.Engine)  # no device handle: only the host-side bookkeeping
    eng._last_qp = last_qp
    return eng


def test_qp_jvp_refuses_without_a_solve():
    eng = _hostside_engine(None)
    for call in (lambda: eng.qp_jvp(c=np.zeros((1, 1, 2))), lambda: eng.qp_jacobian("c")):
        with pytest.raises(capi.CopraB200Error) as e:
            call()
        assert e.value.code == -5


def test_tangent_shapes_are_checked_on_the_host():
    eng = _hostside_engine(dict(n=3, meq=0, m=2, batch=4, live=None))
    k, ts, dev = eng._qp_tangents(dict(c=np.zeros((4, 2, 3)), Q=np.zeros((2, 3, 3)), Aineq=np.zeros((4, 2, 2, 3))))
    assert k == 2 and dev is None
    assert not ts["c"][1] and ts["Q"][1] and not ts["Aineq"][1]
    bad = [dict(c=np.zeros((4, 2, 3)), lb=np.zeros((3, 3))),        # k = 2 and k = 3
           dict(c=np.zeros((4, 2, 4))),                             # wrong n
           dict(c=np.zeros((5, 2, 3))),                             # wrong batch (and not a shared (k, n) either)
           dict(Q=np.zeros((4, 1, 3))),                             # Q needs n x n per direction
           dict(Aeq=np.zeros((1, 0, 3))),                           # no equality rows
           dict(c=np.zeros((0, 3))),                                # k = 0
           dict()]                                                  # nothing given
    for kw in bad:
        with pytest.raises(capi.CopraB200Error) as e:
            eng.qp_jvp(**kw)
        assert e.value.code == -1, kw
    with pytest.raises(capi.CopraB200Error) as e:
        eng.qp_jacobian("x")
    assert e.value.code == -1
