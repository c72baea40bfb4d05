"""CPU checks of the initial-state sensitivity reference (tests/initial_state_sens_reference.py): against central differences
of the exact solution on the oracle's final active set and of the oracle's own solves, the adjoint identity of the VJP and
the JVP, and a symmetric dR."""
import numpy as np
import pytest

from copra_b200 import workloads as wl
from tests import initial_state_sens_reference as ir
from tests.golden import make_golden as mg


def golden():
    return dict(mg.small_cases())["all_kinds_initial_state"]


def variant():
    """the golden initial-state fixture (an equality row at every step, a MIXED inequality) with a finite lower position line
    on its trajectory bound, active at x0* (quirk Q1: the lower rows read x <= lower), and a wider x0 box"""
    v = golden()
    v["constraints"] = [dict(c) for c in v["constraints"]]
    v["x0lb"] = np.array([0.0, -1.5])
    v["constraints"][4] = dict(v["constraints"][4], lower=np.array([0.15, -np.inf]))
    return v


def pinned():
    """C4 without x0lb / x0ub: the bounds default to x0, so x0 itself has a gradient"""
    inst = wl.instance(wl.c4(batch=4, N=12, T=0.12), 2)
    inst["x0lb"] = inst["x0ub"] = None
    return inst


CASES = {
    "c4_0": lambda: wl.instance(wl.c4(batch=4), 0),
    "c4_3": lambda: wl.instance(wl.c4(batch=4), 3),
    "c4_n12": lambda: wl.instance(wl.c4(batch=4, N=12, T=0.12), 1),
    "golden": golden,
    "variant": variant,
    "pinned": pinned,
}


def _cotangent(o, rng):
    s = o["sizes"]
    return rng.normal(size=s["nU"]), rng.normal(size=s["X"])


def _feasible(inst, t):
    """the tangent with x0ub moving like x0lb where the box is pinned (lb = ub), so that the moved problem stays feasible"""
    t = dict(t)
    if inst.get("x0lb") is not None and inst.get("x0ub") is not None:
        same = np.asarray(inst["x0lb"]) == np.asarray(inst["x0ub"])
        t[("x0ub", None)] = np.where(same, t[("x0lb", None)], t[("x0ub", None)])
    return t


@pytest.mark.parametrize("name", sorted(CASES))
def test_vjp_and_jvp_match_active_set_central_differences(name):
    inst = CASES[name]()
    rng = np.random.default_rng(7)
    o = ir.solve(inst)
    assert o["fail"] == 0
    dc, dt = _cotangent(o, rng)
    g = ir.vjp(inst, dc, dt, o)
    for _ in range(2):
        t = ir.random_tangent(inst, rng)
        h = 1e-5
        fd = (ir.active_set_loss(ir.moved(inst, t, h), o["iact"], dc, dt)
              - ir.active_set_loss(ir.moved(inst, t, -h), o["iact"], dc, dt)) / (2 * h)
        assert ir.dot(g, t) == pytest.approx(fd, rel=1e-7, abs=1e-8)
        du, dx = ir.jvp(inst, t, o)
        assert float(dc @ du + dt @ dx) == pytest.approx(fd, rel=1e-7, abs=1e-8)


# the oracle resolves C4's solution to about 1e-9, so its differences take a larger step there (the loss is affine in the
# vectors on the active set and smooth in R).  The pinned box (x0lb = x0ub = x0) is left out: qpgen2 reports some of its
# perturbations infeasible when it adds the second of two coinciding bound rows.
ORACLE_STEP = {"c4_0": 1e-3, "c4_3": 1e-3, "c4_n12": 1e-3, "golden": 1e-6, "variant": 1e-6}


@pytest.mark.parametrize("name", sorted(ORACLE_STEP))
def test_vjp_matches_oracle_central_differences(name):
    inst = CASES[name]()
    rng = np.random.default_rng(11)
    o = ir.solve(inst)
    dc, dt = _cotangent(o, rng)
    g = ir.vjp(inst, dc, dt, o)
    t = _feasible(inst, ir.random_tangent(inst, rng))
    h = ORACLE_STEP[name]
    lp, op = ir.oracle_loss(ir.moved(inst, t, h), dc, dt)
    lm, om = ir.oracle_loss(ir.moved(inst, t, -h), dc, dt)
    assert op["fail"] == om["fail"] == 0
    assert set(op["iact"]) == set(om["iact"]) == set(o["iact"])
    assert ir.dot(g, t) == pytest.approx((lp - lm) / (2 * h), rel=1e-6, abs=1e-7)


@pytest.mark.parametrize("name", sorted(CASES))
def test_adjoint_identity_and_symmetric_dR(name):
    inst = CASES[name]()
    rng = np.random.default_rng(3)
    o = ir.solve(inst)
    dc, dt = _cotangent(o, rng)
    g = ir.vjp(inst, dc, dt, o)
    t = ir.random_tangent(inst, rng)
    du, dx = ir.jvp(inst, t, o)
    assert ir.dot(g, t) == pytest.approx(float(dc @ du + dt @ dx), rel=1e-10, abs=1e-12)
    if ("R", None) in g:
        dR = g[("R", None)]
        assert np.array_equal(dR, dR.T)


def test_x0_gradient_only_through_defaulted_bounds():
    """with both x0 bounds given x0 does not enter the build; with the default (pinned) bounds its gradient is the sum of the
    x0 bound multipliers, i.e. that of x0lb plus that of x0ub had they been given as x0"""
    rng = np.random.default_rng(5)
    inst = wl.instance(wl.c4(batch=4, N=12, T=0.12), 2)
    o = ir.solve(inst)
    dc, dt = _cotangent(o, rng)
    assert np.array_equal(ir.vjp(inst, dc, dt, o)[("x0", None)], np.zeros(2))
    free = pinned()
    given = dict(free, x0lb=np.asarray(free["x0"]), x0ub=np.asarray(free["x0"]))
    gf, gg = ir.vjp(free, dc, dt), ir.vjp(given, dc, dt)
    np.testing.assert_allclose(gf[("x0", None)], gg[("x0lb", None)] + gg[("x0ub", None)], rtol=1e-12, atol=1e-14)
