"""Gradients of LMPC solutions with respect to the cost weights and matrices without a GPU: the closed forms of
tests/vjp_cost_reference.py against central differences of the CPU oracle's builds (exact: Q and c are at most quadratic in
w, M and N) and of its solutions, the host-side refusals of copra_b200_lmpc_vjp_costs and its exported symbols."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import vjp_cost_reference as cr
from tests import vjp_reference as vr

CASES = [("c1", lambda: wl.c1(), [0]), ("c1_trajectory", lambda: wl.c1("trajectory"), [0]),
         ("c2", lambda: wl.c2(batch=8), [3]), ("c3", lambda: wl.c3(batch=4), [0, 3]),
         ("c3_walk", lambda: wl.c3_walk(batch=4), [1, 2]), ("c2_floor", lambda: vr.c2_floor(8), [1, 5]),
         ("c2_mixed", lambda: cr.mixed(8), [0, 6])]


def _solved(bp, i, seed):
    inst = wl.instance(bp, i)
    o = vr.solve(inst)
    assert o["fail"] == 0
    rng = np.random.default_rng(seed)
    dcontrol = rng.normal(size=o["control"].shape)
    dtraj = rng.normal(size=o["trajectory"].shape)
    return inst, o, dcontrol, dtraj, vr.adjoint(o, dcontrol, dtraj)


@pytest.mark.parametrize("name,make,idx", CASES, ids=[c[0] for c in CASES])
def test_closed_forms_match_the_oracle_build(name, make, idx):
    bp = make()
    rng = np.random.default_rng(21)
    for i in idx:
        inst, o, _, _, adj = _solved(bp, i, 17 + i)
        grads = cr.closed_form(inst, o, adj)
        assert set(grads) == set(cr.cost_keys(inst))
        for key in cr.cost_keys(inst):  # one direction per input, so that every gradient is checked on its own
            delta = cr.random_direction(inst, rng, [key])
            ref = cr.directional(inst, o, adj, delta)
            got = cr.dot(grads, delta)
            scale = max(abs(ref), np.abs(grads[key]).sum() * np.abs(delta[key]).max(), 1e-12)
            assert abs(got - ref) <= 1e-9 * scale, (name, i, key, got, ref)


# central differences of the oracle's solutions need a QP whose solution the oracle resolves far below the step: C1 with a
# trajectory cost (weights up to 1e4 over 301 steps) and C3 walking (about 290 active rows) are not, and the build check above
# covers them exactly
FD_CASES = [c for c in CASES if c[0] not in ("c1_trajectory", "c3_walk", "c2_mixed")] + [("c2_mixed", lambda: cr.mixed(8), [0])]


@pytest.mark.parametrize("name,make,idx", FD_CASES, ids=[c[0] for c in FD_CASES])
def test_closed_forms_match_central_differences_of_solutions(name, make, idx):
    bp = make()
    rng = np.random.default_rng(5)
    checked = 0
    for i in idx:
        inst, o, dcontrol, dtraj, adj = _solved(bp, i, 3 + i)
        grads = cr.closed_form(inst, o, adj)
        act = set(o["iact"].tolist())
        for key in cr.cost_keys(inst):
            # relative steps: weights span orders of magnitude (1e-4 .. 1e4), and the solution is a rational function of
            # them; Richardson's extrapolation of two central differences removes the h^2 term
            theta = cr.get_matrix(inst, key)
            delta = {key: rng.normal(size=theta.shape) * np.maximum(np.abs(theta), 1e-2 * np.abs(theta).max())}

            def fd(h):
                ends = [vr.solve(cr.with_matrices(inst, {key: theta + s * h * delta[key]})) for s in (1.0, -1.0)]
                if any(set(e["iact"].tolist()) != act or e["fail"] != 0 for e in ends):
                    return None  # the active set moved: the map is not smooth across [theta - h delta, theta + h delta]
                return (vr.loss(ends[0], dcontrol, dtraj) - vr.loss(ends[1], dcontrol, dtraj)) / (2.0 * h)
            for h in (1e-3, 1e-4, 1e-5):
                f1, f2 = fd(h), fd(h / 2)
                if f1 is not None and f2 is not None:
                    break
            else:
                continue
            est = (4.0 * f2 - f1) / 3.0
            pred = cr.dot(grads, delta)
            mag = max(abs(est), abs(pred), float(np.abs(grads[key] * delta[key]).sum()))
            assert abs(est - pred) <= 1e-5 * mag, (name, i, key, est, pred, h)
            checked += 1
    assert checked >= 2


def test_mixed_variant_has_both_matrices_and_solves():
    bp = cr.mixed(8)
    inst = wl.instance(bp, 0)
    assert ("M", 2) in cr.cost_keys(inst) and ("N", 2) in cr.cost_keys(inst)
    assert capi.cost_shapes(bp) == [(2, True, False), (1, False, True), (2, True, True)]
    assert capi.cost_shapes(wl.c3_walk(batch=2)) == [(2, True, False), (2, False, True)]


def test_vjp_costs_exports():
    lib = capi.load()
    for name in ("copra_b200_lmpc_vjp_costs", "copra_b200_multi_lmpc_vjp_costs"):
        assert name in capi.EXPORTS
        getattr(lib, name)
    assert not set(capi.VJP_COST_WANT) & set(capi.VJP_WANT)  # existing calls run what they ran before


def test_vjp_costs_refuses_without_a_handle_or_a_solve():
    lib = capi.load()
    co = capi.VjpCostOut()
    # null handle; null output descriptions
    assert lib.copra_b200_lmpc_vjp_costs(None, None, None, capi.HOST, None, C.byref(co)) == -1
    assert lib.copra_b200_multi_lmpc_vjp_costs(None, None, None, None, C.byref(co)) == -1
    eng = capi.Engine.__new__(capi.Engine)  # no device handle: only the host-side bookkeeping
    eng._last_bp = None
    eng.solve_count = 0
    with pytest.raises(capi.CopraB200Error) as e:
        eng.lmpc_vjp(want=("w", "M"))
    assert e.value.code == -5


def test_autograd_refuses_a_matrix_the_cost_does_not_have():
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    bp = wl.c2(batch=2)
    problem = dict(bp, costs=[dict(c) for c in bp["costs"]])
    with pytest.raises(ValueError):
        ag._patch_cost_matrix(problem, None, "M", 1, torch.zeros((1, 2), dtype=torch.float64))  # a ControlCost
    with pytest.raises(ValueError):
        ag._patch_cost_matrix(problem, None, "w", 0, torch.zeros(3, dtype=torch.float64))  # 2 rows
