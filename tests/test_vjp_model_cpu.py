"""Gradients of LMPC solutions with respect to the dynamics (A, B, d) and the row constraints' matrices (E, G) without a GPU:
the closed forms of tests/vjp_model_reference.py against central differences of the CPU oracle's builds and of its solutions,
rho_0 against the x0 gradient of tests/vjp_reference, the host-side refusals of copra_b200_lmpc_vjp_model and its exported
symbols."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import vjp_cost_reference as cr
from tests import vjp_model_reference as mr
from tests import vjp_reference as vr

CASES = [("c1", lambda: wl.c1(), [0]), ("c2", lambda: wl.c2(batch=8), [3]), ("c2_floor", lambda: vr.c2_floor(8), [1, 5]),
         ("c2_mixed", lambda: cr.mixed(8), [0]), ("c3", lambda: wl.c3(batch=4), [0]),
         ("c3_walk", lambda: wl.c3_walk(batch=4), [1]), ("c3_g", lambda: mr.c3_g(4), [0, 2]),
         ("c5_tight", lambda: mr.c5_tight(8), [1, 5]), ("c2_two_inputs", lambda: mr.c2_two_inputs(8), [0, 4])]


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
    rng = np.random.default_rng(31)
    for i in idx:
        inst, o, _, dtraj, adj = _solved(bp, i, 7 + i)
        grads, rho0 = mr.closed_form(inst, o, adj, dtraj)
        assert set(grads) == set(mr.model_keys(inst))
        # rho_0 is the x0 gradient of the vector VJP
        nx = inst["nx"]
        dx0 = np.array([vr.directional(inst, adj, {("x0", None): np.eye(nx)[s]}) for s in range(nx)])
        assert np.abs(rho0 - dx0).max() <= 1e-8 * max(1.0, np.abs(dx0).max()), (name, i, rho0, dx0)
        for key in mr.model_keys(inst):  # one direction per input, so that every gradient is checked on its own
            delta = mr.random_direction(inst, rng, [key])
            if key[0] in ("A", "B"):  # the builds are rational in A and B: Richardson's extrapolation of two steps
                f1, f2 = (mr.directional(inst, o, adj, dtraj, delta, h) for h in (1e-5, 5e-6))
                ref, tol = (4.0 * f2 - f1) / 3.0, 1e-6
            else:  # affine in d, E and G: exact
                ref, tol = mr.directional(inst, o, adj, dtraj, delta, 1.0), 1e-9
            got = mr.dot(grads, delta)
            scale = max(abs(ref), np.abs(grads[key]).sum() * np.abs(delta[key]).max(), 1e-12)
            assert abs(got - ref) <= tol * scale, (name, i, key, got, ref)


def test_variants_exercise_every_kind_of_row():
    """the cases cover active quirk-Q1 lower rows, a non-zero G, an active TRAJECTORY constraint, an active CONTROL
    inequality and an equality"""
    def active_rows(bp, i, j):
        inst = wl.instance(bp, i)
        o = vr.solve(inst)
        eq, ineq = mr.general_rows(inst)
        return [r for k, r in enumerate(eq + ineq) if k + 1 in set(o["iact"].tolist()) and r[0] == j]
    # C2-floor's only finite lower entry is the velocity line: its selector rows are the lower family's
    assert np.asarray(vr.c2_floor(8)["constraints"][0]["lower"])[1] == -1.0
    assert [r for r in active_rows(vr.c2_floor(8), 1, 0) if r[2] == 1]
    assert active_rows(mr.c5_tight(8), 1, 0)
    two = mr.c2_two_inputs(8)
    assert len(active_rows(two, 0, 2)) == two["N"] and active_rows(two, 0, 3)
    assert np.abs(mr.c3_g(2)["constraints"][0]["G"]).max() > 0 and active_rows(mr.c3_g(4), 0, 0)


# central differences of the oracle's solutions need a QP whose solution the oracle resolves far below the step (see
# tests/test_vjp_costs_cpu.py) and an active set that stays put across it; the C3 variants (jerk inputs, G entries of 1e-4)
# are not resolved finely enough, and the build check above covers them exactly
FD_CASES = [c for c in CASES if c[0] in ("c2", "c2_floor", "c5_tight", "c2_two_inputs")]


@pytest.mark.parametrize("name,make,idx", FD_CASES, ids=[c[0] for c in FD_CASES])
def test_closed_forms_match_central_differences_of_solutions(name, make, idx):
    bp = make()
    rng = np.random.default_rng(9)
    checked = 0
    for i in idx:
        inst, o, dcontrol, dtraj, adj = _solved(bp, i, 3 + i)
        grads, _ = mr.closed_form(inst, o, adj, dtraj)
        act = set(o["iact"].tolist())
        for key in mr.model_keys(inst):
            theta = mr.get_matrix(inst, key)
            delta = {key: rng.normal(size=theta.shape) * np.maximum(np.abs(theta), 1e-2 * max(np.abs(theta).max(), 1e-3))}

            def fd(h):
                ends = [vr.solve(mr.with_matrices(inst, {key: theta + s * h * delta[key]})) for s in (1.0, -1.0)]
                if any(set(e["iact"].tolist()) != act or e["fail"] != 0 for e in ends):
                    return None  # the active set moved: the map is not smooth across [theta - h delta, theta + h delta]
                return (vr.loss(ends[0], dcontrol, dtraj) - vr.loss(ends[1], dcontrol, dtraj)) / (2.0 * h)
            for h in (1e-4, 1e-5, 1e-6):
                f1, f2 = fd(h), fd(h / 2)
                if f1 is not None and f2 is not None:
                    break
            else:
                continue
            est = (4.0 * f2 - f1) / 3.0
            pred = mr.dot(grads, delta)
            mag = max(abs(est), abs(pred), float(np.abs(grads[key] * delta[key]).sum()))
            assert abs(est - pred) <= 1e-5 * mag, (name, i, key, est, pred, h)
            checked += 1
    assert checked >= 3


def test_constraint_shapes():
    assert capi.cstr_shapes(wl.c3(batch=2)) == [(4, True, True)]
    assert capi.cstr_shapes(wl.c5(batch=2)) == [(8, True, False), (0, False, False)]
    assert capi.cstr_shapes(mr.c2_two_inputs(2)) == [(0, False, False), (0, False, False), (1, False, True), (1, False, True)]


def test_vjp_model_exports():
    lib = capi.load()
    for name in ("copra_b200_lmpc_vjp_model", "copra_b200_multi_lmpc_vjp_model"):
        assert name in capi.EXPORTS
        getattr(lib, name)
    assert not set(capi.VJP_MODEL_WANT) & set(capi.VJP_WANT + capi.VJP_COST_WANT)  # existing calls run what they ran before


def test_vjp_model_refuses_without_a_handle_or_a_solve():
    lib = capi.load()
    mo = capi.VjpModelOut()
    assert lib.copra_b200_lmpc_vjp_model(None, None, None, capi.HOST, None, None, C.byref(mo)) == -1
    assert lib.copra_b200_multi_lmpc_vjp_model(None, None, None, None, None, C.byref(mo)) == -1
    eng = capi.Engine.__new__(capi.Engine)  # no device handle: only the host-side bookkeeping
    eng._last_bp = None
    eng.solve_count = 0
    with pytest.raises(capi.CopraB200Error) as e:
        eng.lmpc_vjp(want=("A", "E"))
    assert e.value.code == -5


def test_autograd_refuses_a_matrix_the_constraint_does_not_have():
    torch = pytest.importorskip("torch")
    from copra_b200 import autograd as ag
    bp = wl.c5(batch=2)
    with pytest.raises(ValueError):
        ag._patch_model_matrix(bp, None, "G", 0, torch.zeros((8, 4), dtype=torch.float64))  # a TrajectoryConstraint
    with pytest.raises(ValueError):
        ag._patch_model_matrix(bp, None, "E", 1, torch.zeros((4, 12), dtype=torch.float64))  # a bound
    with pytest.raises(ValueError):
        ag._patch_model_matrix(bp, None, "A", 0, torch.zeros((12, 11), dtype=torch.float64))
