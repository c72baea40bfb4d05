"""Forward-mode sensitivities of LMPC solutions without a GPU: the dense numpy forward reference (tests/jvp_reference.py)
against central differences of the CPU oracle, its adjoint identity with the VJP reference, the host-side refusals of
copra_b200_lmpc_jvp / copra_b200_lmpc_feedback_gain and their exported symbols."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import jvp_reference as jr
from tests import vjp_reference as vr

CASES = [("c1", lambda: wl.c1(), [0]), ("c2", lambda: wl.c2(batch=8), [3]), ("c3", lambda: wl.c3(batch=4), [0, 3]),
         ("c3_walk", lambda: wl.c3_walk(batch=4), [1, 2]), ("c2_floor", lambda: vr.c2_floor(8), [1, 5])]


def test_one_dimensional_tangent():
    # min 1/2 x^2 - 5x s.t. x <= b, b = 1 active: dx/db = 1, and the cost's linear term does not move x
    o = dict(Q=np.eye(1), Aeq=np.zeros((0, 1)), Aineq=np.ones((1, 1)), iact=np.array([1]))
    A, idx = jr.active_rows(o)
    assert A.shape == (1, 1) and idx.tolist() == [0]
    K = np.block([[o["Q"], A.T], [A, np.zeros((1, 1))]])
    assert np.linalg.solve(K, np.array([-3.0, 1.0]))[0] == pytest.approx(1.0, abs=1e-15)


@pytest.mark.parametrize("name,make,idx", CASES, ids=[c[0] for c in CASES])
def test_reference_matches_central_differences(name, make, idx):
    bp = make()
    rng = np.random.default_rng(12)
    checked = 0
    for i in idx:
        inst = wl.instance(bp, i)
        o = vr.solve(inst)
        assert o["fail"] == 0
        act = set(o["iact"].tolist())
        for key in vr.vector_keys(inst):
            delta = vr.random_direction(inst, rng, [key])
            if not np.any(delta[key]):
                continue
            du, dx = jr.tangent(inst, o, delta)
            scale = max(1.0, np.abs(vr.get_vector(inst, key)).max())
            for h in (1e-2 * scale, 1e-3 * scale, 1e-4 * scale):
                ends = [vr.solve(vr.with_vectors(inst, {key: vr.get_vector(inst, key) + sgn * h * delta[key]}))
                        for sgn in (1.0, -1.0)]
                if all(set(e["iact"].tolist()) == act and e["fail"] == 0 for e in ends):
                    break
            else:
                continue  # the active set moved: the map is not affine across [theta - h delta, theta + h delta]
            for got, out in ((du, "control"), (dx, "trajectory")):
                fd = (ends[0][out] - ends[1][out]) / (2.0 * h)
                # the oracle's own rounding, divided by h, bounds what a difference can resolve in a weak direction
                mag = max(np.abs(fd).max(), np.abs(got).max(), 0.1 * max(1.0, np.abs(o[out]).max()))
                assert np.abs(fd - got).max() <= 1e-5 * mag, (name, i, key, out, np.abs(fd - got).max(), mag)
            checked += 1
    assert checked >= 3


@pytest.mark.parametrize("name,make,idx", CASES, ids=[c[0] for c in CASES])
def test_reference_is_the_adjoint_of_the_vjp_reference(name, make, idx):
    # <gbar, J thetadot> == <J' gbar, thetadot> for a random cotangent and a random direction over every input at once
    bp = make()
    rng = np.random.default_rng(13)
    for i in idx:
        inst = wl.instance(bp, i)
        o = vr.solve(inst)
        dc = rng.normal(size=o["control"].shape)
        dt = rng.normal(size=o["trajectory"].shape)
        delta = vr.random_direction(inst, rng)
        du, dx = jr.tangent(inst, o, delta)
        lhs = float(dc @ du + dt @ dx)
        rhs = vr.directional(inst, vr.adjoint(o, dc, dt), delta)
        # relative to the sum of the magnitudes of the products: the inner product itself may cancel
        scale = float(np.abs(dc * du).sum() + np.abs(dt * dx).sum())
        assert abs(lhs - rhs) <= 1e-10 * max(abs(lhs), abs(rhs), scale), (name, i, lhs, rhs, scale)


def test_jvp_exports():
    lib = capi.load()
    for name in ("copra_b200_lmpc_jvp", "copra_b200_lmpc_feedback_gain", "copra_b200_multi_lmpc_jvp",
                 "copra_b200_multi_lmpc_feedback_gain"):
        assert name in capi.EXPORTS
        getattr(lib, name)


def _bare_engine():
    eng = capi.Engine.__new__(capi.Engine)  # no device handle: only the host-side bookkeeping
    eng._last_bp = None
    eng.solve_count = 0
    return eng


def test_jvp_refuses_without_a_solve():
    lib = capi.load()
    t = capi.JvpIn()
    t.ndir = 1
    # null handle / null tangent description
    assert lib.copra_b200_lmpc_jvp(None, C.byref(t), capi.HOST, None, None) == -1
    assert lib.copra_b200_lmpc_jvp(None, None, capi.HOST, None, None) == -1
    assert lib.copra_b200_lmpc_feedback_gain(None, 1, None, None, capi.HOST) == -1
    assert lib.copra_b200_multi_lmpc_jvp(None, C.byref(t), None, None) == -1
    assert lib.copra_b200_multi_lmpc_feedback_gain(None, 1, None, None) == -1
    eng = _bare_engine()
    for call in (lambda: eng.lmpc_jvp(x0=np.zeros((1, 1, 2))), lambda: eng.lmpc_feedback_gain(1)):
        with pytest.raises(capi.CopraB200Error) as e:
            call()
        assert e.value.code == -5


def test_jvp_checks_tangent_shapes_on_the_host():
    bp = wl.c2(batch=3)
    calls = []

    def call(t, mem, du, dx):
        calls.append((t.ndir, mem))

    with pytest.raises(capi.CopraB200Error):  # no tangent at all
        capi._jvp_call(bp, 3, None, None, None, None, None, call)
    with pytest.raises(capi.CopraB200Error):  # (batch, len) instead of (batch, k, len)
        capi._jvp_call(bp, 3, np.zeros((3, 2)), None, None, None, None, call)
    with pytest.raises(capi.CopraB200Error):  # constraint 0 of C2 is a trajectory bound: it has no f
        capi._jvp_call(bp, 3, None, None, [np.zeros((3, 2, 2))], None, None, call)
    with pytest.raises(capi.CopraB200Error):  # k differs between tangents
        capi._jvp_call(bp, 3, np.zeros((3, 2, 2)), [np.zeros((3, 1, 2))], None, None, None, call)
    assert not calls
    du, dx = capi._jvp_call(bp, 3, np.zeros((3, 4, 2)), None, None, [None, np.zeros((3, 4, 1))], None, call)
    assert calls == [(4, capi.HOST)]
    assert du.shape == (3, 4, 50) and dx.shape == (3, 4, 102)


def test_feedback_gain_layout():
    # the engine writes each instance's (nu*steps) x nx gain column-major; the Python result is (batch, nu*steps, nx)
    bp = wl.c3(batch=2)

    def call(steps, ku, kx, mem):
        ru, rx, nx = 2 * steps, 6 * (steps + 1), 6
        a = np.ctypeslib.as_array(C.cast(ku, C.POINTER(C.c_double)), shape=(2 * nx * ru,))
        a[:] = np.arange(a.size)
        np.ctypeslib.as_array(C.cast(kx, C.POINTER(C.c_double)), shape=(2 * nx * rx,))[:] = 0.0

    ku, kx = capi._gain_call(bp, 2, 3, None, call)
    assert ku.shape == (2, 6, 6) and kx.shape == (2, 24, 6)
    # instance 1, row r, column s sits at 1 * 36 + s * 6 + r
    assert ku[1, 4, 2] == 36 + 2 * 6 + 4
