"""TEST INFRASTRUCTURE -- a dense numpy reference for the Jacobian-vector product of one LMPC instance (copra_b200_lmpc_jvp).

It takes the CPU oracle's QP and active set and solves the forward KKT system densely:
    [Q A'; A 0] [Udot; lamdot] = [-cdot; bdot_act],   trajectory tangent = Phi x0dot + Psi Udot,
with A the active rows in their natural orientation (Aeq / Aineq rows, e_k for either bound), as in vjp_reference.adjoint.
c, beq, bineq, lb and ub are affine in the vector inputs, so cdot and bdot are differenced on the oracle's own builds along the
input direction (vjp_reference.directional does the same for the adjoint).
"""
import numpy as np

from tests import vjp_reference as vr


def active_rows(o):
    """the active rows of a solved oracle instance in iact order, and their indices in [eq | ineq | upper | lower]"""
    n = o["Q"].shape[0]
    meq, m = o["Aeq"].shape[0], o["Aineq"].shape[0]
    idx = np.asarray(o["iact"], int) - 1
    rows = []
    for k in idx:
        if k < meq:
            rows.append(o["Aeq"][k])
        elif k < meq + m:
            rows.append(o["Aineq"][k - meq])
        else:
            e = np.zeros(n)
            e[(k - meq - m) % n] = 1.0
            rows.append(e)
    return np.array(rows).reshape(-1, n), idx


def qp_tangent(inst, delta):
    """(cdot, bdot) of `inst` along the input direction `delta` ({key: array}); bdot in [beq | bineq | ub | lb] order"""
    q0 = vr.build(inst)
    q1 = vr.build(vr.with_vectors(inst, {k: vr.get_vector(inst, k) + d for k, d in delta.items()}))
    bdot = np.concatenate([vr._finite_diff(q0[k], q1[k]) for k in ("beq", "bineq", "ub", "lb")])
    return q1["c"] - q0["c"], bdot


def tangent(inst, o, delta):
    """(dcontrol, dtrajectory) of the solved oracle instance `o` of `inst` along the input direction `delta`"""
    Q = o["Q"]
    n = Q.shape[0]
    A, idx = active_rows(o)
    na = A.shape[0]
    cdot, bdot = qp_tangent(inst, delta)
    K = np.block([[Q, A.T], [A, np.zeros((na, na))]])
    du = np.linalg.solve(K, np.concatenate([-cdot, bdot[idx]]))[:n]
    x0dot = delta.get(("x0", None), np.zeros(o["Phi"].shape[1]))
    return du, o["Phi"] @ x0dot + o["Psi"] @ du
