"""TEST INFRASTRUCTURE -- a dense numpy reference for the Jacobian-vector products of one raw QP (copra_b200_qp_jvp).

    min 1/2 x'Qx + c'x  s.t.  Aeq x = beq,  Aineq x <= bineq,  lb <= x <= ub

With the oracle's final active set written as equalities a_j'x = beta_j in their natural orientation
(tests/vjp_model_reference.active_system) and the forward multipliers lambda (tests/qp_vjp_reference.multipliers), a tangent
(Qdot, cdot, Aeqdot, beqdot, Aineqdot, bineqdot, lbdot, ubdot) moves x by the solution of
    [Q A'; A 0] [xdot; lambdadot] = [-cdot_eff; bdot_eff],
    cdot_eff = cdot + (Qdot + Qdot') x / 2 + sum_active lambda_j adot_j,
    bdot_eff_j = bdot_j - adot_j' x (general row),  ubdot_k / lbdot_k (bound row),
solved with the iterative refinement of tests/qp_vjp_reference.
"""
import numpy as np

from tests import qp_vjp_reference as qr
from tests.util import exact_active_set_solution

KEYS = qr.KEYS


def jvp(o, t):
    """xdot of the oracle solve `o` along the tangent dict `t` (a missing key is a zero tangent)"""
    n = o["Q"].shape[0]
    meq, m = o["Aeq"].shape[0], o["Aineq"].shape[0]
    z = {k: np.zeros_like(o[k], dtype=float) for k in KEYS}
    z.update({k: np.asarray(v, float) for k, v in t.items() if v is not None})
    x = exact_active_set_solution(o)
    cdot = z["c"] + 0.5 * (z["Q"] + z["Q"].T) @ x
    if t.get("Aeq") is not None or t.get("Aineq") is not None:
        lam = qr.multipliers(o)
        cdot = cdot + z["Aeq"].T @ lam[:meq] + z["Aineq"].T @ lam[meq:meq + m]
    bdot = []
    for k in np.asarray(o["iact"], int) - 1:
        if k < meq:
            bdot.append(z["beq"][k] - z["Aeq"][k] @ x)
        elif k < meq + m:
            bdot.append(z["bineq"][k - meq] - z["Aineq"][k - meq] @ x)
        elif k < meq + m + n:
            bdot.append(z["ub"][k - meq - m])
        else:
            bdot.append(z["lb"][k - meq - m - n])
    return qr._kkt_solve(o, np.concatenate([-cdot, np.asarray(bdot, float)]))[:n]


def jacobian(o, wrt):
    """dx/d`wrt` (n x len) for wrt in c, beq, bineq, lb, ub: jvp along the columns of the identity on that input"""
    ln = o[wrt].shape[0]
    cols = []
    for d in range(ln):
        e = np.zeros(ln)
        e[d] = 1.0
        cols.append(jvp(o, {wrt: e}))
    return np.array(cols).T.reshape(o["Q"].shape[0], ln)


def active_rows(o, wrt):
    """the entries of input `wrt` (beq, bineq, lb, ub) whose row is active at the oracle solve `o`"""
    n = o["Q"].shape[0]
    meq, m = o["Aeq"].shape[0], o["Aineq"].shape[0]
    off = dict(beq=0, bineq=meq, ub=meq + m, lb=meq + m + n)[wrt]
    ln = o[wrt].shape[0]
    return sorted(k - off for k in np.asarray(o["iact"], int) - 1 if off <= k < off + ln)
