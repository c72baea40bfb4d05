"""TEST INFRASTRUCTURE -- a dense numpy reference for the vector-Jacobian product of one raw QP (copra_b200_qp_vjp).

    min 1/2 x'Qx + c'x  s.t.  Aeq x = beq,  Aineq x <= bineq,  lb <= x <= ub

With the oracle's final active set written as equalities a_j'x = beta_j in their natural orientation
(tests/vjp_model_reference.active_system), dx = dL/dx, [Q A'; A 0] [v; mu] = [dx; 0] and the forward multipliers lambda of
[Q A'; A 0] [x; lambda] = [-c; beta] (as tests/vjp_model_reference.forward_multipliers, with iterative refinement):
    dL/dc = -v,  dL/dbeta_j = mu_j,  dL/da_j = -lambda_j v - mu_j x,  dL/dQ = -(v x' + x v') / 2,
0 for the inactive rows.  dQ is the gradient along symmetric perturbations of Q.
"""
import numpy as np

from oracle import pyoracle as po
from tests import vjp_model_reference as mr
from tests.util import exact_active_set_solution

KEYS = ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")


def problem(Q, c, Aeq=None, beq=None, Aineq=None, bineq=None, lb=None, ub=None):
    """one raw QP as a dict of float arrays (empty rows for absent constraints, +-inf for absent bounds)"""
    Q = np.asarray(Q, float)
    n = Q.shape[0]
    return dict(Q=Q, c=np.asarray(c, float),
                Aeq=np.zeros((0, n)) if Aeq is None else np.asarray(Aeq, float).reshape(-1, n),
                beq=np.zeros(0) if beq is None else np.asarray(beq, float).reshape(-1),
                Aineq=np.zeros((0, n)) if Aineq is None else np.asarray(Aineq, float).reshape(-1, n),
                bineq=np.zeros(0) if bineq is None else np.asarray(bineq, float).reshape(-1),
                lb=np.full(n, -np.inf) if lb is None else np.asarray(lb, float),
                ub=np.full(n, np.inf) if ub is None else np.asarray(ub, float))


def solve(p):
    """the oracle's solve of problem `p`, merged with its inputs (the dict shape active_system / forward_multipliers take)"""
    o = po.quadprog(*(p[k] for k in KEYS))
    return dict(p, **o)


def _kkt_solve(o, rhs):
    """[Q A'; A 0]^-1 rhs on the active set of `o` (columns of rhs: n + nact rows), with iterative refinement in extended
    precision: LMPC Hessians carry a 1e-6 regulariser and a plain solve loses digits to their conditioning"""
    A, _ = mr.active_system(o)
    na = A.shape[0]
    K = np.block([[o["Q"], A.T], [A, np.zeros((na, na))]])
    Kl, rl = K.astype(np.longdouble), rhs.astype(np.longdouble)
    sol = np.linalg.solve(K, rhs)
    for _ in range(3):
        sol = sol + np.linalg.solve(K, (rl - Kl @ sol.astype(np.longdouble)).astype(float))
    return sol


def multipliers(o):
    """lambda of the forward solve over [eq | ineq | ub | lb] (0 for inactive rows): [Q A'; A 0] [x; lambda] = [-c; beta]"""
    _, beta = mr.active_system(o)
    n = o["Q"].shape[0]
    lam = np.zeros(o["Aeq"].shape[0] + o["Aineq"].shape[0] + 2 * n)
    lam[np.asarray(o["iact"], int) - 1] = _kkt_solve(o, np.concatenate([-o["c"], beta]))[n:]
    return lam


def closed_form(o, dx):
    """the eight gradients of L = dx'x at the oracle solve `o`"""
    n = o["Q"].shape[0]
    meq, m = o["Aeq"].shape[0], o["Aineq"].shape[0]
    na = len(o["iact"])
    sol = _kkt_solve(o, np.concatenate([np.asarray(dx, float), np.zeros(na)]))
    v = sol[:n]
    mu = np.zeros(meq + m + 2 * n)
    mu[np.asarray(o["iact"], int) - 1] = sol[n:]
    lam = multipliers(o)
    x = exact_active_set_solution(o)  # the oracle's x may have drifted off its active set by ~1e-6 (C5)
    da = -np.outer(lam[:meq + m], v) - np.outer(mu[:meq + m], x)
    return dict(Q=-0.5 * (np.outer(v, x) + np.outer(x, v)), c=-v, Aeq=da[:meq], beq=mu[:meq], Aineq=da[meq:], bineq=mu[meq:meq + m],
                ub=mu[meq + m:meq + m + n], lb=mu[meq + m + n:])


def random_direction(p, rng):
    """a random direction over every input: symmetric for Q, 0 on infinite (or DBL_MAX) bound entries"""
    d = {k: rng.normal(size=p[k].shape) for k in KEYS}
    d["Q"] = 0.5 * (d["Q"] + d["Q"].T)
    for k in ("lb", "ub"):
        d[k] = np.where(np.abs(p[k]) < 1e300, d[k], 0.0)
    return d


def moved(p, d, h):
    return {k: p[k] + h * d[k] if k in d else p[k] for k in p}


def dot(g, d):
    return float(sum(np.sum(g[k] * d[k]) for k in d))


def random_qp(rng, n, meq, m):
    """the generator of test_mid_size_qps_general_and_cluster_kernels for one instance, with some bounds tightened to the
    unconstrained optimum's side (active upper and lower rows) and some made infinite"""
    L = rng.normal(size=(n, n))
    Q = L @ L.T / n + 0.5 * np.eye(n)
    c = rng.normal(size=n)
    Aeq = rng.normal(size=(meq, n))
    xf = rng.normal(size=n)
    beq = Aeq @ xf
    Aineq = rng.normal(size=(m, n))
    bineq = Aineq @ xf + rng.uniform(0.0, 1.0, size=m)
    lb = xf - rng.uniform(0.1, 2.0, size=n)
    ub = xf + rng.uniform(0.1, 2.0, size=n)
    free = np.linalg.solve(Q, -c)
    tight = rng.uniform(size=n) < 0.4
    lb = np.where(tight & (free < xf), xf - 0.05, lb)
    ub = np.where(tight & (free > xf), xf + 0.05, ub)
    lb[rng.uniform(size=n) < 0.2] = -np.inf
    ub[rng.uniform(size=n) < 0.2] = np.inf
    return problem(Q, c, Aeq if meq else None, beq if meq else None, Aineq if m else None, bineq if m else None, lb, ub)
