"""TEST INFRASTRUCTURE -- a dense numpy reference for the sensitivities of one initial-state instance
(copra_b200_lmpc_vjp_initial_state / copra_b200_lmpc_jvp_initial_state).

An initial-state build is a QP in z = [x0*; U]: min 1/2 z'Qz + c'z over the rows [Y | A_U] z (<=, =) z_rows and the bounds
[x0lb; lb] <= z <= [x0ub; ub], with Q_tl = R + E Qb^-1 E', c = [r; sum f], b = f - E xi and the x0 bounds defaulting to x0.
The trajectory is Phi x0* + Psi U + xi.  The reverse mode takes the raw-QP closed forms of tests/qp_vjp_reference on the
oracle's QP and active set (dL/dc = -v, dL/dbeta = mu, dL/dQ = -(v z' + z v') / 2) with gbar = [Phi' dtraj; dcontrol + Psi'
dtraj] and chains them through the build: c, b and the bounds are affine in r, p, f, lower, upper, x0, x0lb and x0ub, so each
input's gradient is <dL/dc, dc> + <dL/dbeta, dbeta> over the oracle's own builds along the unit directions of that input; R
enters Q_tl alone, so dL/dR = dL/dQ[0:nx, 0:nx].  The forward mode is the same chain: cdot and betadot from the builds along
the tangent, plus sym(Rdot) x0* in cdot, one KKT solve [Q A'; A 0] [zdot; .] = [-cdot; betadot_act].
"""
import copy

import numpy as np

from oracle import pyoracle as po
from tests import qp_vjp_reference as qr
from tests import vjp_model_reference as mr
from tests.util import exact_active_set_solution

INITIAL = ("R", "r", "x0lb", "x0ub")


def vector_keys(inst):
    """the affine inputs of an instance: ("x0",), ("r",) / ("x0lb",) / ("x0ub",) where given, ("p", i), ("f", j),
    ("lower", j), ("upper", j)"""
    keys = [("x0", None)] + [(k, None) for k in ("r", "x0lb", "x0ub") if inst.get(k) is not None]
    keys += [("p", i) for i in range(len(inst["costs"]))]
    for j, c in enumerate(inst["constraints"]):
        keys += [("lower", j), ("upper", j)] if c["kind"] in ("trajectory_bound", "control_bound") else [("f", j)]
    return keys


def get(inst, key):
    kind, i = key
    if i is None:
        return np.asarray(inst[kind], float)
    return np.asarray((inst["costs"] if kind == "p" else inst["constraints"])[i][kind], float)


def moved(inst, delta, h=1.0):
    """copy of `inst` with every input of `delta` ({key: array}, "R" included) moved by h * delta"""
    out = copy.copy(inst)
    out["costs"] = [dict(c) for c in inst["costs"]]
    out["constraints"] = [dict(c) for c in inst["constraints"]]
    for key, d in delta.items():
        kind, i = key
        v = get(inst, key) + h * np.asarray(d, float)
        if i is None:
            out[kind] = v
        else:
            (out["costs"] if kind == "p" else out["constraints"])[i][kind] = v
    return out


def build(inst):
    return po.lmpc(inst, solve=False)


def solve(inst):
    """the oracle's solve, with z replaced by the exact solution of its final active set"""
    o = po.lmpc(inst)
    o["z"] = exact_active_set_solution(o)
    return o


def _betas(q):
    return [q[k] for k in ("beq", "bineq", "ub", "lb")]


def _finite_diff(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    ok = (np.abs(a) < 1e300) & (np.abs(b) < 1e300)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.where(ok, b - a, 0.0)


def gbar(o, dcontrol=None, dtraj=None):
    nx = o["Phi"].shape[1]
    g = np.zeros(o["Q"].shape[0])
    if dcontrol is not None:
        g[nx:] += dcontrol
    if dtraj is not None:
        g[:nx] += o["Phi"].T @ dtraj
        g[nx:] += o["Psi"].T @ dtraj
    return g


def outputs(o, z):
    """(control, trajectory) of the solution z of the build `o`"""
    nx = o["Phi"].shape[1]
    return z[nx:], o["Phi"] @ z[:nx] + o["Psi"] @ z[nx:] + o["xi"]


def vjp(inst, dcontrol=None, dtraj=None, o=None):
    """{key: dL/dinput} for L = dcontrol' control + dtraj' trajectory: every key of vector_keys, and "R" when given"""
    o = solve(inst) if o is None else o
    qo = dict(o, x=o["z"])
    g = qr.closed_form(qo, gbar(o, dcontrol, dtraj))
    nx = o["Phi"].shape[1]
    q0 = build(inst)
    out = {}
    for key in vector_keys(inst):
        v = get(inst, key)
        grad = np.zeros(v.shape)
        for idx in np.ndindex(v.shape):
            if not np.isfinite(v[idx]):
                continue
            e = np.zeros(v.shape)
            e[idx] = 1.0
            q1 = build(moved(inst, {key: e}))
            val = float(g["c"] @ (q1["c"] - q0["c"]))
            for k in ("beq", "bineq", "ub", "lb"):
                val += float(g[k] @ _finite_diff(q0[k], q1[k]))
            grad[idx] = val
        out[key] = grad
    if inst.get("R") is not None:
        out[("R", None)] = g["Q"][:nx, :nx]
    return out


def jvp(inst, tangent, o=None):
    """(dcontrol, dtrajectory) along `tangent` ({key: array}; ("R", None) moves R through its symmetric part)"""
    o = solve(inst) if o is None else o
    nx = o["Phi"].shape[1]
    vec = {k: v for k, v in tangent.items() if k[0] != "R"}
    q0, q1 = build(inst), build(moved(inst, vec))
    cdot = q1["c"] - q0["c"]
    if ("R", None) in tangent:
        Rd = np.asarray(tangent[("R", None)], float)
        cdot[:nx] += 0.5 * (Rd + Rd.T) @ o["z"][:nx]
    bdot = np.concatenate([_finite_diff(a, b) for a, b in zip(_betas(q0), _betas(q1))])
    act = np.asarray(o["iact"], int) - 1
    n = o["Q"].shape[0]
    zdot = qr._kkt_solve(o, np.concatenate([-cdot, bdot[act]]))[:n]
    return zdot[nx:], o["Phi"] @ zdot[:nx] + o["Psi"] @ zdot[nx:]


def dot(grad, tangent):
    return float(sum(np.sum(np.asarray(grad[k]) * np.asarray(t)) for k, t in tangent.items()))


def random_tangent(inst, rng, with_R=True):
    """a random direction over every input (0 on infinite bound entries; R's direction is not symmetric on purpose)"""
    t = {}
    for k in vector_keys(inst):
        v = get(inst, k)
        t[k] = np.where(np.isfinite(v), rng.normal(size=v.shape), 0.0)
    if with_R and inst.get("R") is not None:
        t[("R", None)] = rng.normal(size=(inst["nx"], inst["nx"]))
    return t


def active_set_loss(inst, iact, dcontrol, dtraj):
    """L at the exact solution of `inst`'s build on the fixed active set `iact`"""
    q = build(inst)
    z = exact_active_set_solution(dict(q, iact=iact))
    u, x = outputs(q, z)
    return float(dcontrol @ u + dtraj @ x)


def oracle_loss(inst, dcontrol, dtraj):
    o = po.lmpc(inst)
    return float(dcontrol @ o["control"] + dtraj @ o["trajectory"]), o
