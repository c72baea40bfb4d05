"""TEST INFRASTRUCTURE -- a dense numpy reference for the vector-Jacobian product of one LMPC instance (copra_b200_lmpc_vjp).

It takes the CPU oracle's QP and active set and solves the adjoint KKT system densely:
    [Q A'; A 0] [v; mu] = [gbar; 0],   gbar = dL/dU + Psi' dL/dtrajectory,
with A the active rows in their natural orientation (Aeq / Aineq rows, e_k for either bound).  Then dL/dc = -v and dL/dbeta_j
= mu_j.  Since c, beq, bineq, lb and ub are affine in the vector inputs, the directional derivative along an input direction
delta is  <dL/dc, c(theta + delta) - c(theta)> + <dL/dbeta, beta(theta + delta) - beta(theta)> + <Phi' dL/dtrajectory, delta_x0>,
with the QP terms differenced on the oracle's own builds.  Per-step entries go to the oracle in their autoSpan'd full-size form
(workloads.spanned), whose vectors have the same layout.
"""
import copy

import numpy as np

from copra_b200 import workloads as wl
from oracle import pyoracle as po


def vector_keys(inst):
    """the vector inputs of an instance: ("x0",), ("p", i), ("f", j), ("lower", j), ("upper", j)"""
    keys = [("x0", None)]
    keys += [("p", i) for i in range(len(inst["costs"]))]
    for j, c in enumerate(inst["constraints"]):
        if c["kind"] in ("trajectory_bound", "control_bound"):
            keys += [("lower", j), ("upper", j)]
        else:
            keys.append(("f", j))
    return keys


def get_vector(inst, key):
    kind, i = key
    if kind == "x0":
        return np.asarray(inst["x0"], float)
    return np.asarray((inst["costs"] if kind == "p" else inst["constraints"])[i][kind], float)


def with_vectors(inst, vecs):
    """copy of `inst` with the vectors of `vecs` ({key: array}) replaced"""
    out = copy.copy(inst)
    out["costs"] = [dict(c) for c in inst["costs"]]
    out["constraints"] = [dict(c) for c in inst["constraints"]]
    for (kind, i), v in vecs.items():
        if kind == "x0":
            out["x0"] = v
        else:
            (out["costs"] if kind == "p" else out["constraints"])[i][kind] = v
    return out


def oracle_problem(inst):
    per_step = any(c.get("per_step") for c in inst["costs"] + inst["constraints"])
    return wl.spanned(inst) if per_step else inst


def solve(inst):
    return po.lmpc(oracle_problem(inst))


def build(inst):
    return po.lmpc(oracle_problem(inst), solve=False)


def loss(o, dcontrol, dtraj):
    val = 0.0
    if dcontrol is not None:
        val += float(np.dot(dcontrol, o["control"]))
    if dtraj is not None:
        val += float(np.dot(dtraj, o["trajectory"]))
    return val


def adjoint(o, dcontrol=None, dtraj=None):
    """dL/dc and dL/d(beq | bineq | ub | lb) of a solved oracle instance (LMPC mode: nvar == nU)"""
    Q = o["Q"]
    n = Q.shape[0]
    meq, m = o["Aeq"].shape[0], o["Aineq"].shape[0]
    gbar = np.zeros(n) if dcontrol is None else np.asarray(dcontrol, float).copy()
    if dtraj is not None:
        gbar += o["Psi"].T @ dtraj
    rows = []
    for k in np.asarray(o["iact"], int) - 1:
        if k < meq:
            rows.append(o["Aeq"][k])
        elif k < meq + m:
            rows.append(o["Aineq"][k - meq])
        else:
            e = np.zeros(n)
            e[(k - meq - m) % n] = 1.0
            rows.append(e)
    A = np.array(rows).reshape(-1, n)
    na = A.shape[0]
    K = np.block([[Q, A.T], [A, np.zeros((na, na))]])
    sol = np.linalg.solve(K, np.concatenate([gbar, np.zeros(na)]))
    v, mu = sol[:n], sol[n:]
    beta = np.zeros(meq + m + 2 * n)
    beta[np.asarray(o["iact"], int) - 1] = mu
    return dict(c=-v, beq=beta[:meq], bineq=beta[meq:meq + m], ub=beta[meq + m:meq + m + n], lb=beta[meq + m + n:],
                x0=(o["Phi"].T @ dtraj) if dtraj is not None else np.zeros(o["Phi"].shape[1]))


def _finite_diff(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    ok = (np.abs(a) < 1e300) & (np.abs(b) < 1e300)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.where(ok, b - a, 0.0)


def directional(inst, adj, delta):
    """<VJP, delta> from the adjoint `adj` of `inst` and an input direction `delta` ({key: array}, 0 on infinite entries)"""
    q0 = build(inst)
    q1 = build(with_vectors(inst, {k: get_vector(inst, k) + d for k, d in delta.items()}))
    val = float(adj["c"] @ (q1["c"] - q0["c"]))
    for k in ("beq", "bineq", "ub", "lb"):
        val += float(adj[k] @ _finite_diff(q0[k], q1[k]))
    if ("x0", None) in delta:
        val += float(adj["x0"] @ delta[("x0", None)])
    return val


def c2_floor(batch):
    """C2 with a finite lower trajectory bound (velocity line) and a full-size control bound.  Quirk Q1: the reference keeps
    the lower rows un-negated, so `lower` acts as v <= -1 at every step -- active for the instances whose velocity target is
    above it; x0 satisfies it."""
    bp = wl.c2(batch=batch)
    N = bp["N"]
    tb, cb = bp["constraints"]
    bp["name"] = "C2-floor"
    bp["constraints"] = [dict(tb, lower=np.array([-np.inf, -1.0])),
                         dict(cb, lower=np.full(N, -np.inf), upper=np.tile(np.asarray(cb["upper"]), (1, N)))]
    return bp


def random_direction(inst, rng, keys=None):
    """a random direction over every vector input (0 on infinite bound entries)"""
    out = {}
    for k in keys or vector_keys(inst):
        v = get_vector(inst, k)
        out[k] = np.where(np.isfinite(v), rng.normal(size=v.shape), 0.0)
    return out
