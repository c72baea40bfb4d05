"""torch.autograd through a batch of LMPC solves: the forward runs copra_b200_lmpc_run on CUDA tensors, the backward the exact
vector-Jacobian product of copra_b200_lmpc_vjp (K8) on the same engine, and forward-mode AD (torch.autograd.forward_ad) the
exact Jacobian-vector product of copra_b200_lmpc_jvp (K9).

    ctrl, traj = copra_b200.autograd.lmpc(engine, bp, x0, p=[...], f=[...], lower=[...], upper=[...], w=[...], M=[...], N=[...],
                                          A=A, B=B, d=d, E=[...], G=[...])

`bp` is a workloads-style batch problem that fixes the matrices (A, B, d, M, N, w, E, G) and the kinds and shapes of every
entry; the vectors are CUDA float64 tensors, batch-major (batch, length), one per cost (p) and one per constraint (f for row
constraints, lower / upper for bounds; None keeps bp's value, which then gets no gradient).  Every instance gets its own
gradient.  The cost weights and matrices w (rows), M (rows, nx) and N (rows, nu) may be given per cost as CUDA float64
tensors too, in reverse mode only (copra_b200_lmpc_vjp_costs): a batched tensor (leading batch axis) gets per-instance
gradients; an unbatched one is shared by the batch (stride 0: the Hessian stays batch-invariant) and its gradient is the sum
over the batch.  The dynamics A (nx, nx), B (nx, nu), d (nx,) and every row constraint's E (rows, nx) / G (rows, nu) may be
given the same way (copra_b200_lmpc_vjp_model), with the same batched / shared rule.  A non-zero forward-mode tangent on any
of these matrices raises NotImplementedError.  The backward and the forward-mode tangent raise if another solve ran on the
engine since this forward: the engine keeps only the last solve.

An initial-state build (copra::InitialStateLMPC: x0 is optimised inside the box [x0lb, x0ub] with the cost
1/2 x0'R x0 + r'x0) is differentiable the same way, in reverse and in forward mode (copra_b200_lmpc_vjp_initial_state /
_jvp_initial_state), with respect to x0 and the vectors and to R, r, x0lb and x0ub:

    ctrl, traj = copra_b200.autograd.initial_state_lmpc(engine, bp, x0, R=..., r=..., x0lb=..., x0ub=..., p=[...], ...)

R (nx, nx), r, x0lb and x0ub (nx,) follow the batched / shared rule above; R is read through its symmetric part, so its
gradient is symmetric.  x0 enters such a build only as the default of an x0 bound that is not given, so its gradient is
zero when both x0lb and x0ub are.

A batch of raw QPs  min 1/2 x'Qx + c'x  s.t.  Aeq x = beq, Aineq x <= bineq, lb <= x <= ub  is differentiable the same way, in
reverse mode (copra_b200_qp_vjp), with respect to every tensor given:

    x, status = copra_b200.autograd.qp(engine, Q, c, Aeq=..., beq=..., Aineq=..., bineq=..., lb=..., ub=...)

Each input is a CUDA float64 tensor with an optional leading batch axis: a batched tensor gets per-instance gradients, an
unbatched one is shared by the batch (stride 0) and its gradient is the sum over the batch.  lb / ub default to -inf / +inf.
Q is read as a symmetric matrix, so its gradient is the symmetric one.  `status` is not differentiable; instances whose status
is not 0 get zero gradients.
"""
import ctypes as C

import numpy as np
import torch

from . import capi


def _vector_entries(bp):
    """(kind, index) of every cost's p and every constraint's f or lower / upper"""
    keys = [("p", i) for i in range(len(bp["costs"]))]
    for j, c in enumerate(bp["constraints"]):
        keys += [("lower", j), ("upper", j)] if c["kind"] in ("trajectory_bound", "control_bound") else [("f", j)]
    return keys


_COST_KEYS = ("w", "M", "N")
_SYSTEM_KEYS = ("A", "B", "d")
_MODEL_KEYS = _SYSTEM_KEYS + ("E", "G")
_MATRIX_KEYS = _COST_KEYS + _MODEL_KEYS  # reverse mode only
_TOP_KEYS = _SYSTEM_KEYS + capi.INITIAL_KEYS  # one per problem, not per cost / constraint
_BASE_NDIM = dict(w=1, M=2, N=2, A=2, B=2, d=1, E=2, G=2, R=2, r=1, x0lb=1, x0ub=1)


def _point(arr, t, base):
    """point the ctypes Array `arr` at the tensor t (logical row-major, base dims plus an optional leading batch axis)"""
    t = t.detach().to(torch.float64)
    if base == 2:
        t = t.transpose(-1, -2)  # the engine reads matrices column-major
    t = t.contiguous()
    arr.ptr, arr.stride = t.data_ptr(), (t[0].numel() if t.dim() > base else 0)
    return t


def _patch_cost_matrix(problem, pr, kind, i, t):
    """point cost i's `kind` (w, M or N) of the packed problem at the tensor t (batched or shared, logical row-major)"""
    rows, has_m, has_n = capi.cost_shapes(problem)[i]
    if (kind == "M" and not has_m) or (kind == "N" and not has_n):
        raise ValueError("cost %d (%s) has no %s" % (i, problem["costs"][i]["kind"], kind))
    base = _BASE_NDIM[kind]
    if t.dim() not in (base, base + 1) or t.shape[-base] != rows:
        raise ValueError("cost %d: %s has shape %s, expected %d rows (with an optional leading batch axis)"
                         % (i, kind, tuple(t.shape), rows))
    return _point(getattr(pr.costs[i], kind), t, base)


def _patch_model_matrix(bp, pr, kind, i, t):
    """point A, B, d, R, r, x0lb or x0ub, or constraint i's E or G, of the packed problem at the tensor t (batched or
    shared)"""
    nx, nu = int(bp["nx"]), int(bp["nu"])
    if kind in ("E", "G"):
        rows, has_e, has_g = capi.cstr_shapes(bp)[i]
        if not (has_e if kind == "E" else has_g):
            raise ValueError("constraint %d (%s) has no %s" % (i, bp["constraints"][i]["kind"], kind))
        shape = (rows, nx if kind == "E" else nu)
    else:
        shape = dict(A=(nx, nx), B=(nx, nu), d=(nx,), R=(nx, nx), r=(nx,), x0lb=(nx,), x0ub=(nx,))[kind]
    if t.dim() not in (len(shape), len(shape) + 1) or tuple(t.shape[t.dim() - len(shape):]) != shape:
        raise ValueError("%s has shape %s, expected %s (with an optional leading batch axis)" % (kind, tuple(t.shape), shape))
    return _point(getattr(pr.cstrs[i] if kind in ("E", "G") else pr, kind), t, len(shape))


def _check_resident(ctx, what):
    if ctx.engine.solve_count != ctx.count:
        raise RuntimeError("copra_b200.autograd: another solve ran on this engine since the forward; the %s needs the active "
                           "sets of the solve being differentiated" % what)


class _LMPC(torch.autograd.Function):
    """an LMPC-mode or an initial-state build (bp["initial_state"]): the forward solves it, the backward and the
    forward-mode tangent run the engine's VJP and JVP of that build mode"""

    @staticmethod
    def forward(ctx, engine, bp, keys, x0, *vecs):
        B = int(bp["batch"])
        dev = x0.device
        problem = dict(bp)
        problem["costs"] = [dict(c) for c in bp["costs"]]
        problem["constraints"] = [dict(c) for c in bp["constraints"]]
        problem["x0"] = np.zeros((B, int(bp["nx"])))
        for (kind, i), v in zip(keys, vecs):
            if v is None:  # shape only: the tensor itself is patched in below
                continue
            if kind in _TOP_KEYS:
                problem[kind] = np.zeros(tuple(v.shape))
            else:
                (problem["costs"] if kind in ("p",) + _COST_KEYS else problem["constraints"])[i][kind] = np.zeros(tuple(v.shape))
        hb = capi.HostBatch(problem, device_tensors=dev)
        live = [x0.detach().contiguous()]
        pr = hb.problem
        pr.x0.ptr, pr.x0.stride = live[0].data_ptr(), live[0].shape[1]
        for (kind, i), v in zip(keys, vecs):
            if v is None:
                continue
            if kind in _COST_KEYS:
                live.append(_patch_cost_matrix(problem, pr, kind, i, v))
                continue
            if kind in _BASE_NDIM:
                live.append(_patch_model_matrix(bp, pr, kind, i, v))
                continue
            t = v.detach().contiguous()
            live.append(t)
            arr = getattr(pr.costs[i] if kind == "p" else pr.cstrs[i], kind)
            arr.ptr, arr.stride = t.data_ptr(), t.shape[1]
        s = engine.sizes(hb)
        control = torch.empty((B, s["nU"]), dtype=torch.float64, device=dev)
        traj = torch.empty((B, s["X"]), dtype=torch.float64, device=dev)
        r = capi.Results()
        r.memory = capi.DEVICE
        r.control, r.trajectory = control.data_ptr(), traj.data_ptr()
        torch.cuda.synchronize(dev)
        engine.solve_count += 1
        engine._last_bp = None
        engine._check(engine.lib.copra_b200_lmpc_run(engine.h, C.byref(pr), C.byref(r)))
        engine._last_bp = problem
        engine.synchronize()
        ctx.engine, ctx.count, ctx.keys, ctx.present = engine, engine.solve_count, keys, [v is not None for v in vecs]
        # the build reads x0 and the matrices where they live: the VJP of the cost and model matrices reads them again
        ctx.live = (hb, live)
        ctx.shared = [v is not None and kind in _BASE_NDIM and v.dim() == _BASE_NDIM[kind] for (kind, _), v in zip(keys, vecs)]
        ctx.initial = bool(bp.get("initial_state"))
        ctx.counts = (B, len(bp["costs"]), len(bp["constraints"]))
        ctx.mark_non_differentiable()
        return control, traj

    @staticmethod
    def jvp(ctx, _engine, _bp, _keys, dx0, *dvecs):
        # forward mode: one tangent direction through copra_b200_lmpc_jvp (_initial_state) (K9); the engine holds everything
        # it needs
        _check_resident(ctx, "JVP")
        B, ncost, ncstr = ctx.counts
        tangents = dict(p=[None] * ncost, f=[None] * ncstr, lower=[None] * ncstr, upper=[None] * ncstr)
        init = {}
        for (kind, i), t, shared in zip(ctx.keys, dvecs, ctx.shared):
            if t is None:
                continue
            if kind in _MATRIX_KEYS:
                if bool(torch.count_nonzero(t)):
                    raise NotImplementedError("copra_b200.autograd: forward-mode derivatives with respect to the cost weights "
                                              "and matrices (w, M, N) and the model (A, B, d, E, G) are not implemented; "
                                              "reverse mode (backward) is")
            elif kind in capi.INITIAL_KEYS:
                init[kind] = (t.expand(B, *t.shape) if shared else t).unsqueeze(1)
            else:
                tangents[kind][i] = t.unsqueeze(1)
        dx0 = dx0.unsqueeze(1) if dx0 is not None else None
        eng = ctx.engine
        du, dx = eng.initial_state_jvp(x0=dx0, **init, **tangents) if ctx.initial else eng.lmpc_jvp(x0=dx0, **tangents)
        return du[:, 0], dx[:, 0]

    @staticmethod
    def backward(ctx, dcontrol, dtraj):
        _check_resident(ctx, "VJP")
        want = capi.VJP_WANT + tuple(k for k in _BASE_NDIM if any(p and kind == k for (kind, _), p in zip(ctx.keys, ctx.present)))
        vjp = ctx.engine.initial_state_vjp if ctx.initial else ctx.engine.lmpc_vjp
        g = vjp(dcontrol=dcontrol, dtrajectory=dtraj, want=want)  # ordered against torch's stream on both sides
        grads = [g["x0"]]
        for (kind, i), present, shared in zip(ctx.keys, ctx.present, ctx.shared):
            grad = (g[kind] if kind in _TOP_KEYS else g[kind][i]) if present else None
            grads.append(grad.sum(0) if shared else grad)  # a shared input's gradient sums its instances'
        return (None, None, None, *grads)


def _apply(engine, bp, keys, x0, given):
    """_LMPC of the inputs `given` (lists indexed by cost / constraint, None entries keep bp's values) in the order of
    `keys`"""
    vecs = [given[k][i] if i < len(given[k]) else None for k, i in keys]
    return _LMPC.apply(engine, bp, keys, x0, *vecs)


def lmpc(engine, bp, x0, p=None, f=None, lower=None, upper=None, w=None, M=None, N=None, A=None, B=None, d=None, E=None,
         G=None):
    """(control, trajectory) of the batch problem `bp` with the given inputs, differentiable with respect to x0 and every
    vector, weight and matrix given (lists indexed by cost / constraint, None entries keep bp's values).  w, M and N are
    (rows,), (rows, nx) and (rows, nu) per cost, A, B and d (nx, nx), (nx, nu) and (nx,), E and G (rows, nx) and (rows, nu)
    per row constraint, each with an optional leading batch axis; reverse mode only for these."""
    ncost, ncstr = len(bp["costs"]), len(bp["constraints"])
    keys = (_vector_entries(bp) + [(k, i) for i in range(ncost) for k in _COST_KEYS] + [(k, 0) for k in _SYSTEM_KEYS]
            + [(k, j) for j in range(ncstr) for k in ("E", "G")])
    return _apply(engine, bp, keys, x0, dict(p=p or [], f=f or [], lower=lower or [], upper=upper or [], w=w or [], M=M or [],
                                             N=N or [], A=[A], B=[B], d=[d], E=E or [], G=G or []))


def initial_state_lmpc(engine, bp, x0, R=None, r=None, x0lb=None, x0ub=None, p=None, f=None, lower=None, upper=None):
    """(control, trajectory) of the initial-state batch problem `bp` with the given inputs, differentiable in reverse and in
    forward mode with respect to x0, R (nx, nx), r, x0lb, x0ub (nx,) (each with an optional leading batch axis) and every
    vector given (lists indexed by cost / constraint, as lmpc); None keeps bp's value, which then gets no gradient"""
    if not bp.get("initial_state"):
        raise ValueError("initial_state_lmpc takes an initial-state problem; copra_b200.autograd.lmpc takes LMPC-mode ones")
    keys = [(k, 0) for k in capi.INITIAL_KEYS] + _vector_entries(bp)
    return _apply(engine, bp, keys, x0, dict(R=[R], r=[r], x0lb=[x0lb], x0ub=[x0ub], p=p or [], f=f or [], lower=lower or [],
                                             upper=upper or []))


class _QP(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, keys, *arrs):
        live = [a.detach() for a in arrs]
        given = dict(zip(keys, live))
        r = engine.solve_qp_batch(*[given.get(k) for k in capi.QP_VJP_WANT])  # keeps its device inputs alive for the VJP
        ctx.engine, ctx.count, ctx.keys = engine, engine.solve_count, keys
        ctx.shared = [a.dim() == capi.QP_BASE_NDIM[k] for k, a in zip(keys, arrs)]
        ctx.mark_non_differentiable(r["status"])
        ctx.x_like = (tuple(r["x"].shape), r["x"].device)
        return r["x"], r["status"]

    @staticmethod
    def jvp(ctx, _engine, _keys, *tangents):
        if any(t is not None and bool(torch.count_nonzero(t)) for t in tangents):
            raise NotImplementedError("copra_b200.autograd.qp: forward-mode derivatives of a raw QP batch are not implemented; "
                                      "reverse mode (backward) is")
        shape, dev = ctx.x_like
        return torch.zeros(shape, dtype=torch.float64, device=dev), None

    @staticmethod
    def backward(ctx, dx, _dstatus):
        eng = ctx.engine
        if eng.solve_count != ctx.count:
            raise RuntimeError("copra_b200.autograd: another solve ran on this engine since the forward; the VJP needs the "
                               "active sets of the solve being differentiated")
        want = tuple(k for k, need in zip(ctx.keys, ctx.needs_input_grad[2:]) if need)
        if not want:
            return (None,) * (2 + len(ctx.keys))
        g = eng.qp_vjp(dx, want=want)  # ordered against torch's stream on both sides
        grads = [None if g[k] is None else (g[k].sum(0) if shared else g[k]) for k, shared in zip(ctx.keys, ctx.shared)]
        return (None, None, *grads)


def qp(engine, Q, c, Aeq=None, beq=None, Aineq=None, bineq=None, lb=None, ub=None):
    """(x, status) of the batch of raw QPs given as CUDA float64 tensors (see the module docstring), differentiable with
    respect to every tensor given; lb / ub default to -inf / +inf"""
    n = Q.shape[-1]
    if lb is None:
        lb = torch.full((n,), -torch.inf, dtype=torch.float64, device=Q.device)
    if ub is None:
        ub = torch.full((n,), torch.inf, dtype=torch.float64, device=Q.device)
    given = dict(Q=Q, c=c, Aeq=Aeq, beq=beq, Aineq=Aineq, bineq=bineq, lb=lb, ub=ub)
    keys = tuple(k for k in capi.QP_VJP_WANT if given[k] is not None)
    return _QP.apply(engine, keys, *[given[k] for k in keys])
