"""torch.autograd through a batch of LMPC solves: the forward runs copra_b200_lmpc_run on CUDA tensors, the backward the exact
vector-Jacobian product of copra_b200_lmpc_vjp (K8) on the same engine, and forward-mode AD (torch.autograd.forward_ad) the
exact Jacobian-vector product of copra_b200_lmpc_jvp (K9).

    ctrl, traj = copra_b200.autograd.lmpc(engine, bp, x0, p=[...], f=[...], lower=[...], upper=[...])

`bp` is a workloads-style batch problem that fixes the matrices (A, B, d, M, N, w, E, G) and the kinds and shapes of every
entry; the vectors are CUDA float64 tensors, batch-major (batch, length), one per cost (p) and one per constraint (f for row
constraints, lower / upper for bounds; None keeps bp's value, which then gets no gradient).  Every instance gets its own
gradient.  The backward and the forward-mode tangent raise if another solve ran on the engine since this forward: the
engine keeps only the last solve.
"""
import ctypes as C

import numpy as np
import torch

from . import capi


def _vec_entries(bp):
    """(kind, index) of every vector input after x0, in the order of the Function's arguments"""
    keys = [("p", i) for i in range(len(bp["costs"]))]
    for j, c in enumerate(bp["constraints"]):
        keys += [("lower", j), ("upper", j)] if c["kind"] in ("trajectory_bound", "control_bound") else [("f", j)]
    return keys


class _LMPC(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, bp, keys, x0, *vecs):
        B = int(bp["batch"])
        dev = x0.device
        problem = dict(bp)
        problem["costs"] = [dict(c) for c in bp["costs"]]
        problem["constraints"] = [dict(c) for c in bp["constraints"]]
        problem["x0"] = np.zeros((B, int(bp["nx"])))
        for (kind, i), v in zip(keys, vecs):
            if v is not None:  # shape only: the tensor itself is patched in below
                (problem["costs"] if kind == "p" else problem["constraints"])[i][kind] = np.zeros(tuple(v.shape))
        hb = capi.HostBatch(problem, device_tensors=dev)
        live = [x0.detach().contiguous()]
        pr = hb.problem
        pr.x0.ptr, pr.x0.stride = live[0].data_ptr(), live[0].shape[1]
        for (kind, i), v in zip(keys, vecs):
            if v is None:
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
        ctx.counts = (len(bp["costs"]), len(bp["constraints"]))
        ctx.mark_non_differentiable()
        return control, traj

    @staticmethod
    def jvp(ctx, _engine, _bp, _keys, dx0, *dvecs):
        # forward mode: one tangent direction through copra_b200_lmpc_jvp (K9); the engine holds everything it needs
        eng = ctx.engine
        if eng.solve_count != ctx.count:
            raise RuntimeError("copra_b200.autograd: another solve ran on this engine since the forward; the JVP needs the "
                               "active sets of the solve being differentiated")
        ncost, ncstr = ctx.counts
        tangents = dict(p=[None] * ncost, f=[None] * ncstr, lower=[None] * ncstr, upper=[None] * ncstr)
        for (kind, i), t in zip(ctx.keys, dvecs):
            if t is not None:
                tangents[kind][i] = t.unsqueeze(1)
        du, dx = eng.lmpc_jvp(x0=dx0.unsqueeze(1) if dx0 is not None else None, **tangents)
        return du[:, 0], dx[:, 0]

    @staticmethod
    def backward(ctx, dcontrol, dtraj):
        eng = ctx.engine
        if eng.solve_count != ctx.count:
            raise RuntimeError("copra_b200.autograd: another solve ran on this engine since the forward; the VJP needs the "
                               "active sets of the solve being differentiated")
        g = eng.lmpc_vjp(dcontrol=dcontrol, dtrajectory=dtraj)  # ordered against torch's stream on both sides
        grads = [g["x0"]]
        for (kind, i), present in zip(ctx.keys, ctx.present):
            grads.append(g[kind][i] if present else None)
        return (None, None, None, *grads)


def lmpc(engine, bp, x0, p=None, f=None, lower=None, upper=None):
    """(control, trajectory) of the batch problem `bp` with the given vector inputs, differentiable with respect to x0 and
    every vector given (lists indexed by cost / constraint, None entries keep bp's values)."""
    keys = _vec_entries(bp)
    given = dict(p=p or [], f=f or [], lower=lower or [], upper=upper or [])
    vecs = [given[k][i] if i < len(given[k]) else None for k, i in keys]
    return _LMPC.apply(engine, bp, keys, x0, *vecs)
