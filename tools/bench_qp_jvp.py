"""Cost of the forward-mode sensitivities of a raw QP batch (copra_b200_qp_jvp, copra_b200_qp_jacobian) against the forward
solve (copra_b200_solve_qp_batch) and the k = 1 VJP (copra_b200_qp_vjp) on the B200.

Workloads (those of tools/bench_qp_vjp.py): C2's QPs x 4096, downloaded from a build, through gi_small with the Hessian shared
(stride 0) and per instance; and a mid-size random batch (n = 128, meq = 4, m = 96, 2048 instances) through the general
kernel.  Each is timed five ways: the forward solve, the VJP without the Aeq / Aineq gradients (k = 1), the JVP along one
cdot per instance (k = 1), the JVP along 8 directions of every input including Aeq / Aineq (k = 8, with the lambda pass) and
the Jacobian dx/dc (k = n).  Inputs, tangents and outputs are device-resident; the engine runs on its own stream, each call
sits between CUDA events on it with the L2 overwritten before (a 256 MB fill, completed before the timed window); mean of
--steps after --warmup.  Prints the card's name and power limit and writes JSON to --out.

    python tools/bench_qp_jvp.py --out DIR [--steps 10 --warmup 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from copra_b200 import capi, workloads as wl  # noqa: E402

KEYS = capi.QP_VJP_WANT
KDIR = 8  # directions of the all-inputs JVP


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def c2_qps(eng, B):
    bp = wl.c2(batch=B)
    hb = capi.HostBatch(bp)
    eng.lmpc_run(hb)
    st = {k: eng.download(hb, k) for k in KEYS}
    return st


def random_qps(B, n, meq, m, seed=3):
    rng = np.random.default_rng(seed)
    L = rng.normal(size=(n, n))
    Q0 = L @ L.T / n + 0.5 * np.eye(n)
    Q = np.broadcast_to(Q0, (B, n, n)) + np.eye(n) * rng.uniform(0.0, 1.0, size=(B, 1, 1))
    xf = rng.normal(size=(B, n))
    Aeq = rng.normal(size=(meq, n))
    Aineq = rng.normal(size=(m, n))
    return dict(Q=Q, c=rng.normal(size=(B, n)), Aeq=np.broadcast_to(Aeq, (B, meq, n)), beq=xf @ Aeq.T,
                Aineq=np.broadcast_to(Aineq, (B, m, n)), bineq=xf @ Aineq.T + rng.uniform(0.0, 1.0, size=(B, m)),
                lb=xf - rng.uniform(0.1, 2.0, size=(B, n)), ub=xf + rng.uniform(0.1, 2.0, size=(B, n)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    eng = capi.Engine(0, stream=C.c_void_p(stream.cuda_stream))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB of L2
    results = dict(gpu=gpu_info(), lines=[])
    c2 = c2_qps(eng, 4096)
    c2_shared = dict(c2, Q=c2["Q"][0])
    workloads = (("C2 x 4096, shared Q", c2_shared), ("C2 x 4096, per-instance Q", c2),
                 ("random n=128 x 2048", random_qps(2048, 128, 4, 96)))
    for name, qp in workloads:
        n = qp["Q"].shape[-1]
        B = qp["c"].shape[0]
        meq = qp["Aeq"].shape[-2] if qp["Aeq"].size else 0
        m = qp["Aineq"].shape[-2] if qp["Aineq"].size else 0
        base = dict(Q=2, c=1, Aeq=2, beq=1, Aineq=2, bineq=1, lb=1, ub=1)
        live, cargs = [], []
        for k in KEYS:
            arr = capi.Array()
            v = np.asarray(qp[k], float)
            if v.size and (k not in ("Aeq", "beq") or meq) and (k not in ("Aineq", "bineq") or m):
                t = torch.tensor(np.swapaxes(v, -1, -2) if base[k] == 2 else v, device=dev).contiguous()
                live.append(t)
                arr.ptr, arr.stride = t.data_ptr(), (t[0].numel() if v.ndim > base[k] else 0)
            cargs.append(arr)
        x = torch.empty((B, n), dtype=torch.float64, device=dev)
        ints = {k: torch.empty((B, w), dtype=torch.int32, device=dev) for k, w in (("status", 1), ("iters", 2), ("nact", 1), ("iact", n))}
        gen = torch.Generator(device=dev).manual_seed(1)
        dx = torch.randn((B, n), dtype=torch.float64, device=dev, generator=gen)
        outs = dict(Q=(n, n), c=(n,), Aeq=(meq, n), beq=(meq,), Aineq=(m, n), bineq=(m,), lb=(n,), ub=(n,))
        grads = {k: torch.empty((B,) + s, dtype=torch.float64, device=dev) for k, s in outs.items() if all(s)}
        part = capi.QpVjpOut()
        for k, g in grads.items():
            if k not in ("Aeq", "Aineq"):
                setattr(part, k, g.data_ptr())
        # tangents: one cdot per instance (k = 1), and 8 random directions per instance of every input (k = 8)
        tc1 = torch.randn((B, 1, n), dtype=torch.float64, device=dev, generator=gen)
        t8 = {k: torch.randn((B, KDIR) + s, dtype=torch.float64, device=dev, generator=gen) for k, s in outs.items() if all(s)}
        jin1, jin8 = capi.QpJvpIn(), capi.QpJvpIn()
        jin1.ndir, jin8.ndir = 1, KDIR
        jin1.c.ptr, jin1.c.stride = tc1.data_ptr(), n
        for k, t in t8.items():
            getattr(jin8, k).ptr, getattr(jin8, k).stride = t.data_ptr(), t[0].numel()
        xd1 = torch.empty((B, 1, n), dtype=torch.float64, device=dev)
        xd8 = torch.empty((B, KDIR, n), dtype=torch.float64, device=dev)
        jac = torch.empty((B, n, n), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()

        def forward():
            eng._check(eng.lib.copra_b200_solve_qp_batch(eng.h, n, meq, m, B, *cargs, x.data_ptr(), ints["status"].data_ptr(),
                                                         ints["iters"].data_ptr(), ints["nact"].data_ptr(),
                                                         ints["iact"].data_ptr(), capi.DEVICE))

        def vjp():
            eng._check(eng.lib.copra_b200_qp_vjp(eng.h, dx.data_ptr(), capi.DEVICE, C.byref(part)))

        def jvp(t, out):
            return lambda: eng._check(eng.lib.copra_b200_qp_jvp(eng.h, C.byref(t), capi.DEVICE, out.data_ptr()))

        def jacobian():
            eng._check(eng.lib.copra_b200_qp_jacobian(eng.h, capi.QP_WRT["c"], jac.data_ptr(), capi.DEVICE))

        forward()
        solver = eng.last_solver()
        times, launches = {}, {}
        for key, call in (("forward", forward), ("vjp_k1", vjp), ("jvp_k1", jvp(jin1, xd1)), ("jvp_k8_all", jvp(jin8, xd8)),
                          ("jacobian_c", jacobian)):
            ts = []
            for k in range(a.warmup + a.steps):
                flush.fill_(k & 0xFF)
                torch.cuda.synchronize()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n0 = eng.launch_count()
                ev0.record(stream)
                call()
                ev1.record(stream)
                torch.cuda.synchronize()
                launches[key] = eng.launch_count() - n0
                if k >= a.warmup:
                    ts.append(ev0.elapsed_time(ev1))
            times[key] = ts
        st, na = ints["status"][:, 0].cpu().numpy(), ints["nact"][:, 0].cpu().numpy()
        ok = st == 0
        mean = {k: float(np.mean(v)) for k, v in times.items()}
        line = dict(name=name, batch=B, n=n, meq=meq, m=m, k=KDIR, shared_Q=bool(qp["Q"].ndim == 2), solver=solver,
                    **{k + "_ms": v for k, v in mean.items()},
                    **{k + "_over_forward": mean[k] / mean["forward"] for k in mean if k != "forward"},
                    **{k + "_over_vjp_k1": mean[k] / mean["vjp_k1"] for k in ("jvp_k1", "jvp_k8_all", "jacobian_c")},
                    launches=launches, **{k + "_ms_all": v for k, v in times.items()},
                    nact_mean=float(na[ok].mean()), nact_max=int(na[ok].max()), solved_ok=int(ok.sum()))
        print(json.dumps({k: v for k, v in line.items() if not k.endswith("_all")}), flush=True)
        results["lines"].append(line)
    print("gpu:", results["gpu"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_qp_jvp.json"), "w") as fh:
        json.dump(results, fh, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
