"""Cost of the sensitivities of an initial-state batch (copra_b200_lmpc_vjp_initial_state / _jvp_initial_state) against the
forward step on the B200.

Workload: C4 (copra::InitialStateLMPC, nx = 2, N = 50, nvar = 52) x 8192 in one process, timed five ways: the forward step
(copra_b200_lmpc_run: build, solve, rollout), the vector VJP (x0, p, lower / upper), the VJP with R, r, x0lb and x0ub as well,
and the JVP along 1 and along nx tangent directions (r and x0lb).  Parameters, cotangents, tangents and outputs are
device-resident; the engine runs on its own stream, each call sits between CUDA events on it with the L2 overwritten before
(a 256 MB fill, completed before the timed window); mean of --steps after --warmup.  The sensitivities refer to the last
forward step.  Prints the card's name and power limit and writes JSON to --out.

    python tools/bench_initial_state_sens.py --out DIR [--steps 10 --warmup 3 --batch 8192]
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8192)
    a = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    eng = capi.Engine(0, stream=C.c_void_p(stream.cuda_stream))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB of L2
    B = a.batch
    bp = wl.c4(batch=B)
    hb = capi.HostBatch(bp, device_tensors=dev)
    s = eng.sizes(hb)
    nx, nU, X = int(bp["nx"]), s["nU"], s["X"]
    res = dict(control=torch.empty((B, nU), dtype=torch.float64, device=dev),
               trajectory=torch.empty((B, X), dtype=torch.float64, device=dev),
               status=torch.empty(B, dtype=torch.int32, device=dev), nact=torch.empty(B, dtype=torch.int32, device=dev))
    r = capi.Results()
    r.memory = capi.DEVICE
    for k, t in res.items():
        setattr(r, k, t.data_ptr())
    gen = torch.Generator(device=dev).manual_seed(1)
    dc = torch.randn((B, nU), dtype=torch.float64, device=dev, generator=gen)
    dt = torch.randn((B, X), dtype=torch.float64, device=dev, generator=gen)
    nplen = [int(np.asarray(c["p"]).shape[-1]) for c in bp["costs"]]
    g = dict(x0=torch.empty((B, nx), dtype=torch.float64, device=dev),
             p=[torch.empty((B, n), dtype=torch.float64, device=dev) for n in nplen],
             upper=torch.empty((B, 1), dtype=torch.float64, device=dev),
             R=torch.empty((B, nx, nx), dtype=torch.float64, device=dev),
             **{k: torch.empty((B, nx), dtype=torch.float64, device=dev) for k in ("r", "x0lb", "x0ub")})
    pp = (C.c_void_p * len(nplen))(*[t.data_ptr() for t in g["p"]])
    up = (C.c_void_p * 1)(g["upper"].data_ptr())
    out = capi.VjpOut()
    out.x0, out.p, out.upper = g["x0"].data_ptr(), C.cast(pp, C.POINTER(C.c_void_p)), C.cast(up, C.POINTER(C.c_void_p))
    init = capi.VjpInitialOut()
    for k in capi.INITIAL_KEYS:
        setattr(init, k, g[k].data_ptr())
    tang = {k: torch.randn((B, k, nx), dtype=torch.float64, device=dev, generator=gen) for k in (1, nx)}
    tr = {k: torch.randn((B, k, nx), dtype=torch.float64, device=dev, generator=gen) for k in (1, nx)}
    jout = {k: (torch.empty((B, k, nU), dtype=torch.float64, device=dev), torch.empty((B, k, X), dtype=torch.float64, device=dev))
            for k in (1, nx)}
    torch.cuda.synchronize()

    def forward():
        eng._check(eng.lib.copra_b200_lmpc_run(eng.h, C.byref(hb.problem), C.byref(r)))

    def vjp(ini):
        return lambda: eng._check(eng.lib.copra_b200_lmpc_vjp_initial_state(eng.h, dc.data_ptr(), dt.data_ptr(), capi.DEVICE,
                                                                            C.byref(out), ini and C.byref(ini)))

    def jvp(k):
        t = capi.JvpIn()
        t.ndir = k
        ti = capi.JvpInitialIn()
        ti.r, ti.x0lb = tr[k].data_ptr(), tang[k].data_ptr()
        du, dx = jout[k]
        return lambda: eng._check(eng.lib.copra_b200_lmpc_jvp_initial_state(eng.h, C.byref(t), C.byref(ti), capi.DEVICE,
                                                                            du.data_ptr(), dx.data_ptr()))

    forward()
    solver = eng.last_solver()
    times = {}
    for key, call in (("forward", forward), ("vjp_vectors", vjp(None)), ("vjp_with_initial", vjp(init)), ("jvp_k1", jvp(1)),
                      ("jvp_knx", jvp(nx))):
        ts = []
        for k in range(a.warmup + a.steps):
            flush.fill_(k & 0xFF)
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            call()
            ev1.record(stream)
            torch.cuda.synchronize()
            if k >= a.warmup:
                ts.append(ev0.elapsed_time(ev1))
        times[key] = ts
    st, na = res["status"].cpu().numpy(), res["nact"].cpu().numpy()
    ok = st == 0
    mean = {k: float(np.mean(v)) for k, v in times.items()}
    line = dict(name="C4 x %d" % B, batch=B, nvar=s["nvar"], solver=solver, **{k + "_ms": v for k, v in mean.items()},
                **{k + "_over_forward": v / mean["forward"] for k, v in mean.items() if k != "forward"},
                **{k + "_ms_all": v for k, v in times.items()},
                nact_mean=float(na[ok].mean()), nact_max=int(na[ok].max()), solved_ok=int(ok.sum()))
    print(json.dumps({k: v for k, v in line.items() if not k.endswith("_all")}), flush=True)
    results = dict(gpu=gpu_info(), steps=a.steps, warmup=a.warmup, lines=[line])
    print("gpu:", results["gpu"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_initial_state_sens.json"), "w") as fh:
        json.dump(results, fh, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
