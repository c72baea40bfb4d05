"""Cost of the gradients with respect to the dynamics and the row constraints' matrices (copra_b200_lmpc_vjp_model: K8 with
the forward solve as a second right-hand side, then k8_model_grad) against a plain VJP and the forward step on the B200.

For C3 x 16384, C3-walk x 16384 and C2 x 4096: the forward step (build + solve, copra_b200_lmpc_run with device-resident
inputs and outputs), one VJP with device-resident cotangents and gradients (dL/dcontrol and dL/dtrajectory in, every vector
gradient out) and the same VJP with the A, B, d gradients and every row constraint's E and G gradient as well, each between
CUDA events on the engine's stream with the L2 overwritten before it (a 256 MB fill, completed before the timed window), mean
of --steps after --warmup.  Records the ratios of the model-gradient VJP to the plain VJP and to the forward step; prints the
card's name and power limit and writes JSON to --out.

    python tools/bench_vjp_model.py --out DIR [--steps 5 --warmup 2]
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
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    import torch
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    eng = capi.Engine(0, stream=C.c_void_p(stream.cuda_stream))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB of L2
    results = dict(gpu=gpu_info(), lines=[])
    for name, bp in (("C3", wl.c3(16384)), ("C3-walk", wl.c3_walk(16384)), ("C2", wl.c2(4096))):
        hb = capi.HostBatch(bp, device_tensors=dev)
        s = eng.sizes(hb)
        B = bp["batch"]
        bufs = dict(control=torch.empty((B, s["nU"]), dtype=torch.float64, device=dev),
                    trajectory=torch.empty((B, s["X"]), dtype=torch.float64, device=dev),
                    status=torch.empty(B, dtype=torch.int32, device=dev), nact=torch.empty(B, dtype=torch.int32, device=dev))
        r = capi.Results()
        r.memory = capi.DEVICE
        for k, t in bufs.items():
            setattr(r, k, t.data_ptr())
        g = torch.Generator(device=dev).manual_seed(1)
        dc = torch.randn((B, s["nU"]), dtype=torch.float64, device=dev, generator=g)
        dt = torch.randn((B, s["X"]), dtype=torch.float64, device=dev, generator=g)
        eng._last_bp = bp

        def forward():
            eng._check(eng.lib.copra_b200_lmpc_run(eng.h, C.byref(hb.problem), C.byref(r)))

        def vjp():
            eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt)

        def vjp_model():
            eng.lmpc_vjp(dcontrol=dc, dtrajectory=dt, want=capi.VJP_WANT + capi.VJP_MODEL_WANT)

        times = {}
        for key, call in (("forward", forward), ("vjp", vjp), ("vjp_model", vjp_model)):
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
        st, na = bufs["status"].cpu().numpy(), bufs["nact"].cpu().numpy()
        ok = st == 0
        fwd, vjp_ms, model_ms = (float(np.mean(times[k])) for k in ("forward", "vjp", "vjp_model"))
        line = dict(name=name, batch=B, n=s["nvar"], forward_ms=fwd, vjp_ms=vjp_ms, vjp_model_ms=model_ms,
                    forward_ms_all=times["forward"], vjp_ms_all=times["vjp"], vjp_model_ms_all=times["vjp_model"],
                    vjp_model_over_vjp=model_ms / vjp_ms, vjp_model_over_forward=model_ms / fwd,
                    model_grad_extra_over_vjp=(model_ms - vjp_ms) / vjp_ms,
                    nact_mean=float(na[ok].mean()), nact_max=int(na[ok].max()), solved_ok=int(ok.sum()), solver=eng.last_solver())
        print(json.dumps({k: v for k, v in line.items() if not k.endswith("_all")}), flush=True)
        results["lines"].append(line)
    print("gpu:", results["gpu"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_vjp_model.json"), "w") as fh:
        json.dump(results, fh, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
