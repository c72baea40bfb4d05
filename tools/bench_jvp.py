"""Cost of the forward-mode sensitivities (copra_b200_lmpc_jvp / copra_b200_lmpc_feedback_gain, K9) on the B200.

For C3 x 16384, C3-walk x 16384 and C2 x 4096, each between CUDA events on the engine's stream with the L2 overwritten
before it, mean of --steps after --warmup, device-resident inputs and outputs:
  forward      the forward step (build + solve, copra_b200_lmpc_run)
  gain1        copra_b200_lmpc_feedback_gain(steps = 1), Ku only
  gainN        copra_b200_lmpc_feedback_gain(steps = N), Ku and Kx
  jvp1         copra_b200_lmpc_jvp with one random direction on x0, every p and every f / lower / upper
  vjp_nu       nu VJPs with unit dcontrol (dL/dx0 only): the way to get du0/dx0 without K9
Prints the card's name and power limit, and the ratios to the forward step; writes JSON to --out.

    python tools/bench_jvp.py --out DIR [--steps 5 --warmup 2]
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
    f64 = dict(dtype=torch.float64, device=dev)
    for name, bp in (("C3", wl.c3(16384)), ("C3-walk", wl.c3_walk(16384)), ("C2", wl.c2(4096))):
        hb = capi.HostBatch(bp, device_tensors=dev)
        s = eng.sizes(hb)
        B, nx, nu, N = bp["batch"], bp["nx"], bp["nu"], bp["N"]
        bufs = dict(control=torch.empty((B, s["nU"]), **f64), trajectory=torch.empty((B, s["X"]), **f64),
                    status=torch.empty(B, dtype=torch.int32, device=dev), nact=torch.empty(B, dtype=torch.int32, device=dev))
        r = capi.Results()
        r.memory = capi.DEVICE
        for k, t in bufs.items():
            setattr(r, k, t.data_ptr())
        eng._last_bp = bp
        # device-resident outputs and inputs
        Ku1 = torch.empty((B, nx, nu), **f64)
        KuN, KxN = torch.empty((B, nx, s["nU"]), **f64), torch.empty((B, nx, s["X"]), **f64)
        du, dx = torch.empty((B, s["nU"]), **f64), torch.empty((B, s["X"]), **f64)
        g = torch.Generator(device=dev).manual_seed(1)
        nx_, plen, clen = capi.vjp_lengths(bp)
        bound = [c["kind"] in ("trajectory_bound", "control_bound") for c in bp["constraints"]]
        keep = [torch.randn((B, nx), **f64, generator=g)]
        t = capi.JvpIn()
        t.ndir, t.x0 = 1, keep[0].data_ptr()
        for key, lens, on in (("p", plen, [True] * len(plen)), ("f", clen, [not x for x in bound]),
                              ("lower", clen, bound), ("upper", clen, bound)):
            ptrs = []
            for n_, use in zip(lens, on):
                if use:
                    keep.append(torch.randn((B, n_), **f64, generator=g))
                    ptrs.append(keep[-1].data_ptr())
                else:
                    ptrs.append(None)
            arr = (C.c_void_p * max(1, len(ptrs)))(*ptrs)
            keep.append(arr)
            setattr(t, key, C.cast(arr, C.POINTER(C.c_void_p)))
        units = []
        for k in range(nu):
            e = torch.zeros((B, s["nU"]), **f64)
            e[:, k] = 1.0
            units.append(e)
        gx0 = torch.empty((B, nx), **f64)
        vo = capi.VjpOut()
        vo.x0 = gx0.data_ptr()
        lib, h = eng.lib, eng.h

        def forward():
            eng._check(lib.copra_b200_lmpc_run(h, C.byref(hb.problem), C.byref(r)))

        def gain1():
            eng._check(lib.copra_b200_lmpc_feedback_gain(h, 1, Ku1.data_ptr(), None, capi.DEVICE))

        def gain_n():
            eng._check(lib.copra_b200_lmpc_feedback_gain(h, N, KuN.data_ptr(), KxN.data_ptr(), capi.DEVICE))

        def jvp1():
            eng._check(lib.copra_b200_lmpc_jvp(h, C.byref(t), capi.DEVICE, du.data_ptr(), dx.data_ptr()))

        def vjp_nu():
            for e in units:
                eng._check(lib.copra_b200_lmpc_vjp(h, C.c_void_p(e.data_ptr()), None, capi.DEVICE, C.byref(vo)))

        torch.cuda.synchronize()
        times = {}
        for key, call in (("forward", forward), ("gain1", gain1), ("gainN", gain_n), ("jvp1", jvp1), ("vjp_nu", vjp_nu)):
            ts = []
            for k in range(a.warmup + a.steps):
                flush.fill_(k & 0xFF)
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
        fwd = float(np.mean(times["forward"]))
        line = dict(name=name, batch=B, n=s["nvar"], nx=nx, nu=nu, solver=eng.last_solver(), solved_ok=int(ok.sum()),
                    nact_mean=float(na[ok].mean()), nact_max=int(na[ok].max()))
        for key, ts in times.items():
            line[key + "_ms"] = float(np.mean(ts))
            line[key + "_ms_all"] = ts
            if key != "forward":
                line[key + "_over_forward"] = float(np.mean(ts)) / fwd
        line["gain1_over_vjp_nu"] = line["gain1_ms"] / line["vjp_nu_ms"]
        print(json.dumps({k: v for k, v in line.items() if not k.endswith("_all")}), flush=True)
        results["lines"].append(line)
    print("gpu:", results["gpu"])
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_jvp.json"), "w") as fh:
        json.dump(results, fh, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
