"""Per-step references and limits on the B200: what a moving ZMP box and velocity reference cost.

One GPU, device-resident inputs, CUDA events on the launching stream, L2 overwritten between timed steps (as bench.py):
  c3            C3 with step-size entries (the comparison line)
  c3_walk       C3 walking (workloads.c3_walk): per-step f and p, full build + solve per step
  retarget      the next tick of the walk (new x0, every window moved by one tick) through copra_b200_lmpc_retarget, cold
  retarget_warm the same with copra_b200_set_warm_start(1), seeded with the active sets of the previous tick (mean iterations
                after the seed reported)
  dense/per_step at --dense-batch: the same walk as copra's autoSpan'd full-size entries against the per-step form
With --compare DIR (another checkout of the project, its library built) it also runs `bench.py --gpus 1` there and here,
alternating, and reports both C3 lines.  Prints the card's name and power limit; writes JSON to --out.

    python tools/bench_walk.py --out DIR [--compare OTHER_CHECKOUT]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from copra_b200 import capi, workloads as wl  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(torch, stream, flush, steps, call, after=None):
    """`steps` calls, each between CUDA events on the stream with the L2 overwritten before it; ms per call"""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for k in range(steps):
        flush.fill_(k & 0xFF)
        ev0.record(stream)
        call()
        ev1.record(stream)
        torch.cuda.synchronize()
        times.append(ev0.elapsed_time(ev1))
        if after:
            after()
    return times


def line(name, batch, times, eng, status, iters, **extra):
    ms = float(np.mean(times))
    out = dict(name=name, batch=batch, ms_per_step=ms, p50_ms=float(np.median(times)), solves_per_s=batch / (ms * 1e-3),
               solver=eng.last_solver(), hessian_shared=eng.hessian_is_shared(), solved_ok=int((status == 0).sum()),
               mean_outer_iterations=float(iters[:, 0].mean()), stage_ms=eng.timing())
    out.update(extra)
    print(json.dumps({k: v for k, v in out.items() if k != "stage_ms"}), flush=True)
    return out


def run_lines(torch, args, dev, stream, flush):
    res = {}
    for name, bp in (("c3", wl.c3(args.batch)), ("c3_walk", wl.c3_walk(args.batch))):
        r = bench.Runner(torch, capi, dev, 0, bp, stream)
        for _ in range(args.warmup):
            r.step_device()
        t = timed(torch, stream, flush, args.steps, r.step_device)
        res[name] = line(name, bp["batch"], t, r.eng, r.d_status.cpu().numpy(), r.d_iters.view(-1, 2).cpu().numpy())
        if name == "c3_walk":
            # the next tick: every window of the plan moved by one tick, x0 halfway to the solved next state (a state exactly
            # on a face of the ZMP box would leave the step-0 rows, which no control reaches, infeasible by rounding)
            nxt = wl.c3_walk(args.batch, tick=1)
            nxt["x0"] = 0.5 * (bp["x0"] + r.d_traj.view(bp["batch"], -1)[:, 6:12].cpu().numpy())
            hb = capi.HostBatch(nxt, device_tensors=dev)
            hb.problem.flags |= capi.FLAG_STABLE_BOUND_PATTERN

            def retarget():
                rc = r.lib.copra_b200_lmpc_retarget(r.eng.h, C.byref(hb.problem), C.byref(r.rd))
                if rc:
                    r.eng._check(rc)
            r.step_device()
            retarget()
            t = timed(torch, stream, flush, args.steps, retarget)
            res["retarget"] = line("retarget", bp["batch"], t, r.eng, r.d_status.cpu().numpy(), r.d_iters.view(-1, 2).cpu().numpy(),
                                   ratio_to_full_step=float(np.mean(t)) / res["c3_walk"]["ms_per_step"])
            cold_iters = r.d_iters.view(-1, 2).cpu().numpy()
            r.eng.set_warm_start(True)
            r.step_device()  # the seed: the active sets at the previous tick
            its = []
            t = timed(torch, stream, flush, args.steps, retarget,
                      after=lambda: (its.append(r.d_iters.view(-1, 2).cpu().numpy()), r.step_device()))
            r.eng.set_warm_start(False)
            res["retarget_warm"] = line("retarget_warm", bp["batch"], t, r.eng, r.d_status.cpu().numpy(), its[0],
                                        ratio_to_full_step=float(np.mean(t)) / res["c3_walk"]["ms_per_step"],
                                        mean_iterations_after_seed=float(its[0][:, 0].mean()),
                                        mean_iterations_cold=float(cold_iters[:, 0].mean()))
        r.close()
    # the dense (autoSpan'd) form against the per-step one at a batch the dense form fits
    bp = wl.c3_walk(args.dense_batch)
    for name, prob in (("per_step", bp), ("dense", wl.spanned(bp))):
        eng = capi.Engine(0, stream=stream.cuda_stream)
        hb = capi.HostBatch(prob, device_tensors=dev)
        sz = eng.sizes(hb)
        B = prob["batch"]
        status = torch.empty(B, dtype=torch.int32, device=dev)
        iters = torch.empty(2 * B, dtype=torch.int32, device=dev)
        control = torch.empty(B * sz["nU"], dtype=torch.float64, device=dev)
        rd = capi.Results()
        rd.memory = capi.DEVICE
        rd.status, rd.iters, rd.control = status.data_ptr(), iters.data_ptr(), control.data_ptr()

        def run():
            rc = eng.lib.copra_b200_lmpc_run(eng.h, C.byref(hb.problem), C.byref(rd))
            if rc:
                eng._check(rc)
        for _ in range(args.warmup):
            run()
        t = timed(torch, stream, flush, max(3, args.steps // 2), run)
        res["walk_%s_%d" % (name, B)] = line("walk_%s" % name, B, t, eng, status.cpu().numpy(), iters.view(-1, 2).cpu().numpy(),
                                             h2d_bytes=hb.h2d_bytes)
        res["walk_%s_%d" % (name, B)]["control_sample"] = control.view(B, -1)[:4].cpu().numpy().tolist()
        eng.close()
        del hb
        torch.cuda.empty_cache()
    a, b = (np.array(res["walk_%s_%d" % (k, args.dense_batch)].pop("control_sample")) for k in ("per_step", "dense"))
    res["walk_dense_vs_per_step"] = dict(speedup=res["walk_dense_%d" % args.dense_batch]["ms_per_step"] /
                                         res["walk_per_step_%d" % args.dense_batch]["ms_per_step"],
                                         max_control_diff_first4=float(np.abs(a - b).max()))
    print(json.dumps(res["walk_dense_vs_per_step"]), flush=True)
    return res


def bench_c3(tree, steps, warmup):
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline",
                        "--no-extras"], cwd=tree, capture_output=True, text=True)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode or not lines:
        raise RuntimeError("bench.py in %s failed: %s" % (tree, r.stderr[-2000:]))
    d = json.loads(lines[-1])
    return dict(value=d.get("value"), ms_per_step=d.get("ms_per_step"), unit=d.get("unit"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=16384)
    ap.add_argument("--dense-batch", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--compare", help="another checkout of the project (library built): bench.py there and here, alternating")
    ap.add_argument("--rounds", type=int, default=2)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch
    card = gpu_info()
    print("card (name, power limit):", card, flush=True)
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    out = dict(card=card, l2="overwritten between timed steps (256 MiB fill)", steps=args.steps, warmup=args.warmup)
    with torch.cuda.stream(stream):
        out["lines"] = run_lines(torch, args, dev, stream, flush)
    del flush
    torch.cuda.empty_cache()
    if args.compare:
        runs = []
        for k in range(args.rounds):
            for name, tree in (("other", os.path.abspath(args.compare)), ("this", ROOT)):
                t0 = time.time()
                runs.append(dict(tree=name, round=k, **bench_c3(tree, args.steps, args.warmup), wall_s=time.time() - t0))
                print(json.dumps(runs[-1]), flush=True)
        out["bench_c3_alternating"] = runs
    with open(os.path.join(args.out, "bench_walk.json"), "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
