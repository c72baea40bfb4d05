"""Compare two `bench.py --dump-outputs` directories (a reference build and a candidate) on the same workload.

    python tools/compare_dumps.py OLD_DIR NEW_DIR [--config c3] [--batch 16384]

Reports whether `status` is identical, the largest `control` and `trajectory` difference per instance scaled by
max(1, |old|) (tests/util.x_err), and how many sampled instances differ in `iters`, `nact` or the active set.  Reordered
floating-point sums can flip a near-tie, so every instance whose active set differs is re-solved by the CPU oracle and each
differing row must be weakly active there (tests/util.active_set_excused); the script exits non-zero otherwise, or when the
statuses differ or a scaled difference exceeds --tol.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from copra_b200 import workloads as wl  # noqa: E402
from tests.util import active_set, active_set_excused, x_err  # noqa: E402


def load(d):
    return {name: np.load(os.path.join(d, name + ".npy"))
            for name in ("instance", "control", "trajectory", "status", "iters", "nact", "iact")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--config", default="c3", choices=sorted(wl.CONFIGS))
    ap.add_argument("--batch", type=int, default=16384, help="instances of the benchmarked batch (bench.py's --batch)")
    ap.add_argument("--tol", type=float, default=1e-8)
    args = ap.parse_args()
    a, b = load(args.old), load(args.new)
    assert np.array_equal(a["instance"], b["instance"]), "the two dumps sample different instances"
    idx = a["instance"].astype(np.int64)
    rep = dict(instances=int(idx.size), status_identical=bool(np.array_equal(a["status"], b["status"])))
    for k in ("control", "trajectory"):
        errs = [x_err(b[k][j], a[k][j]) for j in range(idx.size)]
        j = int(np.argmax(errs))
        rep[k + "_max_scaled_diff"] = errs[j]
        rep[k + "_worst_instance"] = int(idx[j])
    rep["iters_differ"] = int((a["iters"].reshape(idx.size, -1) != b["iters"].reshape(idx.size, -1)).any(axis=1).sum())
    rep["nact_differ"] = int((a["nact"] != b["nact"]).sum())
    sets_a = [active_set(a["iact"][j], int(a["nact"][j])) for j in range(idx.size)]
    sets_b = [active_set(b["iact"][j], int(b["nact"][j])) for j in range(idx.size)]
    differ = [j for j in range(idx.size) if sets_a[j] != sets_b[j]]
    rep["active_set_differ"] = len(differ)
    ok = rep["status_identical"] and max(rep["control_max_scaled_diff"], rep["trajectory_max_scaled_diff"]) <= args.tol
    if differ:
        from oracle import pyoracle as po
        bp = wl.CONFIGS[args.config]() if args.config == "c1" else wl.CONFIGS[args.config](batch=args.batch, seed_offset=0)
        rep["excused_rows"] = {}
        for j in differ:
            o = po.lmpc(wl.instance(bp, int(idx[j])))
            try:
                rep["excused_rows"][int(idx[j])] = [active_set_excused(sets_a[j], o), active_set_excused(sets_b[j], o)]
            except AssertionError as e:
                rep.setdefault("not_excused", {})[int(idx[j])] = str(e)
                ok = False
    rep["ok"] = bool(ok)
    print(json.dumps(rep))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
