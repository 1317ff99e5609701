"""Cost of output times and checkpoint snapshots in the exponential solvers (vo_exp_set_t_list + vo_exp_enable_snapshots).

Each workload of tools/exp_small_bench.py ((a) 2^22 qubits CFM4, (b) 10^6 three-qubit chains magnus_42 with the applied commutator,
(c) 2^20 two-qubit systems adaptive CFM4), plus (d) 2^16 systems of n = 64 on the tensor-core tiles (CFM4, bench.py's shape), runs
from t = 0 to a horizon T to completion twice per repetition, alternating: with the default list [0, T], and with a 10-entry list
linspace(0, T, 10) and snapshots on. On the fixed-step workloads the entries fall on the step grid, so the difference is the
checkpoint events themselves (one call each, which the reference spends too), the [N][n] snapshot writes and, where the accumulated t
misses an entry by more than 2^-52, one clipped step of a few ulps (check_step's rule); on the adaptive one the entries also clip
steps. The report gives the accepted steps and Chkpt events of both modes. Times are CUDA events around `run`, after `reset`. Usage:
  python tools/exp_checkpoint_bench.py [--reps 3] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HORIZON = {"a": 9.0, "b": 4.5, "c": 1.8, "d": 2.7}  # every ninth of the horizon a multiple of the step (0.05; 0.1 for d)


def workload(vo, name):
    import exp_small_bench as esb
    if name != "d":
        return esb.workload(name)
    N = 1 << 16
    H0, H1 = vo.workloads.schrodinger_system(64)
    return dict(scheme="cfm4", basis=np.stack([-1j * H0, -1j * H1]), gp=vo.workloads.schrodinger_drive(N), M_gen=2, h=0.1, adaptive=False,
                applied=False, N=N)


def measure(reps):
    import torch
    import vecode_b200 as vo
    import exp_small_bench as esb
    ctx = vo.Context(0, arith="strict")
    out = {}
    for name in ("a", "b", "c", "d"):
        w = workload(vo, name)
        T = HORIZON[name]
        solvers = {}
        for mode in ("default", "tlist10_snapshots"):
            s, sp = esb.make_solver(vo, ctx, w, tf=T)
            if mode != "default":
                s.set_t_list(np.linspace(0.0, T, 10)).enable_snapshots()
            s.run(adaptive=w["adaptive"])  # warm-up
            solvers[mode] = (s, sp)
        res = {m: {"times_s": [], "accepted_steps": None, "chkpt_events": None} for m in solvers}
        for _ in range(reps):
            for mode, (s, _) in solvers.items():
                s.reset()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                st = s.run(adaptive=w["adaptive"])
                e1.record()
                torch.cuda.synchronize()
                assert st.kind == "Done"
                res[mode]["times_s"].append(e0.elapsed_time(e1) / 1e3)
                res[mode]["accepted_steps"], res[mode]["chkpt_events"] = st.counts["Step"], st.counts["Chkpt"]
        for m in res:
            res[m]["traj_steps_per_s"] = res[m]["accepted_steps"] / min(res[m]["times_s"])
        res["time_ratio_best"] = min(res["tlist10_snapshots"]["times_s"]) / min(res["default"]["times_s"])
        res.update(N=w["N"], n=int(w["basis"].shape[1]), scheme=w["scheme"] + (" applied commutator" if w["applied"] else "") + (" adaptive" if w["adaptive"] else ""),
                   horizon=T)
        out[name] = res
        del solvers
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also write the report as JSON to this file")
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = {"card": card, "workloads": measure(args.reps)}
    if args.out:
        json.dump(report, open(args.out, "w"), indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
