"""Cost of expectation values in the exponential solvers (vo_exp_set_observables) against the list alone and against snapshots.

The four workloads of tools/exp_checkpoint_bench.py ((a) 2^22 qubits CFM4, (b) 10^6 three-qubit chains magnus_42 with the applied
commutator, (c) 2^20 two-qubit systems adaptive CFM4, (d) 2^16 systems of n = 64 CFM4 on the tensor-core tiles) run with a 100-entry
list linspace(0, T, 100), T = 99 h, so that on the fixed-step workloads every entry falls on the step grid. Three modes alternate in
every repetition: the list alone, the list with snapshots, and the list with K = 3 observables (a diagonal, a random Hermitian and a
random non-Hermitian n x n operator). The report gives, per mode, the time of a whole solve (CUDA events around `run`, after `reset`),
the bytes of output the mode keeps on the device (from the shapes: len N n complex for snapshots, len N K complex for observables)
and the time relative to the list alone. The card's name, power limit and maximum SM clock are read in the same call. Usage:
  python tools/exp_observables_bench.py [--reps 3] [--out FILE.json]
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

ENTRIES, K = 100, 3
MODES = ("tlist100", "tlist100_snapshots", "tlist100_obs3")


def operators(n):
    rng = np.random.default_rng(11)
    G = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    return np.stack([np.diag(np.arange(n, dtype=float)).astype(complex), (G + G.conj().T) / 2.0,
                     rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))])


def output_bytes(mode, N, n):
    per = {"tlist100": 0, "tlist100_snapshots": n, "tlist100_obs3": K}[mode]
    return 16 * ENTRIES * N * per


def measure(reps):
    import torch
    import vecode_b200 as vo
    import exp_checkpoint_bench as ecb
    import exp_small_bench as esb
    ctx = vo.Context(0, arith="strict")
    out = {}
    for name in ("a", "b", "c", "d"):
        w = ecb.workload(vo, name)
        T = 99 * w["h"]
        n = int(w["basis"].shape[1])
        solvers = {}
        for mode in MODES:
            s, sp = esb.make_solver(vo, ctx, w, tf=T)
            s.set_t_list(np.linspace(0.0, T, ENTRIES))
            if mode == "tlist100_snapshots":
                s.enable_snapshots()
            elif mode == "tlist100_obs3":
                s.set_observables(operators(n))
            s.run(adaptive=w["adaptive"])  # warm-up
            solvers[mode] = (s, sp)
        res = {m: {"times_s": [], "accepted_steps": None, "chkpt_events": None, "output_bytes": output_bytes(m, w["N"], n)} for m in MODES}
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
        base = min(res["tlist100"]["times_s"])
        for m in MODES:
            res[m]["time_ratio_best"] = min(res[m]["times_s"]) / base
            res[m]["spread"] = (max(res[m]["times_s"]) - min(res[m]["times_s"])) / min(res[m]["times_s"])
        res.update(N=w["N"], n=n, scheme=w["scheme"] + (" applied commutator" if w["applied"] else "") + (" adaptive" if w["adaptive"] else ""),
                   horizon=T, entries=ENTRIES, K=K)
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
