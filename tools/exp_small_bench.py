"""Throughput of the exponential integrators for systems of 1 to 8 levels (exp_small_kernel, one system per thread).

  (a) 2^22 driven qubits, M = 3 (sigma_z detuning spread, cosine sigma_x drive), CFM4, fixed step
  (b) 10^6 three-qubit transverse-field Ising chains (n = 8), magnus_42 with the applied commutator, fixed step
  (c) 2^20 two-qubit systems (n = 4), adaptive CFM4

Every state array is larger than the 126 MB L2. Rates are trajectory-steps/s from CUDA events around `run`; FLOPs per step are
algorithmic (each system's own Taylor plan, as bench.py's exp_algorithmic_terms counts them, times 8 n^2 per application of an
n x n operator); bytes per step are the state, control values and generator parameters one event reads and writes. The
event-fusion comparison re-runs the timings with a build whose vo_exp_run launches one event at a time
(tools/build_variant.sh fuse1 "-DVO_EXP_SMALL_FUSE=1" exp exp_small). Usage: python tools/exp_small_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SX = np.array([[0, 1], [1, 0]], complex)
SZ = np.array([[1, 0], [0, -1]], complex)


def _kron(*ms):
    out = np.eye(1)
    for m in ms:
        out = np.kron(out, m)
    return out


def workload(name, N=None):
    rng = np.random.default_rng(1)
    if name == "a":
        N = N or (1 << 22)
        basis = np.stack([-0.5j * SZ, -0.5j * SZ, -0.5j * SX])
        gp = np.zeros((N, 2, 3))
        gp[:, 0, 0] = rng.uniform(-0.3, 0.3, N)                      # detuning spread (omega = 0: constant)
        gp[:, 1, 0], gp[:, 1, 1] = rng.uniform(0.5, 1.0, N), 1.0 + rng.uniform(-0.1, 0.1, N)
        return dict(scheme="cfm4", basis=basis, gp=gp, M_gen=3, h=0.05, adaptive=False, applied=False, N=N)
    if name == "b":
        N = N or 1_000_000
        I2 = np.eye(2)
        zz = _kron(SZ, SZ, I2) + _kron(I2, SZ, SZ)
        xs = _kron(SX, I2, I2) + _kron(I2, SX, I2) + _kron(I2, I2, SX)
        basis = np.stack([1j * zz, 1j * xs])                          # H = -J sum ZZ - h_x(t) sum X, J = 1
        gp = np.stack([rng.uniform(0.5, 1.5, N), rng.uniform(0.5, 2.0, N), rng.uniform(0, np.pi, N)], axis=1)[:, None, :]
        return dict(scheme="magnus42", basis=basis, gp=gp, M_gen=2, h=0.05, adaptive=False, applied=True, N=N)
    if name == "c":
        N = N or (1 << 20)
        G = [rng.standard_normal((4, 4)) + 1j * rng.standard_normal((4, 4)) for _ in range(2)]
        basis = np.stack([-0.5j * (g + g.conj().T) for g in G])
        gp = np.stack([rng.uniform(0.2, 1.0, N), rng.uniform(0.5, 3.0, N), rng.uniform(0, np.pi, N)], axis=1)[:, None, :]
        return dict(scheme="cfm4", basis=basis, gp=gp, M_gen=2, h=0.05, adaptive=True, applied=False, N=N)
    raise KeyError(name)


def make_solver(vo, ctx, w, tf=1.0e9):
    N, n = w["N"], w["basis"].shape[1]
    psi0 = np.zeros((N, n), complex)
    psi0[:, 0] = 1.0
    sp = vo.DenseBasisSplit(ctx, w["basis"])
    if w["scheme"] == "cfm4":
        s = vo.ExpCFMSolver(sp, w["gp"], 0.0, tf, psi0, w["h"], M_gen=w["M_gen"])
    else:
        s = vo.MagnusExpLinearSolver(sp, w["gp"], 0.0, tf, psi0, w["h"], M_gen=w["M_gen"], applied_commutator=w["applied"])
    return (s.with_tolerance(1e-8, 1e-8) if w["adaptive"] else s.no_adaptive()), sp


def terms_per_step(w, n_sys=512, n_times=48, t_max=20.0):
    """Taylor terms per trajectory-step of ONE system (its own theta), averaged over systems and step times (bench.exp_algorithmic_terms)."""
    import bench
    basis, gp, h = w["basis"], w["gp"], w["h"]
    if w["scheme"] == "magnus42":
        return bench.exp_algorithmic_terms("magnus_applied", basis, gp, h, n_sys, n_times, t_max)[0]
    terms = bench.exp_algorithmic_terms("cfm4", basis, gp, h, n_sys, n_times, t_max)[0]
    if w["adaptive"]:  # + the embedded exponential, row CFM_R2_J1_GL = (1/2, 1/2) on the same nodes
        rng = np.random.default_rng(5)
        idx = np.linspace(0, gp.shape[0] - 1, n_sys).astype(np.int64)
        t = rng.uniform(0.0, t_max, n_times)[None, :]
        norm1 = np.array([np.abs(b).sum(axis=0).max() for b in basis])
        M = basis.shape[0]

        def gen(tt):
            out = np.ones((len(idx), tt.shape[1], M))
            for m in range(1, M):
                out[..., m] = gp[idx, m - 1, 0, None] * np.cos(gp[idx, m - 1, 1, None] * tt + gp[idx, m - 1, 2, None])
            return out
        k = 0.5 * (gen(t + 0.21132486540518711775 * h) + gen(t + 0.78867513459481288225 * h)) * h
        terms += bench._plan_terms((np.abs(k) * norm1).sum(axis=-1)).mean()
    return float(terms)


def measure(names, calls):
    """Rates of the listed workloads with the library this process loaded (VECODE_B200_SO selects a variant)."""
    import torch
    import vecode_b200 as vo
    ctx = vo.Context(0, arith="strict")
    out = {}
    for name in names:
        w = workload(name)
        s, sp = make_solver(vo, ctx, w)
        s.run(adaptive=w["adaptive"], max_calls=calls)  # warm-up (and past the checkpoint at t0)
        times, steps = [], []
        for _ in range(3):
            acc0 = int(s.stats()["accepted"].sum())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st = s.run(adaptive=w["adaptive"], max_calls=calls)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
            steps.append(int(s.stats()["accepted"].sum()) - acc0)
            assert st.kind != "Err"
        out[name] = {"times_s": times, "accepted_steps": steps, "launches_per_run": st.counts["launches"]}
        del s, sp
    ctx.close()
    return out


def oracle_check(name, n_sys=1000, steps=10):
    import vecode_b200 as vo
    from oracle import oracle_lib
    w = workload(name, N=n_sys)
    ctx = vo.Context(0, arith="strict")
    s, _ = make_solver(vo, ctx, w, tf=steps * w["h"])
    s.run(adaptive=w["adaptive"])
    got = s.current()[1]
    psi0 = np.zeros_like(got)
    psi0[:, 0] = 1.0
    if w["applied"]:  # no structure tensor on this basis: magnus_42 restated with dense matrices and scipy expm
        from scipy.linalg import expm
        B, gp, h, c_mid = w["basis"], w["gp"], w["h"], 0.288675134594812882254574390251
        err = 0.0
        for i in range(n_sys):
            L = lambda t: B[0] + gp[i, 0, 0] * np.cos(gp[i, 0, 1] * t + gp[i, 0, 2]) * B[1]
            x, t = psi0[i].copy(), 0.0
            for _ in range(steps):
                l0, l1 = L(t + h / 2 - c_mid * h), L(t + h / 2 + c_mid * h)
                x, t = expm((l0 + l1) * (h / 2) + (l0 @ l1 - l1 @ l0) * (h * h * -0.144337567297406441127287195125)) @ x, t + h
            err = max(err, float(np.abs(got[i] - x).max()))
        ctx.close()
        return err
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-8) if w["adaptive"] else dict(no_adaptive=True)
    ref = oracle_lib.exp_ensemble(w["scheme"], w["basis"], w["gp"], psi0, 0.0, steps * w["h"], w["h"], M_gen=w["M_gen"], n_threads=16, **kw)
    ctx.close()
    return float(np.abs(got - ref["psi"]).max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the report as JSON to this file")
    ap.add_argument("--calls", type=int, default=64)
    ap.add_argument("--measure-only", default="")
    args = ap.parse_args()
    names = ["a", "b", "c"]
    if args.measure_only:
        print(json.dumps(measure(args.measure_only.split(","), args.calls)))
        return
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    peaks = json.load(open(os.path.join(ROOT, "profiles", "fp64_peaks.json")))
    variant = os.path.join(ROOT, "vec-ode_b200", "variants", "libvecode_b200_fuse1.so")

    def sub(env_so):
        env = dict(os.environ)
        if env_so:
            env["VECODE_B200_SO"] = env_so
        r = subprocess.run([sys.executable, __file__, "--measure-only", ",".join(names), "--calls", str(args.calls)], env=env, capture_output=True, text=True)
        if r.returncode:
            raise RuntimeError(r.stderr[-4000:])
        return json.loads(r.stdout.strip().splitlines()[-1])

    fused, single = sub(None), sub(variant) if os.path.exists(variant) else None
    fused2 = sub(None)  # repeat of the fused build: the run-to-run spread
    report = {"card": card, "fp64_peaks": {k: peaks[k] for k in ("dfma_tflops", "sm_mhz")}, "calls_per_run": args.calls, "workloads": {}}
    for name in names:
        w = workload(name)
        n = w["basis"].shape[1]
        terms = terms_per_step(w)
        ops = 5 if (w["applied"] and n > 4) else 1          # applications of an n x n operator per Taylor term
        flop = terms * ops * 8.0 * n * n
        M_gen = w["M_gen"]
        bytes_event = 2 * 16 * n + 2 * (4 * 8 + 3 * 4) + 8 * 3 * (M_gen - 1)
        r = {"N": w["N"], "n": n, "M": int(w["basis"].shape[0]), "scheme": w["scheme"] + (" applied commutator" if w["applied"] else "") + (" adaptive" if w["adaptive"] else ""),
             "taylor_terms_per_step": terms, "algorithmic_flop_per_step": flop, "bytes_per_step_one_event_per_launch": bytes_event}
        for label, res in (("fused", fused), ("fused_repeat", fused2), ("one_event_per_launch", single)):
            if res is None:
                continue
            m = res[name]
            rate = max(np.array(m["accepted_steps"]) / np.array(m["times_s"]))
            r[label] = {"traj_steps_per_s": rate, "launches_per_run": m["launches_per_run"], "times_s": m["times_s"],
                        "fp64_share_of_measured_dfma_peak": rate * flop / (peaks["dfma_tflops"] * 1e12),
                        "hbm_share_of_7.7TBps_at_one_event_per_launch": rate * bytes_event / 7.7e12}
        try:
            r["max_abs_err_vs_oracle_1000_systems"] = oracle_check(name)
        except Exception as e:
            r["max_abs_err_vs_oracle_1000_systems"] = f"not checked: {type(e).__name__}: {e}"
        report["workloads"][name] = r
    if args.out:
        json.dump(report, open(args.out, "w"), indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
