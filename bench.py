#!/usr/bin/env python
"""bench.py — ensemble trajectory-steps/s of the time-stepping hot path on N B200s (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload vdp_dopri5|lorenz_rk4|heat_rk4|heat_rk4_fused|heat_rk4_dd|schrodinger_cfm4|
                   schrodinger_magnus_applied|schrodinger_magnus_dense]
                  [--arith strict|fast]
The default workload is config 3 (adaptive DoPri5, 10^6 Van der Pol oscillators), the configuration the north-star target is
quoted on; at N = 1 the other configs are measured in the same run and reported under `also`, each with its own roofline.
  python bench.py --impl reference ...      # the CPU restatement of the reference path on the host cores
  python bench.py --dump-outputs DIR ...    # also write what the last timed step computed, DIR/<name>.npy: the same arguments give the
                                            # same inputs on every run, so two builds can be compared output for output

A "step" is ONE pass of the hot path over ONE batch: one kernel launch that advances every trajectory of a
10^6-trajectory ensemble by one RK step (lorenz_rk4) / one adaptive attempt (vdp_dopri5), or one RK4 step of the
2^26-point heat state (heat_rk4, 4 stage launches). The device-resident number (`value`) rotates over enough independent
batches that the working set exceeds the 126 MB L2, so every launch streams its state from HBM. `e2e` is the same metric
through the public API with HOST buffers: per e2e step one whole solve of the named config (upload from pinned memory,
integrate, download) — see DESIGN.md §Measurement.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TRAJ = 1_000_000
GROUP_SIMILAR = os.environ.get("VECODE_BENCH_GROUP", "1") != "0"  # schrodinger_cfm4: tiles of systems with similar drive amplitude
DYN_GROUP = os.environ.get("VECODE_BENCH_DYNGROUP", "1") != "0"  # ... re-sorted by the norm bound of the coming step before every event (vo_exp_set_dynamic_grouping)
DD_K = int(os.environ.get("VECODE_BENCH_DD_K", "4"))  # heat_rk4_dd: RK steps between ghost refreshes (ghost zone = 4 * DD_K points per side)
E2E_PARTS = int(os.environ.get("VECODE_BENCH_E2E_PARTS", "4"))  # chunks of the e2e solve (vec-ode_b200/pipeline.py); 1 = one solver
L2_MB = 126


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        v = json.load(open(p)).get(workload)
        return float(v) if isinstance(v, (int, float)) else None
    return None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for (ts, r) in self.rows if t0 - 0.05 <= ts <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------------------------
def solver_outputs(s, x):
    """What a caller reads back after a solver's last step: the state `x` and, per trajectory, its time and next step size."""
    st = s.stats()
    return {"x": x, "t": st["t"], "h": st["h"]}


class Batches:
    """Independent batches of one ensemble (`solvers`, all started from `x0`), one launch each in turn (vo.step_many)."""
    adaptive = False

    def restart(self):
        """Every batch back to its initial state, then its first call (the Chkpt event at t0, no launch), as after construction."""
        for s in self.solvers:
            s.reset(self.x0)
        self.vo.step_many(self.solvers, self.adaptive, 1)

    def run_steps(self, k):
        nb = len(self.solvers)
        if k >= nb:
            self.vo.step_many(self.solvers, self.adaptive, k // nb)
        if k % nb:
            self.vo.step_many(self.solvers[: k % nb], self.adaptive, 1)
        if k:
            self.last = self.solvers[(k % nb or nb) - 1]

    def outputs(self):
        """The batch the last step advanced."""
        return solver_outputs(self.last, self.last.current()[1].to_host())


class LorenzRK4(Batches):
    name = "lorenz_rk4"
    label = "config 2: fixed-step RK4, 10^6 Lorenz-63 trajectories per batch, f64, h=1e-3"
    bytes_per_unit = 48.0  # SURVEY.md §8(d): read state + write state, 2*d*8
    unit_name = "trajectory-step"
    state_mb = 24
    steps_per_solve = 1001  # t in [0,1], h = 1e-3: 1000 steps + the remainder step (SURVEY.md §3.1)

    def __init__(self, vo, ctx, rank, world, n_batches):
        self.vo, self.ctx = vo, ctx
        self.tableau = vo.ButcherTableu.builtin("RK4")
        self.rhs = vo.Rhs(ctx, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
        first = rank * N_TRAJ
        self.x0_host = vo.workloads.lorenz_x0(N_TRAJ, first=first)
        self.x0 = vo.Ensemble.from_host(ctx, self.x0_host)
        self.solvers = [vo.RK45Solver(self.rhs, 0.0, 1.0e9, self.x0, 1e-3, tableau=self.tableau) for _ in range(n_batches)]
        vo.step_many(self.solvers, False, 1)  # the first call of every solver is the Chkpt event at t0 (no launch)

    def units(self, k):
        return float(k) * N_TRAJ

    def e2e_setup(self, group=None):
        import torch
        vo = self.vo
        self.pin_in = torch.from_numpy(self.x0_host.copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        tab = self.tableau

        def make(ctx, lo, hi, x0):
            return vo.RK45Solver(vo.Rhs(ctx, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS)), 0.0, 1.0, x0, 1e-3, tableau=tab)
        # the ensemble in E2E_PARTS chunks, each on its own stream and host thread: copies overlap the integration
        self.e_sharded = None
        if group is not None and group.world > 1:  # N > 1: one ensemble of world x 10^6 trajectories, gathered to rank 0 chunk by chunk
            self.n_total = N_TRAJ * group.world
            self.pin_full = torch.empty((self.n_total, 3), dtype=torch.float64).pin_memory() if group.ranks[0] == 0 else None
            self.e_sharded = vo.pipeline.ShardedChunkedSolve(group, self.n_total, 3, make, parts=E2E_PARTS, arith=self.ctx.arith)
        else:
            self.e_chunked = vo.pipeline.ChunkedSolve(self.ctx.device, self.ctx.arith, N_TRAJ, 3, make, parts=E2E_PARTS)

    def e2e_step(self):
        if self.e_sharded is not None:  # H2D of this rank's shard, whole solve, NCCL gather + ONE D2H of the whole ensemble on rank 0
            sts = self.e_sharded.solve(self.pin_in.numpy(), None if self.pin_full is None else self.pin_full.numpy())
            return float(sum(st.counts["Step"] for st in sts)), self.pin_in.numel() * 8, 0 if self.pin_full is None else self.pin_full.numel() * 8
        sts = self.e_chunked.solve(self.pin_in.numpy(), self.pin_out.numpy())  # H2D from pinned memory, whole solve, D2H of the result
        return float(sum(st.counts["Step"] for st in sts)), self.pin_in.numel() * 8, self.pin_out.numel() * 8


class VdpDopri5(Batches):
    name = "vdp_dopri5"
    label = "config 3: adaptive DoPri5, 10^6 Van der Pol oscillators per batch (mu sweep 0.5..20), rtol 1e-6, per-trajectory control"
    bytes_per_unit = 80.0  # SURVEY.md §8(d): state in/out + t,h,prev_h in/out
    unit_name = "attempted trajectory-step"
    state_mb = 60
    adaptive = True

    def __init__(self, vo, ctx, rank, world, n_batches):
        self.vo, self.ctx = vo, ctx
        self.tableau = vo.ButcherTableu.builtin("DOPRI5")
        n_total = N_TRAJ * world
        self.mu = vo.workloads.vdp_mu(n_total, N_TRAJ, rank * N_TRAJ)
        self.rhs = vo.Rhs(ctx, "VDP", 2, [self.mu])
        self.x0_host = vo.workloads.vdp_x0(N_TRAJ)
        self.x0 = vo.Ensemble.from_host(ctx, self.x0_host)
        self.solvers = [vo.RK45Solver(self.rhs, 0.0, 1.0e9, self.x0, 1e-3, tableau=self.tableau).with_tolerance(1e-6, 1e-6)
                        for _ in range(n_batches)]
        if os.environ.get("VECODE_BENCH_NO_DX_NORM"):  # experiment switch: drop the per-attempt ODEAdaptiveData.dx_norm record (8 B)
            for s_ in self.solvers:
                s_.set_record_dx_norm(False)
        if os.environ.get("VECODE_BENCH_NO_BLOCKED"):  # experiment switch: keep the sweep on the public layout (rk_ctl2w_staged_kernel)
            for s_ in self.solvers:
                s_.set_blocked(False)
        if os.environ.get("VECODE_BENCH_MIXED"):  # experiment switch: store prev_h on every attempt (vo_solver_set_mixed_stepping)
            for s_ in self.solvers:
                s_.set_mixed_stepping(True)
        vo.step_many(self.solvers, True, 1)
        self._attempts0 = None

    def attempts(self):
        tot = 0
        for s in self.solvers:
            st = s.stats()
            tot += int(st["accepted"].sum()) + int(st["rejected"].sum())
        return tot

    def units(self, k):
        return float(k) * N_TRAJ  # every lane is live (tf = 1e9): one attempt per trajectory per sweep

    def e2e_setup(self, group=None):
        import torch
        vo = self.vo
        self.pin_in = torch.from_numpy(self.x0_host.copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        tab, mu = self.tableau, self.mu

        def make(ctx, lo, hi, x0):
            return vo.RK45Solver(vo.Rhs(ctx, "VDP", 2, [mu[lo:hi].copy()]), 0.0, 20.0, x0, 1e-3, tableau=tab).with_tolerance(1e-6, 1e-6)
        self.e_sharded = None
        if group is not None and group.world > 1:
            # N > 1: ONE ensemble of world x 10^6 oscillators (mu swept over the whole of it), sharded round-robin so that every
            # rank sees the whole mu range (the cost of a trajectory grows with mu), gathered to rank 0 chunk by chunk
            G, r = group.world, group.ranks[0]
            self.n_total = N_TRAJ * G
            mu_il = vo.workloads.vdp_mu(self.n_total)[r::G].copy()

            def make_il(ctx, lo, hi, x0):
                return vo.RK45Solver(vo.Rhs(ctx, "VDP", 2, [mu_il[lo:hi].copy()]), 0.0, 20.0, x0, 1e-3, tableau=tab).with_tolerance(1e-6, 1e-6)
            self.pin_full = torch.empty((self.n_total, 2), dtype=torch.float64).pin_memory() if r == 0 else None
            self.e_sharded = vo.pipeline.ShardedChunkedSolve(group, self.n_total, 2, make_il, parts=E2E_PARTS, arith=self.ctx.arith, interleave=True)
        else:
            self.e_chunked = vo.pipeline.ChunkedSolve(self.ctx.device, self.ctx.arith, N_TRAJ, 2, make, parts=E2E_PARTS)

    def e2e_step(self):
        if self.e_sharded is not None:
            sts = self.e_sharded.solve(self.pin_in.numpy(), None if self.pin_full is None else self.pin_full.numpy(), adaptive=True)
            return (float(sum(st.counts["Step"] + st.counts["Reject"] for st in sts)), self.pin_in.numel() * 8,
                    0 if self.pin_full is None else self.pin_full.numel() * 8)
        sts = self.e_chunked.solve(self.pin_in.numpy(), self.pin_out.numpy(), adaptive=True)
        return float(sum(st.counts["Step"] + st.counts["Reject"] for st in sts)), self.pin_in.numel() * 8, self.pin_out.numel() * 8


class HeatRK4:
    name = "heat_rk4"
    label = "config 4: RK4 on the semi-discretised 1-D heat equation, one state of 2^26 points, stage path"
    bytes_per_unit = 104.0  # SURVEY.md §8(d): 13 vector passes x 8 B per grid-point-step
    unit_name = "grid-point-step"
    state_mb = 512
    D = 1 << 26

    def __init__(self, vo, ctx, rank, world, n_batches):
        self.vo, self.ctx = vo, ctx
        self.tableau = vo.ButcherTableu.builtin("RK4")
        self.rhs = vo.Rhs(ctx, "HEAT1D", self.D, [1.0])
        self.x0_host = vo.workloads.heat_u0(self.D)[None, :]
        self.x0 = vo.Ensemble.from_host(ctx, self.x0_host)
        self.solvers = [vo.RK45Solver(self.rhs, 0.0, 1.0e9, self.x0, 0.25, tableau=self.tableau)]
        self.solvers[0].step()

    def restart(self):
        self.solvers[0].reset(self.x0)
        self.solvers[0].step()

    def run_steps(self, k):
        self.vo.step_many(self.solvers, False, k)

    def outputs(self):
        return solver_outputs(self.solvers[0], self.solvers[0].current()[1].to_host()[0])

    def units(self, k):
        return float(k) * self.D

    def e2e_setup(self, group=None):
        import torch
        self.pin_in = torch.from_numpy(self.x0_host.copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        self.e_x0 = self.vo.Ensemble(self.ctx, self.D, 1)
        self.e_solver = self.vo.RK45Solver(self.rhs, 0.0, 25.0, self.e_x0, 0.25, tableau=self.tableau)

    def e2e_step(self):
        self.e_x0.upload(self.pin_in.numpy(), "soa")
        self.e_solver.reset(self.e_x0)
        st = self.e_solver.run()
        self.e_solver.current()[1].to_host("soa", out=self.pin_out.numpy())
        return float(st.counts["Step"]) * self.D, self.pin_in.numel() * 8, self.pin_out.numel() * 8


class HeatRK4Fused(HeatRK4):
    """Config 4 through the whole-step kernel (rk_heat_fused.cuh): every stage of an RK4 step inside one kernel, the state read
    once and written once. Not the stage path BASELINE.json names for config 4 — reported beside it."""
    name = "heat_rk4_fused"
    label = "config 4, whole-step kernel: RK4 on the 1-D heat equation, one state of 2^26 points, all four stages in one launch"
    bytes_per_unit = 16.0  # read x, write next_x

    def __init__(self, vo, ctx, rank, world, n_batches):
        super().__init__(vo, ctx, rank, world, n_batches)
        self.solvers[0].set_fused_step()

    def e2e_setup(self, group=None):
        super().e2e_setup(group)
        self.e_solver.set_fused_step()


class HeatRK4DD:
    """Row N4 (SURVEY.md §8f): config 4's single state of 2^26 points split into one slab per GPU with ghost zones
    (vec-ode_b200/domain.py). STRONG scaling: the whole job is always 2^26 points."""
    name = "heat_rk4_dd"
    label = ("config 4 domain-decomposed: RK4 on the 1-D heat equation, ONE state of 2^26 points split into one slab per GPU, "
             f"ghost zones of {4 * DD_K} points refreshed every {DD_K} steps (one all-gather of {8 * DD_K} doubles per rank)")
    bytes_per_unit = 104.0
    unit_name = "grid-point-step"
    state_mb = 512
    D = 1 << 26

    def __init__(self, vo, ctx, rank, world, n_batches):
        self.vo, self.ctx = vo, ctx
        self.ds = vo.domain.HeatSlabSolver(ctx, self.D, lambda j: vo.workloads.heat_u0_at(j, self.D), 1.0, 0.0, 1.0e9, 0.25, steps_per_exchange=DD_K)
        self.ds.step()  # Chkpt at t0
        self.solvers = []
        self.x0 = vo.Ensemble.from_host(ctx, vo.workloads.heat_u0_at(self.ds.slab.global_index(), self.D)[None, :])  # the slab, ghosts included

    def restart(self):
        self.ds.reset(self.x0)
        self.ds.step()

    def run_steps(self, k):
        for _ in range(k):
            self.ds.step()

    def outputs(self):
        return solver_outputs(self.ds.solver, self.ds.local_interior())

    def units(self, k):
        return float(k) * self.ds.slab.m  # owned points only: the ghost points are redundant work

    def e2e_setup(self, group=None):
        import torch
        slab = self.ds.slab
        self.pin_in = torch.from_numpy(self.vo.workloads.heat_u0_at(slab.global_index(), self.D)[None, :].copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        self.e_x0 = self.vo.Ensemble(self.ctx, slab.local_len, 1)
        self.e_ds = self.vo.domain.HeatSlabSolver(self.ctx, self.D, lambda j: self.vo.workloads.heat_u0_at(j, self.D), 1.0, 0.0, 25.0, 0.25,
                                                  steps_per_exchange=DD_K)

    def e2e_step(self):
        self.e_x0.upload(self.pin_in.numpy(), "soa")
        self.e_ds.reset(self.e_x0)
        st = self.e_ds.run()
        self.e_ds.solver.current()[1].to_host("soa", out=self.pin_out.numpy())
        n_steps = 100  # t in [0, 25], h = 0.25
        return float(n_steps) * self.e_ds.slab.m, self.pin_in.numel() * 8, self.pin_out.numel() * 8


# ---- algorithmic Taylor degrees of the exponential integrators, exactly as the kernels plan them ------------------------------------
def _plan_terms(theta):
    """sub-steps x degree of the scaled Taylor series at theta = ||L||_1 (exp_kernels.cuh: taylor_plan), vectorised"""
    theta = np.asarray(theta, dtype=np.float64)
    sq = np.where(theta > 1.0, np.ceil(theta), 1.0)
    x = theta / sq
    term, deg, done = np.ones_like(x), np.zeros_like(x), np.zeros(x.shape, dtype=bool)
    for k in range(1, 61):
        term = np.where(done, term, term * x / k)
        deg = np.where(done, deg, k)
        done |= term <= 1.1102230246251565e-16
    return sq * deg


def exp_algorithmic_terms(scheme, basis, gp, h, n_sys=512, n_times=48, t_max=20.0):
    """Mean number of Taylor terms per exponential-application that ONE system needs (its own theta, not its tile's), averaged over a
    sample of systems and of step times t in [0, t_max), with the generator evaluated like the kernels do — the `m*` of SURVEY.md §8(d).
    Returns (terms per trajectory-step summed over the exponentials of a step, largest theta)."""
    rng = np.random.default_rng(5)
    idx = np.linspace(0, gp.shape[0] - 1, n_sys).astype(np.int64)
    t = rng.uniform(0.0, t_max, n_times)[None, :]                     # [1][T]
    g = gp[idx]                                                       # [S][M-1][3]
    norm1 = np.array([np.abs(b).sum(axis=0).max() for b in basis])    # induced 1-norms, as vo_split_basis_create computes them
    M = basis.shape[0]

    def gen(tt):  # [S][T][M] real coefficients of L(t) = B_0 + sum_m g_m(t) B_m
        out = np.ones(g.shape[:1] + tt.shape[1:] + (M,))
        for m in range(1, M):
            out[..., m] = g[:, m - 1, 0, None] * np.cos(g[:, m - 1, 1, None] * tt + g[:, m - 1, 2, None])
        return out
    if scheme == "cfm4":  # cfm_general with the tables of dat/mod.rs:4, 67-74: two exponentials per step
        c = (0.21132486540518711775, 0.78867513459481288225)
        alpha = ((0.53867513459481288225, -0.038675134594812882255), (-0.038675134594812882255, 0.53867513459481288225))
        v = [gen(t + cq * h) for cq in c]
        terms, thmax = 0.0, 0.0
        for row in alpha:
            k = (row[0] * v[0] + row[1] * v[1]) * h
            th = (np.abs(k) * norm1).sum(axis=-1)
            terms, thmax = terms + _plan_terms(th).mean(), max(thmax, float(th.max()))
        return float(terms), thmax
    c_mid, b1, b2 = 0.288675134594812882254574390251, h * 0.5, h * h * 0.144337567297406441127287195125
    l0, l1 = gen(t + b1 - c_mid * h), gen(t + b1 + c_mid * h)
    if scheme == "magnus_applied":  # theta bound of exp_step_kernel: ||W1|| + 2 |b2| ||L0|| ||L1||
        th = (np.abs((l0 + l1) * b1) * norm1).sum(axis=-1) + 2.0 * b2 * (np.abs(l0) * norm1).sum(axis=-1) * (np.abs(l1) * norm1).sum(axis=-1)
        return float(_plan_terms(th).mean()), float(th.max())
    if scheme == "magnus_dense":    # magnus_dense_kernel takes ||Omega||_1 of the matrix itself: form it for a smaller sample
        ths = []
        for si in range(0, l0.shape[0], 8):
            for ti in range(0, l0.shape[1], 6):
                L0 = np.tensordot(l0[si, ti], basis, axes=1)
                L1 = np.tensordot(l1[si, ti], basis, axes=1)
                om = (L0 + L1) * b1 - b2 * (L0 @ L1 - L1 @ L0)
                ths.append(np.abs(om).sum(axis=0).max())
        ths = np.array(ths)
        return float(_plan_terms(ths).mean()), float(ths.max())
    raise KeyError(scheme)



class SchrodingerCFM4:
    name = "schrodinger_cfm4"
    label = ("config 5: commutator-free Magnus CFM4, 10^5 driven 64-level Schroedinger systems (complex f64) per GPU, h = 0.1, "
             "fixed step, shared basis {-iH0, -iH1}" + ("; device order grouped by drive amplitude (group_similar), host buffers in the caller's order" if GROUP_SIMILAR else ""))
    unit_name = "trajectory-step"
    bytes_per_unit = None  # compute-bound: the roofline is the FP64 tensor pipe
    state_mb = 102
    N_SYS = 100_000
    NDIM = 64

    def __init__(self, vo, ctx, rank, world, n_batches):
        self.vo, self.ctx = vo, ctx
        H0, H1 = vo.workloads.schrodinger_system(self.NDIM)
        self.basis = np.stack([-1j * H0, -1j * H1])
        self.sp = vo.DenseBasisSplit(ctx, self.basis)
        self.gp = vo.workloads.schrodinger_drive(self.N_SYS * world, self.N_SYS, rank * self.N_SYS)
        self.psi0 = np.zeros((self.N_SYS, self.NDIM), dtype=np.complex128)
        self.psi0[:, 0] = 1.0
        self.solver = vo.ExpCFMSolver(self.sp, self.gp, 0.0, 1.0e9, self.psi0, 0.1, group_similar=GROUP_SIMILAR).no_adaptive()
        if DYN_GROUP:
            self.solver.dynamic_grouping()
        self.solver.step()  # Chkpt at t0
        self.solvers = []
        # algorithmic FLOPs per trajectory-step (SURVEY.md §8d): sum over the step's E = 2 exponentials of m*_e x M x 8 n^2, with m*_e the
        # Taylor degree ONE system needs at its own theta = ||k_e||_1 (generator evaluated at the Gauss nodes like the kernel does),
        # averaged over systems and step times. The kernel plans per 16-system tile with the tile's largest theta, so it executes
        # at least this many terms.
        terms, self.theta = exp_algorithmic_terms("cfm4", self.basis, self.gp, 0.1)
        self.m_star = terms / 2.0
        self.flops_per_unit = terms * 2 * 8 * self.NDIM ** 2
        # round 1 quoted the degree at the a-priori bound theta_i <= h (|alpha_0| + |alpha_1|) (||B_0|| + a_i ||B_1||) (|cos| <= 1): kept beside
        # the exact figure as `frac_at_bound_degree` so that the two rounds can be compared
        norm1 = [np.abs(b).sum(axis=0).max() for b in self.basis]
        bound = 0.1 * (0.53867513459481288225 + 0.038675134594812882255) * (norm1[0] + self.gp[:, 0, 0] * norm1[1])
        self.flops_per_unit_bound = float(_plan_terms(bound[:: max(1, len(bound) // 4096)]).mean()) * 2 * 2 * 8 * self.NDIM ** 2
        self.bytes_per_unit = None

    def restart(self):
        self.solver.reset()  # back to the initial states the solver keeps on the device
        self.solver.step()

    def run_steps(self, k):
        self.solver.run(max_calls=k)

    def outputs(self):
        st = self.solver.stats()
        return {"psi": self.solver.current()[1].view(np.float64).reshape(self.N_SYS, self.NDIM, 2), "t": st["t"], "h": st["h"]}

    def units(self, k):
        return float(k) * self.N_SYS

    def e2e_setup(self, group=None):
        import torch
        self.pin_in = torch.from_numpy(self.psi0.view(np.float64).copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        self.e_solver = self.vo.ExpCFMSolver(self.sp, self.gp, 0.0, 10.0, self.psi0, 0.1, group_similar=GROUP_SIMILAR).no_adaptive()
        if DYN_GROUP:
            self.e_solver.dynamic_grouping()

    def e2e_step(self):
        self.e_solver.reset(self.pin_in.numpy().view(np.complex128))  # H2D of the initial states
        st = self.e_solver.run()
        self.e_solver.current(out=self.pin_out.numpy().view(np.complex128))  # D2H of the final states
        return float(st.counts["Step"]), self.pin_in.numel() * 8, self.pin_out.numel() * 8


class SchrodingerMagnusDense(SchrodingerCFM4):
    """Config 5 with THREE generator matrices (H0 and two independently driven couplings) whose commutators leave their span: 4th-order
    Magnus (exp/magnus.rs:28-83) with commutator(l0, l1) formed densely per system on the tensor cores (vo_exp_set_dense_commutator)."""
    name = "schrodinger_magnus_dense"
    label = ("config 5, generators not closed under commutation: Magnus-4 (one commutator), 10^5 driven 64-level systems with three generator "
             "matrices, h = 0.1, fixed step; [L0, L1] = two dense 64 x 64 complex products per system and step on the FP64 tensor cores")

    def __init__(self, vo, ctx, rank, world, n_batches):
        self.vo, self.ctx = vo, ctx
        H0, H1 = vo.workloads.schrodinger_system(self.NDIM)
        _, H2 = vo.workloads.schrodinger_system(self.NDIM, seed_h1=19)
        self.basis = np.stack([-1j * H0, -1j * H1, -1j * H2])
        self.sp = vo.DenseBasisSplit(ctx, self.basis)
        g1 = vo.workloads.schrodinger_drive(self.N_SYS * world, self.N_SYS, rank * self.N_SYS)
        g2 = vo.workloads.schrodinger_drive(self.N_SYS * world, self.N_SYS, rank * self.N_SYS, seed=23)
        self.gp = np.concatenate([g1, g2 * np.array([0.5, 1.0, 1.0])], axis=1)
        self.psi0 = np.zeros((self.N_SYS, self.NDIM), dtype=np.complex128)
        self.psi0[:, 0] = 1.0
        self.solver = vo.MagnusExpLinearSolver(self.sp, self.gp, 0.0, 1.0e9, self.psi0, 0.1, dense_commutator=True).no_adaptive()
        self.solver.step()  # Chkpt at t0
        self.solvers = []
        # algorithmic FLOPs per trajectory-step: the commutator (2 complex n x n products = 2 * 8 n^3) on the tensor cores, plus the Taylor
        # series of exp(Omega) applied by matrix-vector products (m* terms of 8 n^2, m* at the 1-norm of Omega itself, as the kernel plans)
        self.m_star, self.theta = exp_algorithmic_terms("magnus_dense", self.basis, self.gp, 0.1)
        self.flops_per_unit = 2 * 8 * self.NDIM ** 3 + self.m_star * 8 * self.NDIM ** 2
        self.bytes_per_unit = None

    def e2e_setup(self, group=None):
        import torch
        self.pin_in = torch.from_numpy(self.psi0.view(np.float64).copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        self.e_solver = self.vo.MagnusExpLinearSolver(self.sp, self.gp, 0.0, 1.0, self.psi0, 0.1, dense_commutator=True).no_adaptive()


class SchrodingerMagnusApplied(SchrodingerMagnusDense):
    """The same problem with the commutator APPLIED inside the Taylor series (vo_exp_set_applied_commutator): Omega T = W1 T + b2 (L0 (L1 T) -
    L1 (L0 T)), three passes over the shared basis per term on the tensor cores, no matrix formed per system."""
    name = "schrodinger_magnus_applied"
    label = ("config 5, generators not closed under commutation: Magnus-4 with the commutator applied by products inside the Taylor series "
             "(never formed), 10^5 driven 64-level systems with three generator matrices, h = 0.1, fixed step")

    def __init__(self, vo, ctx, rank, world, n_batches):
        super().__init__(vo, ctx, rank, world, n_batches)
        self.solver = vo.MagnusExpLinearSolver(self.sp, self.gp, 0.0, 1.0e9, self.psi0, 0.1, group_similar=GROUP_SIMILAR, applied_commutator=True).no_adaptive()
        if DYN_GROUP:
            self.solver.dynamic_grouping()
        self.solver.step()
        # algorithmic FLOPs per trajectory-step: 3 passes x M (3 basis matrices) x 8 n^2 per Taylor term; the degree is the one a system
        # needs at the bound ||Omega||_1 <= ||W1|| + 2 |b2| ||L0|| ||L1|| the kernel plans with (generator at the Gauss nodes)
        self.m_star, self.theta = exp_algorithmic_terms("magnus_applied", self.basis, self.gp, 0.1)
        self.flops_per_unit = 3 * 3 * self.m_star * 8 * self.NDIM ** 2

    def e2e_setup(self, group=None):
        import torch
        self.pin_in = torch.from_numpy(self.psi0.view(np.float64).copy()).pin_memory()
        self.pin_out = torch.empty_like(self.pin_in).pin_memory()
        self.e_solver = self.vo.MagnusExpLinearSolver(self.sp, self.gp, 0.0, 1.0, self.psi0, 0.1, group_similar=GROUP_SIMILAR, applied_commutator=True).no_adaptive()
        if DYN_GROUP:
            self.e_solver.dynamic_grouping()


WORKLOADS = {w.name: w for w in (LorenzRK4, VdpDopri5, HeatRK4, HeatRK4Fused, HeatRK4DD, SchrodingerCFM4, SchrodingerMagnusDense, SchrodingerMagnusApplied)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU side: the oracle in the reference's un-fused shape (one solver object per trajectory), all host threads
# ---------------------------------------------------------------------------------------------------------------------
def cpu_run(workload, n_traj, n_steps, threads):
    """Returns (units, seconds) for n_traj trajectories x n_steps RK steps (or attempts) on the host."""
    from oracle import oracle_lib as ol
    import vecode_b200 as vo
    if workload == "lorenz_rk4":
        x0 = vo.workloads.lorenz_x0(n_traj)
        params = np.tile(vo.workloads.LORENZ_PARAMS, (n_traj, 1))
        t0 = time.perf_counter()
        r = ol.rk_ensemble("LORENZ63", params, ol.builtin_tableau(1), 0.0, 1.0e9, x0, 1e-3, n_threads=threads, max_calls=n_steps + 1)
        dt = time.perf_counter() - t0
        return float(r["accepted"].sum()), dt
    if workload == "vdp_dopri5":
        mu = vo.workloads.vdp_mu(N_TRAJ)[:: max(1, N_TRAJ // n_traj)][:n_traj]
        x0 = vo.workloads.vdp_x0(len(mu))
        t0 = time.perf_counter()
        r = ol.rk_ensemble("VDP", mu[:, None], ol.builtin_tableau(2), 0.0, 1.0e9, x0, 1e-3, n_threads=threads, adaptive=True, rtol=1e-6,
                           max_calls=n_steps + 1)
        dt = time.perf_counter() - t0
        return float(r["accepted"].sum() + r["rejected"].sum()), dt
    if workload == "schrodinger_cfm4":
        H0, H1 = vo.workloads.schrodinger_system(64)
        basis = np.stack([-1j * H0, -1j * H1])
        gp = vo.workloads.schrodinger_drive(SchrodingerCFM4.N_SYS)[:n_traj]
        psi0 = np.zeros((n_traj, 64), dtype=np.complex128)
        psi0[:, 0] = 1.0
        t0 = time.perf_counter()
        r = ol.exp_ensemble("cfm4", basis, gp, psi0, 0.0, 1.0e9, 0.1, no_adaptive=True, max_calls=n_steps + 1, n_threads=threads)
        dt = time.perf_counter() - t0
        return float(r["accepted"].sum()), dt
    if workload == "heat_rk4":
        d = n_traj  # here: grid points
        u0 = vo.workloads.heat_u0(d)
        t0 = time.perf_counter()
        _, out, _ = ol.rk_solve("HEAT1D", [1.0], ol.builtin_tableau(1), 0.0, 1.0e9, u0, 0.25, max_calls=n_steps + 1)
        dt = time.perf_counter() - t0
        return float(out.n_accept) * d, dt
    raise KeyError(workload)


def cpu_baseline(workload, budget_s=12.0):
    from oracle import oracle_lib as ol
    name = workload
    workload = "heat_rk4" if workload.startswith("heat_rk4") else workload  # the reference's path is the same single-state solve
    threads = ol.hardware_threads() if workload != "heat_rk4" else 1
    if workload == "heat_rk4":
        n, steps = 1 << 20, 2
    elif workload == "schrodinger_cfm4":
        n, steps = 4 * threads, 2
    else:
        n, steps = 64 * threads, 50
    units, dt = cpu_run(workload, n, steps, threads)  # calibration
    rate = units / max(dt, 1e-6)
    target = budget_s * rate  # units of work that fill the budget
    if workload == "heat_rk4":
        steps = int(min(40, max(2, target / n)))
    elif workload == "schrodinger_cfm4":
        steps = 10
        n = int(min(SchrodingerCFM4.N_SYS, max(n, target / steps)))
    else:
        steps = 1000
        n = int(min(N_TRAJ, max(n, target / steps)))
    units, dt = cpu_run(workload, n, steps, threads)
    what = f"{n} grid points x {steps} RK4 steps" if workload == "heat_rk4" else f"{n} trajectories x {steps} calls of step()"
    out = {"value": units / dt, "unit": f"{WORKLOADS[name].unit_name}s/s", "cores": threads, "kind": "port",
           "sample": f"{what}, one solver object per trajectory, un-fused LinearCombination passes ({dt:.1f} s)"}
    if threads > 1:  # the reference itself is single-threaded: the same code on ONE core, on a 1/threads share of the sample (SURVEY.md §8d)
        n1 = max(1, n // threads)
        u1, d1 = cpu_run(workload, n1, steps, 1)
        out["single_core_value"] = u1 / d1
        out["single_core_sample"] = f"{n1} trajectories x {steps} calls of step() on one core ({d1:.1f} s)"
    return out


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path. The crate is Rust and cannot be compiled in
    this image, so this times the source-faithful C++ restatement (oracle/) with all host threads."""
    if rank != 0:
        return
    from oracle import oracle_lib as ol
    wl = "heat_rk4" if args.workload.startswith("heat_rk4") else args.workload
    threads = ol.hardware_threads() if wl != "heat_rk4" else 1
    total = args.steps + args.warmup
    per_step_budget = min(0.5, 90.0 / max(total, 1))
    if wl == "heat_rk4":
        n, inner = 1 << 18, 1
    elif wl == "schrodinger_cfm4":
        n, inner = 2 * threads, 1
    else:
        n, inner = 32 * threads, 250  # long enough that building one solver object per trajectory (the reference's shape) is amortised
    units, dt = cpu_run(wl, n, inner, threads)
    rate = units / max(dt, 1e-6)
    grow = max(1.0, per_step_budget * rate / units)
    n = int(min(N_TRAJ if wl != "heat_rk4" else (1 << 24), n * grow))
    for _ in range(args.warmup):
        cpu_run(wl, n, inner, threads)
    tot_units, t0 = 0.0, time.perf_counter()
    for _ in range(args.steps):
        u, _ = cpu_run(wl, n, inner, threads)
        tot_units += u
    el = time.perf_counter() - t0
    W = WORKLOADS[wl]
    val = tot_units / el
    sample = (f"each step = {n} {'grid points' if wl == 'heat_rk4' else 'trajectories'} x {inner} RK step(s) of the C++ restatement "
              f"(one solver object per trajectory, un-fused passes)")
    line = {"impl": "reference", "metric": "ensemble trajectory-steps/sec", "value": val, "unit": f"{W.unit_name}s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl, "what": W.label, "arith": "reference order (no FMA)"},
            "cpu_baseline": {"value": val, "unit": f"{W.unit_name}s/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": f"{W.unit_name}s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def roofline_of(W, w, units_per_rank, ms, launches, events_per_launch, peak, peak_src):
    """The `roofline` object of the dominant kernel from one timed region: algorithmic bytes (or FLOPs) per launch over the
    mean launch duration (CUDA events around the region, kernels back to back on the launching stream)."""
    kernel_ms = ms / max(launches, 1)
    if W in (SchrodingerCFM4, SchrodingerMagnusDense, SchrodingerMagnusApplied):
        p64 = os.path.join(ROOT, "profiles", "fp64_peaks.json")
        peak_tf, src = (json.load(open(p64))["dmma_tflops"], "measured by profiles/microbench/peaks.cu (profiles/fp64_peaks.json: dmma_tflops)") \
            if os.path.exists(p64) else (45.0, "nominal B200 FP64 tensor peak (no measured figure committed)")
        n_kernel = launches // 2 if (DYN_GROUP and W in (SchrodingerCFM4, SchrodingerMagnusApplied) and launches % 2 == 0) else launches  # the grouping's key kernel is counted too
        kernel_ms = ms / max(n_kernel, 1)
        ach = w.flops_per_unit * (units_per_rank / max(n_kernel, 1)) / (kernel_ms * 1e-3) / 1e12
        extra = {}
        if getattr(w, "flops_per_unit_bound", None):
            extra = {"frac_at_bound_degree": w.flops_per_unit_bound * (units_per_rank / max(n_kernel, 1)) / (kernel_ms * 1e-3) / 1e12 / peak_tf,
                     "bound_degree_note": "Taylor degree at the a-priori bound of theta (|cos| <= 1, |alpha_0| + |alpha_1|): the figure round 1 quoted; `frac` uses the exact per-system degree"}
        return {**extra, "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": ncu_traffic(W.name),
                "peak_source": src, "algorithmic_flops_per_unit": w.flops_per_unit, "taylor_degree": w.m_star, "theta": w.theta,
                "kernel_us": kernel_ms * 1e3,
                "note": ("FP64 tensor pipe (mma.sync DMMA): algorithmic FLOPs = sum over the step's 2 exponentials of m*_e x M(2 basis matrices) x 8 n^2 per trajectory-step, m*_e = the Taylor degree one system needs at its own theta (exp_algorithmic_terms); `taylor_degree` = mean m*_e; the step time includes the dynamic grouping (key kernel + radix sort)"
                         if W is SchrodingerCFM4 else
                         "FP64 tensor pipe: algorithmic FLOPs = 3 passes x m* x M(3 basis matrices) x 8 n^2 per trajectory-step (the commutator is applied, never formed)"
                         if W is SchrodingerMagnusApplied else
                         "algorithmic FLOPs = 2 x 8 n^3 (the dense commutator, on the FP64 tensor pipe) + m* x 8 n^2 (Taylor series of exp(Omega) by matrix-vector "
                         "products, FP64 FMA pipe) per trajectory-step, against the DMMA peak")}
    bytes_per_launch = W.bytes_per_unit * (units_per_rank / max(launches, 1)) / events_per_launch
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(W.name),
            "peak_source": peak_src, "algorithmic_bytes_per_unit": W.bytes_per_unit, "kernel_us": kernel_ms * 1e3,
            "note": "achieved = algorithmic bytes per launch / mean launch duration (CUDA events over the timed region, kernels back to back)"}


def n_batches_for(W, n_traj):
    """Independent batches rotated per GPU so that the working set is >= 3x the L2 (each launch then streams from HBM)."""
    if W in (HeatRK4, HeatRK4Fused, HeatRK4DD, SchrodingerCFM4, SchrodingerMagnusDense, SchrodingerMagnusApplied):
        return 1
    if os.environ.get("VECODE_BENCH_BATCHES"):  # experiment switch (e.g. 1 = L2-resident state): the reported line says so in config.l2
        return int(os.environ["VECODE_BENCH_BATCHES"])
    state_mb = W.state_mb * n_traj / 1.0e6
    return int(min(256, max(2, -(-3 * L2_MB // max(state_mb, 1e-9)))))


def multi_gpu_legs(vo, torch, dist, args, W, group, rank, world, local, barrier, max_over_ranks, peak, peak_src):
    """N > 1 only: (a) STRONG scaling — ONE ensemble of 10^6 trajectories sharded over the ranks, device-resident sweeps and
    whole solves gathered to rank 0; (b) config 5 sharded — 10^5 Schroedinger systems in all, CFM4, gathered to rank 0."""
    out = {}
    n_total = 1_000_000
    lo, hi = vo.workloads.shard_range(n_total, rank, world)
    n_loc = hi - lo
    try:
        ctx = vo.Context.on_torch_stream(local, arith=args.arith)
        adaptive = W is VdpDopri5
        if adaptive:
            tab, d = vo.ButcherTableu.builtin("DOPRI5"), 2
            mu = vo.workloads.vdp_mu(n_total, n_loc, lo)
            x0_host = vo.workloads.vdp_x0(n_loc)
            mk_rhs = lambda c, a, b: vo.Rhs(c, "VDP", 2, [mu[a:b].copy()])
            mk = lambda c, rhs, x0, tf: vo.RK45Solver(rhs, 0.0, tf, x0, 1e-3, tableau=tab).with_tolerance(1e-6, 1e-6)
            tf = 20.0
        else:
            tab, d = vo.ButcherTableu.builtin("RK4"), 3
            x0_host = vo.workloads.lorenz_x0(n_loc, first=lo)
            mk_rhs = lambda c, a, b: vo.Rhs(c, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
            mk = lambda c, rhs, x0, tf: vo.RK45Solver(rhs, 0.0, tf, x0, 1e-3, tableau=tab)
            tf = 1.0
        # device-resident sweeps: enough batches of this rank's shard to exceed the L2
        nb = int(min(256, max(2, -(-3 * L2_MB // max(W.state_mb * n_loc / 1.0e6, 1e-9)))))
        rhs = mk_rhs(ctx, 0, n_loc)
        x0 = vo.Ensemble.from_host(ctx, x0_host)
        solvers = [mk(ctx, rhs, x0, 1.0e9) for _ in range(nb)]
        vo.step_many(solvers, adaptive, 1 + max(1, int(40.0e-3 / (nb * 4.0e-6))))  # Chkpt + ~40 ms of spin-up
        steps = 2000
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        vo.step_many(solvers, adaptive, steps // nb)
        ev1.record()
        barrier()
        ms = max_over_ranks(ev0.elapsed_time(ev1))
        done = (steps // nb) * nb
        out["strong_scaling"] = {"what": f"ONE ensemble of {n_total} trajectories sharded over {world} GPUs ({n_loc} per GPU), device-resident sweeps, {nb} batches per GPU",
                                 "value": done * float(n_total) / (ms * 1e-3), "unit": f"{W.unit_name}s/s", "ms_per_step": ms / done, "steps": done, "scaling": "strong"}
        del solvers
        # whole solves of the one ensemble through the sharded pipeline, gathered to rank 0
        pin_in = torch.from_numpy(x0_host.copy()).pin_memory()
        pin_full = torch.empty((n_total, d), dtype=torch.float64).pin_memory() if rank == 0 else None

        def make(c, a, b, x0c):
            return mk(c, mk_rhs(c, a, b), x0c, tf)
        il = adaptive  # round-robin sharding balances the mu sweep
        if il:
            n_il = max(0, -(-(n_total - rank) // world))
            mu_il = vo.workloads.vdp_mu(n_total)[rank::world].copy()
            pin_in = torch.from_numpy(vo.workloads.vdp_x0(n_il)).pin_memory()

            def make(c, a, b, x0c):  # noqa: F811
                return mk(c, vo.Rhs(c, "VDP", 2, [mu_il[a:b].copy()]), x0c, tf)
        sh = vo.pipeline.ShardedChunkedSolve(group, n_total, d, make, parts=E2E_PARTS, arith=args.arith, interleave=il)
        full = None if pin_full is None else pin_full.numpy()
        sh.solve(pin_in.numpy(), full, adaptive=adaptive)
        barrier()
        g0 = time.perf_counter()
        units = 0.0
        for _ in range(3):
            sts = sh.solve(pin_in.numpy(), full, adaptive=adaptive)
            units += float(sum(st.counts["Step"] + st.counts["Reject"] for st in sts))
        barrier()
        e_ms = max_over_ranks((time.perf_counter() - g0) * 1e3)
        u = torch.tensor([units], device="cuda", dtype=torch.float64)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
        out["strong_scaling"]["e2e"] = {"value": float(u.item()) / (e_ms * 1e-3), "unit": f"{W.unit_name}s/s", "ms_per_solve": e_ms / 3,
                                        "what": "whole solves of the one ensemble: shard upload, integrate, chunk-wise NCCL gather + device-to-host copy on rank 0"}
    except Exception as e:
        out["strong_scaling_error"] = repr(e)
    try:
        n_sys = SchrodingerCFM4.N_SYS
        lo, hi = vo.workloads.shard_range(n_sys, rank, world)
        ctx5 = group.ctxs[0]
        H0, H1 = vo.workloads.schrodinger_system(64)
        sp = vo.DenseBasisSplit(ctx5, np.stack([-1j * H0, -1j * H1]))
        gp = vo.workloads.schrodinger_drive(n_sys, hi - lo, lo)
        psi0 = np.zeros((hi - lo, 64), dtype=np.complex128)
        psi0[:, 0] = 1.0
        solver = vo.ExpCFMSolver(sp, gp, 0.0, 10.0, psi0, 0.1, group_similar=GROUP_SIMILAR).no_adaptive()
        if DYN_GROUP:
            solver.dynamic_grouping()
        pin_full = torch.empty((n_sys, 128), dtype=torch.float64).pin_memory() if rank == 0 else None
        rows = [vo.workloads.shard_range(n_sys, r, world) for r in range(world)]

        def solve_once():
            solver.reset(psi0)
            st = solver.run()
            state = solver.state_ensemble()  # [n_loc][64] complex in the caller's order, as an ensemble of 128-component rows (AoS = SoA for the copy)
            group.gather_placed([state], [(b - a) * 128 for a, b in rows], [a * 128 for a, _ in rows], None if pin_full is None else pin_full.numpy().reshape(1, -1),
                                root=0, layout="soa")
            group.sync()
            return float(st.counts["Step"])
        solve_once()
        barrier()
        g0 = time.perf_counter()
        units = sum(solve_once() for _ in range(2))
        barrier()
        e_ms = max_over_ranks((time.perf_counter() - g0) * 1e3)
        u = torch.tensor([units], device="cuda", dtype=torch.float64)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
        ok = None
        if rank == 0:
            nrm = np.linalg.norm(pin_full.numpy().view(np.complex128), axis=1)
            ok = bool(np.all(np.abs(nrm - 1.0) < 1e-10))
        out["schrodinger_cfm4_sharded"] = {"what": f"config 5: {n_sys} systems in all, CFM4, 100 steps, sharded over {world} GPUs, final states gathered to rank 0 (NCCL + one D2H)",
                                           "value": float(u.item()) / (e_ms * 1e-3), "unit": "trajectory-steps/s", "ms_per_solve": e_ms / 2, "scaling": "strong",
                                           "unitarity_ok": ok}
    except Exception as e:
        out["schrodinger_cfm4_sharded_error"] = repr(e)
    return out


def HOST_SYNC_DEFAULT(world):
    """Several ranks per box share the host's hardware threads (8 ranks x 5 threads on 16): waits yield there. Measured on one GPU
    (profiles/r02_host_sync.md): with all hardware threads free spin 6.46 / yield 6.48 / blocking 7.81 ms per e2e solve, pinned to two
    hardware threads 6.73 / 6.49 / 7.25 ms."""
    return "yield" if world > 1 else "spin"


def host_sync_policy(local, mode):
    """How this process's synchronisations wait (flags of the device's primary context, set before anything initialises it):
    "spin" = CUDA's default, "yield" = spin but give the hardware thread away between polls (CU_CTX_SCHED_YIELD), "blocking" = sleep on
    an interrupt (CU_CTX_SCHED_BLOCKING_SYNC). A rank's e2e pipeline runs four chunk threads that wait in stream synchronisations; with
    4-8 ranks per box that is 20-40 waiting threads on the box's 16 hardware threads, and some rank's last chunk is late in most solves
    (DESIGN.md §6). Yielding keeps the wake-up latency of a spin when hardware threads are free and lets the threads that have launches
    or copies to issue run when they are not; a blocking wait pays its wake-up latency at every upload, reset and read-back."""
    import ctypes
    flag = {"yield": 2, "blocking": 4}.get(mode)
    if flag is None:
        return "spin (CUDA default)"
    try:
        cu = ctypes.CDLL("libcuda.so.1")
        dev = ctypes.c_int()
        if cu.cuInit(0) != 0 or cu.cuDeviceGet(ctypes.byref(dev), int(local)) != 0:
            return "spin (driver API unavailable)"
        fn = getattr(cu, "cuDevicePrimaryCtxSetFlags_v2", None) or cu.cuDevicePrimaryCtxSetFlags
        rc = fn(dev, flag)
        name = "yield (CU_CTX_SCHED_YIELD)" if flag == 2 else "blocking (CU_CTX_SCHED_BLOCKING_SYNC)"
        return name if rc == 0 else f"spin (cuDevicePrimaryCtxSetFlags -> {rc})"
    except Exception as e:  # noqa: BLE001
        return f"spin ({e!r})"


def numa_bind(torch, local):
    """Run this rank's host threads on the CPUs of its GPU's NUMA node, so that the pinned staging buffers it allocates
    (first touch) and the threads that drive its copies are local to the GPU's PCIe root. Returns the node, or None."""
    try:
        p = torch.cuda.get_device_properties(local)
        dev = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


# Blocking kernel (nvbench's method): after the synchronize and BEFORE the first event a spin kernel of this many microseconds is enqueued
# on the launching stream, so that the K timed launches are already queued when the device reaches the first event and the events
# bracket DEVICE time of the K steps — not the host's luck in getting its first launches out. One process on an idle box shows no
# difference (0.725 vs 0.731, r2h / r2i); with 2-8 processes per box the host side jitters (17.4 / 17.5 us per step without, 17.1 / 16.5
# with, 2 GPUs). 0 switches it off.
GATE_US = float(os.environ.get("VECODE_BENCH_GATE_US", "150"))
SPIN_UP_MS = 40.0  # untimed load right before the timed region, whatever --warmup says: clocks and caches in their steady state
DUMP_BYTES = 64_000_000  # --dump-outputs: all files together, headers included


def dump_outputs(path, arrays):
    """Writes `arrays` as path/<name>.npy in float64. Above DUMP_BYTES in all, the arrays of the most rows keep a fixed seeded sample of
    their rows (the same rows for each, ascending), whose indices go to path/rows.npy."""
    n = max(len(a) for a in arrays.values())
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        per_row = sum(a.nbytes // n for a in arrays.values() if len(a) == n) + 8
        rest = sum(a.nbytes for a in arrays.values() if len(a) != n) + 4096 * (len(arrays) + 1)
        rows = np.sort(np.random.default_rng(0).choice(n, (DUMP_BYTES - rest) // per_row, replace=False))
        arrays = {k: a[rows] if len(a) == n else a for k, a in arrays.items()}
        arrays["rows"] = rows
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def main():
    global N_TRAJ
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="vdp_dopri5", choices=sorted(WORKLOADS),
                    help="default: config 3, the configuration BASELINE.json's north-star target (>= 70 %% of HBM peak) is quoted on")
    ap.add_argument("--arith", default="fast", choices=["strict", "fast"],
                    help="fast: FMA contraction and the reformulated controller (adaptive runs within rtol, fixed-step <= 1e-12 of the oracle, "
                         "tests/test_gpu_rk.py); strict: the reference's un-fused operation order, bit-identical to the oracle")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--events-per-launch", type=int, default=1)
    ap.add_argument("--n-traj", type=int, default=N_TRAJ, help="trajectories per batch (experiments only; the named configs use 10^6)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary workload summary")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float64, rank 0's "
                    f"trajectories, at most {DUMP_BYTES // 1_000_000} MB in all: a fixed sample of the rows of a larger output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed (--impl b200)")
    args.warmup = max(args.warmup, 3)
    N_TRAJ = args.n_traj
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import vecode_b200 as vo

    # VECODE_BENCH_HOST_SYNC = spin | yield | blocking (VECODE_BENCH_BLOCKING_SYNC=1: the older name of "blocking"). Blocking waits measured
    # 6.5 -> 7.8 ms per e2e solve at 2 GPUs, so they stay an experiment switch.
    sync_mode = os.environ.get("VECODE_BENCH_HOST_SYNC", "blocking" if os.environ.get("VECODE_BENCH_BLOCKING_SYNC") == "1" else HOST_SYNC_DEFAULT(world))
    host_sync = host_sync_policy(local, sync_mode)
    torch.cuda.set_device(local)
    numa = numa_bind(torch, local) if world > 1 else None  # pinned buffers and copy threads next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    peak, peak_src = peaks()

    def device_leg(Wc, arith, steps, warmup, k_events=1, r=0, wsize=1, sync_ranks=False):
        """W untimed warm-up steps (after one pass over EVERY batch and a spin-up), then exactly `steps` timed steps between
        barrier + synchronize, CUDA events on the launching stream, max over ranks."""
        c2 = vo.Context.on_torch_stream(local, arith=arith)
        nb = n_batches_for(Wc, N_TRAJ)
        w2 = Wc(vo, c2, r, wsize, nb)
        for s_ in getattr(w2, "solvers", []):
            s_.set_events_per_launch(k_events)
        w2.run_steps(max(nb, 1))  # every batch has been through the kernel once (first-touch, module load, lazy allocations)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        w2.run_steps(max(nb, 4))
        ev1.record()
        torch.cuda.synchronize()
        per_step_ms = max(ev0.elapsed_time(ev1) / max(nb, 4), 1e-4)
        if sync_ranks:
            per_step_ms = max_over_ranks(per_step_ms)  # every rank runs the same number of spin-up steps (heat_rk4_dd has a collective inside)
        spin = int(min(max(SPIN_UP_MS / per_step_ms, 1), 100000))
        w2.run_steps(spin)
        # the spin-up's length follows the measured step time: start over, so that what the warm-up and the timed steps compute depends
        # on the arguments alone (two builds compare output for output, --dump-outputs)
        w2.restart()
        w2.run_steps(max(nb, 1))
        w2.run_steps(warmup)
        if sync_ranks:
            barrier()
        else:
            torch.cuda.synchronize()
        l0 = c2.launch_count
        if GATE_US > 0:
            # torch's spin kernel, untimed, not counted in gpu_launches; it touches no solver state, so no vo_ctx_fence(): the first timed launch
            # follows it in stream order and finds its own predecessor's generation flag already published
            torch.cuda._sleep(int(GATE_US * 1.9e3))
        ev0.record()
        w2.run_steps(steps)
        ev1.record()
        if sync_ranks:
            barrier()
        else:
            torch.cuda.synchronize()
        ms2 = ev0.elapsed_time(ev1)
        if sync_ranks:
            ms2 = max_over_ranks(ms2)
        launches = c2.launch_count - l0
        units = w2.units(steps) * k_events
        return w2, c2, nb, ms2, launches, units

    W = WORKLOADS[args.workload]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t_wall0 = time.time()
    w, ctx, n_batches, ms, launches, units_per_rank = device_leg(W, args.arith, args.steps, args.warmup, args.events_per_launch, rank, world, sync_ranks=True)
    outputs = w.outputs() if args.dump_outputs and rank == 0 else None  # before the load below steps on
    # keep the same load up until the clock sampler has seen it (short timed regions are over before the first sample)
    while time.time() - t_wall0 < 0.6:
        w.run_steps(max(args.steps // 4, 16))
        torch.cuda.synchronize()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None

    value = units_per_rank * world / (ms * 1e-3)
    launches_per_step = launches / max(args.steps, 1)
    roofline = roofline_of(W, w, units_per_rank, ms, launches, args.events_per_launch, peak, peak_src)

    # ---- end to end through the public API with host buffers -----------------------------------------------------------
    # N > 1: the ranks form a vo_group (NCCL inside the library; torch.distributed only carries the 128-byte id) and every
    # e2e step ends with the final gather of the whole ensemble into rank 0's pinned host array, inside the timed region.
    group = None
    if world > 1:
        group = vo.group.Group.from_torch_distributed(vo.Context(local, arith=args.arith, urgency=8))  # the gather stream goes ahead of the chunks still integrating
    w.e2e_setup(group)
    w.e2e_step()  # warm
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e_units, h2d, d2h = 0.0, 0, 0
    for _ in range(args.e2e_steps):
        u, h2d, d2h = w.e2e_step()
        e_units += u
    e1.record()
    barrier()
    e_ms = max_over_ranks(e0.elapsed_time(e1))
    if world > 1:
        u = torch.tensor([e_units], device="cuda", dtype=torch.float64)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
        e_units = float(u.item())
    sharded = world > 1 and getattr(w, "e_sharded", None) is not None
    e2e = {"value": e_units / (e_ms * 1e-3), "unit": f"{W.unit_name}s/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "steps": args.e2e_steps, "ms_per_step": e_ms / args.e2e_steps,
           "what": "per e2e step: upload x0 from pinned host memory, one whole solve of the config through RK45Solver.run(), download the final state"
                   + (f"; the ensemble in {E2E_PARTS} chunks on their own streams and host threads (pipeline.ChunkedSolve), copies overlapping the integration"
                      if W in (LorenzRK4, VdpDopri5) and E2E_PARTS > 1 else "")
                   + (f"; ONE ensemble of {world} x {N_TRAJ} trajectories: every rank uploads its shard, and each finished chunk is gathered to rank 0 with "
                      "vo_group_gather_placed (NCCL over NVLink from device state, then one device-to-host copy into rank 0's pinned array of the WHOLE "
                      "ensemble) inside the timed region; h2d bytes are per rank, d2h bytes are rank 0's" if sharded else "")}

    gather_ms = None
    if sharded:
        # the final gather on its own, for reference: the rank's whole shard in one piece -> rank 0's pinned host array
        shard_ens = vo.Ensemble.from_host(group.ctxs[0], w.x0_host)
        full = w.pin_full.numpy() if rank == 0 else None
        group.gather([shard_ens], N_TRAJ * world, root=0, out=full)  # NCCL sets up its channels on first use
        barrier()
        g0 = time.perf_counter()
        for _ in range(3):
            group.gather([shard_ens], N_TRAJ * world, root=0, out=full)
        barrier()
        gather_ms = max_over_ranks((time.perf_counter() - g0) * 1e3 / 3)
        if rank == 0:
            assert np.array_equal(full[-N_TRAJ:], vo.workloads.lorenz_x0(N_TRAJ, first=(world - 1) * N_TRAJ) if W is LorenzRK4 else vo.workloads.vdp_x0(N_TRAJ))

    multi = None
    if world > 1 and not args.no_also and W in (LorenzRK4, VdpDopri5):
        multi = multi_gpu_legs(vo, torch, dist, args, W, group, rank, world, local, barrier, max_over_ranks, peak, peak_src)

    also = None
    if rank == 0 and world == 1 and not args.no_also:
        # The other configs and arithmetic modes, short runs, each a full roofline object measured the same way as the headline.
        del w
        also = {}

        def leg(key, Wc, arith, steps, k_events=1):
            try:
                w2, c2, nb, ms2, l2, units = device_leg(Wc, arith, steps, 3, k_events)
                out = {"value": units / (ms2 * 1e-3), "unit": f"{Wc.unit_name}s/s", "arith": arith, "events_per_launch": k_events, "steps": steps,
                       "ms_per_step": ms2 / steps, "gpu_launches": int(l2), "batches": nb}
                if k_events == 1:
                    out["roofline"] = roofline_of(Wc, w2, units, ms2, l2, 1, peak, peak_src)
                del w2
                also[key] = out
            except Exception as e:  # secondary figures only
                also[key] = {"error": str(e)}

        other = "strict" if args.arith == "fast" else "fast"
        if W is not VdpDopri5:
            leg("vdp_dopri5_fast", VdpDopri5, "fast", 1400)
        leg(f"vdp_dopri5_{other}" if W is VdpDopri5 else "vdp_dopri5_strict", VdpDopri5, other if W is VdpDopri5 else "strict", 1400)
        if W is not LorenzRK4:
            leg("lorenz_rk4_fast", LorenzRK4, "fast", 3200)
        leg(f"lorenz_rk4_{other}" if W is LorenzRK4 else "lorenz_rk4_strict", LorenzRK4, other if W is LorenzRK4 else "strict", 3200)
        leg("lorenz_rk4_fused16", LorenzRK4, "fast", 320, k_events=16)
        if W not in (HeatRK4, HeatRK4Fused):
            leg("heat_rk4", HeatRK4, "fast", 40)
            leg("heat_rk4_fused", HeatRK4Fused, "fast", 100)
        if W is not SchrodingerCFM4:
            leg("schrodinger_cfm4", SchrodingerCFM4, "fast", 10)
        if W is not SchrodingerMagnusApplied:
            leg("schrodinger_magnus_applied", SchrodingerMagnusApplied, "fast", 6)
        if W is not SchrodingerMagnusDense:
            leg("schrodinger_magnus_dense", SchrodingerMagnusDense, "fast", 4)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cpu = cpu_baseline(args.workload)
        except KeyError:  # no CPU restatement of this variant (e.g. the dense-commutator Magnus)
            cpu = None

    if rank == 0:
        line = {"metric": "ensemble trajectory-steps/sec", "value": value, "unit": f"{W.unit_name}s/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / max(args.steps, 1), "higher_is_better": True, "scaling": "strong" if W is HeatRK4DD else "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": W.name, "what": W.label, "trajectories_per_gpu": (1 if W in (HeatRK4, HeatRK4Fused, HeatRK4DD) else SchrodingerCFM4.N_SYS if W in (SchrodingerCFM4, SchrodingerMagnusDense, SchrodingerMagnusApplied) else N_TRAJ),
                           "arith": args.arith, "events_per_launch": args.events_per_launch,
                           "l2": f"{n_batches} independent batches of {W.state_mb} MB rotated per GPU (> {L2_MB} MB L2), so each launch streams from HBM"
                           if W not in (HeatRK4, HeatRK4Fused, HeatRK4DD, SchrodingerCFM4, SchrodingerMagnusDense, SchrodingerMagnusApplied) else ("state 512 MB per buffer > 126 MB L2" if W in (HeatRK4, HeatRK4Fused) else
                                                                        f"slab of {512 // world} MB per buffer per GPU" if W is HeatRK4DD else
                                                                        "compute-bound: 102 MB of state per launch, streamed once"),
                           "warmup_note": f"every batch touched once, then ~{SPIN_UP_MS:.0f} ms of the same launches, a restart from the initial state with every batch "
                                          f"touched once more, and the {args.warmup} warm-up steps, all untimed, before the {args.steps} timed steps",
                           "timing": ((f"barrier + synchronize, a {GATE_US:.0f} us blocking kernel (torch.cuda._sleep, untimed), event, {args.steps} steps, event, barrier + synchronize: the "
                                       "launches are queued behind the blocking kernel, so the events bracket device time of the steps (VECODE_BENCH_GATE_US=0: without). "
                                       if GATE_US > 0 else "barrier + synchronize, event, steps, event, barrier + synchronize (no blocking kernel). ") +
                                      "A region of K launches costs about 14 us + K x the steady launch time (tools/offset_probe.py): the first launch has no predecessor "
                                      "to overlap its ramp-up with and the last none to hide its tail"),
                           "parallelism": (f"domain-decomposed x{world}: ghost refresh (all-gather of {8 * DD_K} doubles per rank) every {DD_K} steps" if W is HeatRK4DD
                                           else f"trajectory-sharded x{world}, no data-path collective")},
                "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "launches_per_step": launches_per_step, "clocks": clocks}
        if numa is not None:
            line["config"]["numa_node_rank0"] = numa
        line["config"]["host_sync"] = host_sync
        if gather_ms is not None:
            line["final_gather_ms"] = gather_ms
            line["final_gather_note"] = (f"vo_group_gather of the whole ensemble ({world} x {W.state_mb if W is LorenzRK4 else 16} MB of state) on its own: NCCL into rank 0's "
                                         "device buffer + one device-to-host copy into pinned memory; inside e2e the same transfer runs chunk by chunk")
        if multi:
            line["multi_gpu"] = multi
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if also:
            line["also"] = also
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
