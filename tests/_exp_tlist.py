"""Both CPU restatements of the exponential solvers driven through an output-time list (ODEData.t_list, ode.rs:89) — test
infrastructure for tests/test_exp_tlist_oracle.py and tests/test_gpu_exp_checkpoints.py.

  exp_ensemble(...)  the C++ oracle (oracle/vecode_oracle.cpp, whose source tests/harness/exp_tlist_oracle.cpp includes) with a list,
                     the state of every system at each Chkpt / End event and the event of every call; compiled with the oracle's
                     flags into a temporary directory on first use.
  solve(...)         the pure-Python restatement (oracle/exp_oracle.py's schemes) through the same state machine, one system.

With the default list both compute what oracle_lib.exp_ensemble / exp_oracle.solve_fixed compute; the two must agree bit for bit.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle import exp_oracle as eo
from oracle import oracle_lib as ol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "harness", "exp_tlist_oracle.cpp")
STEP, CHKPT, REJECT, END = 0, 1, 2, 3  # ODEStep, ode.rs:42-48 (the oracle's EV_*)


class ExpTlistCfg(C.Structure):
    _fields_ = list(ol.ExpCfg._fields_) + [("n_tlist", C.c_int32), ("t_list", C.c_void_p), ("snap", C.c_void_p), ("events", C.c_void_p),
                                            ("events_cap", C.c_int64)]


_lib = None


def lib():
    """The shared object, built once per source version (-ffp-contract=off, like oracle/Makefile: no FMA may change a bit)."""
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in (SRC, os.path.join(ROOT, "oracle", "vecode_oracle.cpp")):
            h.update(open(p, "rb").read())
        so = os.path.join(tempfile.gettempdir(), f"vecode_exp_tlist_{h.hexdigest()[:16]}_{os.getuid()}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=c++17", "-pthread", "-shared", "-o", tmp, SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def exp_ensemble(scheme, basis, gp, psi0, t0, tf, h0, t_list=None, snapshots=False, events_cap=0, M_gen=None, cs=None, adaptive=False,
                 no_adaptive=True, rtol=1e-4, min_dt=1e-6, max_dt=1.0, order=3.0, alpha=0.9, max_calls=0, n_threads=1, tables=None):
    """oracle_lib.exp_ensemble's arguments and results, plus `t_list` in place of [t0, tf] and,
    when asked, "snap" [len(t_list)][N][n] complex (the state at each entry's Chkpt / End event) and "events" [N][events_cap] int8
    (STEP, CHKPT, REJECT, END of every call, -1 after the last)."""
    basis = np.ascontiguousarray(basis, dtype=np.complex128)
    M, n, _ = basis.shape
    M_gen = M if M_gen is None else M_gen
    psi = np.ascontiguousarray(psi0, dtype=np.complex128).copy()
    N = psi.shape[0]
    gp = np.ascontiguousarray(gp, dtype=np.float64).reshape(N, max(M_gen - 1, 0), 3)
    tl = None if t_list is None else np.ascontiguousarray(t_list, dtype=np.float64).ravel()
    snap = np.zeros((2 if tl is None else tl.size, N, n), dtype=np.complex128) if snapshots else None
    events = np.full((N, events_cap), -1, dtype=np.int8) if events_cap else None
    cfg = ExpTlistCfg(n, M, {"midpoint": 0, "cfm4": 1, "magnus42": 2, "cfm_table": 3}[scheme], int(adaptive), int(no_adaptive), 0, t0, tf, h0,
                      rtol, min_dt, max_dt, order, alpha, max_calls)
    if scheme == "cfm_table":  # cfm_general with run-time tables (c[k], alpha[s][k], alpha_err[s_err][k] | None), as oracle_lib takes them
        c_a = np.ascontiguousarray(tables[0], dtype=np.float64)
        a_a = np.ascontiguousarray(tables[1], dtype=np.float64).reshape(-1, c_a.size)
        e_a = None if tables[2] is None else np.ascontiguousarray(tables[2], dtype=np.float64).reshape(-1, c_a.size)
        cfg.n_nodes, cfg.n_rows, cfg.n_rows_err = c_a.size, a_a.shape[0], 0 if e_a is None else e_a.shape[0]
        cfg.c, cfg.alpha_tab, cfg.alpha_err_tab = c_a.ctypes.data, a_a.ctypes.data, None if e_a is None else e_a.ctypes.data
    cfg.n_tlist = 0 if tl is None else tl.size
    cfg.t_list = None if tl is None else tl.ctypes.data
    cfg.snap = None if snap is None else snap.ctypes.data
    cfg.events, cfg.events_cap = (None, 0) if events is None else (events.ctypes.data, events_cap)
    t, h = np.zeros(N), np.zeros(N)
    acc, rej = np.zeros(N, dtype=np.int64), np.zeros(N, dtype=np.int64)
    csa = None if cs is None else np.ascontiguousarray(cs, dtype=np.float64)
    P = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    lib().orc_exp_tlist_ensemble(C.byref(cfg), P(basis.view(np.float64)), P(gp), C.c_int32(M_gen), P(csa), C.c_int64(N), P(psi.view(np.float64)),
                                 P(t), P(h), P(acc), P(rej), C.c_int32(n_threads))
    out = dict(psi=psi, t=t, h=h, accepted=acc, rejected=rej)
    if snap is not None:
        out["snap"] = snap
    if events is not None:
        out["events"] = events
    return out


def solve(scheme, sp, gp_i, M_gen, psi0, t0, tf, h, t_list=None, adaptive=False, rtol=1e-4, min_dt=1e-6, max_dt=1.0, order=3.0,
          alpha=0.9, max_calls=0, cs=None, adaptive_from=None):
    """One system through ODEData / ODEAdaptiveData (base/ode.rs:79-206, 249-253, 311-341) as orc_exp_ensemble drives it:
    step_size_of against t_list[tgt_t] (ode.rs:165-176), the scheme's try_step (exp_oracle.py), the controller on the 2-norm of the
    embedded error when `adaptive`, then advance / checkpoint_update. `adaptive_from` = c: calls 0 .. c-1 are step() (fixed), calls
    from c on step_adaptive(), as a caller who switches in mid-list makes them (None: `adaptive` for every call).
    Returns dict(x, t, h, accepted, rejected, events, dt, snap): `dt[j]` the step size of call j (0.0 for Chkpt / End),
    `snap[k]` the state x at the Chkpt / End event for t_list[k]."""
    from oracle.vecode_oracle import _libm, _rmax, _rmin, check_step
    g = eo.gen_cos(gp_i, M_gen, sp.M)
    gv = lambda ts: [g(tt) for tt in ts]
    tl = [t0, tf] if t_list is None else list(t_list)
    x, t, tgt, cur_h, prev_h = list(psi0), t0, 0, h, h
    acc = rej = calls = 0
    events, dts, snap = [], [], [None] * len(tl)
    pw = 1.0 / order
    while max_calls <= 0 or calls < max_calls:
        ada = adaptive if adaptive_from is None else calls >= adaptive_from
        calls += 1
        ev, dt = (END, 0.0) if tgt >= len(tl) else (STEP, check_step(t, tl[tgt], cur_h))
        if ev == STEP and dt is None:
            ev, dt = (END if tgt >= len(tl) - 1 else CHKPT), 0.0
        h0 = cur_h
        if ev == STEP:
            if scheme == "midpoint":
                xf, xe = eo.midpoint(sp, g, t, x, dt), None
            elif scheme == "cfm4":
                xf, xe = eo.cfm_general(sp, gv, t, x, dt, eo.C_GAUSS_LEGENDRE_4, eo.CFM_R4_J2_GL, eo.CFM_R2_J1_GL if ada else None)
            else:
                xf, xe = eo.magnus_42(sp, g, t, x, dt, cs, want_err=ada)
            if ada:  # handle_step_adaptive, ode.rs:311-334
                nn = 0.0
                for a, b in xe:
                    nn = nn + (a * a + b * b)
                dxn = math.sqrt(nn)
                f = rtol / dxn if dxn != 0.0 else math.inf
                fp = _rmin(_rmax(alpha * _libm.pow(f, pw), 0.3), 2.0)
                prev_h, cur_h = cur_h, _rmin(_rmax(fp * h0, min_dt), max_dt)
                if f <= 1.0:
                    ev = REJECT
        events.append(ev)
        dts.append(dt)
        if ev == STEP:  # advance, ode.rs:184-188
            x, t = xf, t + dt
            acc += 1
        elif ev == REJECT:
            rej += 1
        else:  # checkpoint_update, ode.rs:192-195
            if tgt < len(tl):
                snap[tgt] = list(x)
            tgt, cur_h = tgt + 1, prev_h
            if ev == END:
                break
    return dict(x=x, t=t, h=cur_h, accepted=acc, rejected=rej, events=events, dt=dts, snap=snap)
