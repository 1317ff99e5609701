"""Output times and checkpoint snapshots of the Runge-Kutta solvers (vo_solver_set_t_list, vo_solver_enable_snapshots,
vo_solver_snapshot; ODEData.t_list, ode.rs:89, 165-176, 192-195): every trajectory raises Chkpt at each entry of t_list before
the last and End at the last, restores h = prev_h there, and the solver keeps the state it shows at each of those events.

Case table: the row, the kernel it reaches and the rule of small_plan (rk_small_launch.cuh) or solver.cu that selects it.

  row  kernel                              how it is reached
  F1   rk_fixed_kernel                     lock-step fixed steps, N odd (333); HARMONIC2D N = 64 (below one tile)
  F2   rk_fixed_staged_kernel              N even in [128, 1024) (640); N = 2048 with a 3-stage tableau (the S = 0 instantiation)
  F3   rk_fixed2w_staged_kernel            N even >= 1024, S in {4, 6, 7} (2500: ragged tail of 196)
  F4   lock-step stage path                set_stage_path(True) (640; HARMONIC2D N = 96)
  C1   rk_ctl_kernel                       per-trajectory control, N odd (333), adaptive and set_h_array; HARMONIC2D N = 64
  C2   rk_ctl_staged_kernel<CFG 1>         adaptive L2 through run() (8 events per launch): N = 2500 and 640
  C3   rk_ctl_staged_kernel<CFG 0>         with_norm("LINF"); fixed steps with set_h_array (2500)
  C4   rk_ctl2w_staged_kernel              adaptive L2, one event per launch, N = 2500 and 4096
  C5   per-trajectory stage path           ctl_prepare_kernel / ctl_commit_kernel (640; HARMONIC2D N = 96)
  C6   run-time compiled modules           a user RHS body (its ctl2w and CFG 1 kernels) and a user norm (CFG 0)
  H1   stage_heat_kernel                   one HEAT1D state, lock-step RK4, d = 4099
  H2   stage_heat_tma_kernel               d = 2^16
  H3   heat_fused_step_kernel              set_fused_step, d = 4099
  H4   stage path, host controller         one HEAT1D state, adaptive DOPRI5, d = 4096

Lists: every row takes a 5-entry list off the step grid (L5); every kernel takes one of 9 entries (L9, the shortest list read
from device memory) and one of 41 (L41); F3, C2 and C4 also take exactly 8 entries (L8, the last one held inline). F3, C2, C4,
C5 and H1 take EDGE: a first entry after t0 (the first call is a Step), a repeated entry (two Chkpt with no step between them,
two equal snapshots), entries closer together than h, and entries at t >= 4 on the grid of h = 0.1 where the accumulated t
misses the entry by one ulp (more than 2^-52) and check_step takes a clipped step of one ulp.

Reference: snapshot k is the final state of the oracle's solve whose list stops at entry k. The state machine reads only
t_list[tgt], so that solve makes the same calls up to entry k, and its End runs the same checkpoint_update as Chkpt: its final
h is the h restored at entry k.
Bars: fixed steps (STRICT) bit-identical, with equal per-trajectory accepted counts and t and event totals; adaptive (STRICT)
per-trajectory accepted and rejected counts equal, snapshots within 1e-12 relative and h within 1e-6 relative (see _h_close);
GPU against GPU bit-identical; FAST fixed steps within 1e-12 relative."""
import functools
from collections import namedtuple

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
L5 = (0.0, 0.1937, 0.4226, 0.7123, 1.0)
L8 = (0.0, 0.0611, 0.1937, 0.3, 0.4226, 0.55, 0.7123, 1.0)
L9 = (0.0, 0.0611, 0.1937, 0.3, 0.4226, 0.55, 0.7123, 0.8377, 1.0)
L41 = tuple(np.linspace(0.0, 1.0, 41))
# absolute times, h = 0.1: 0.2 is reached in two full steps, then 3.0 -> 3.3 -> 4.2 and 4.3 -> 4.5 in full steps whose sum falls
# one ulp short of the entry (a clipped step of 8.9e-16 follows); 4.2 twice; 4.2, 4.25, 4.3 closer together than h
EDGE = (0.2, 0.2, 3.0, 3.3, 4.2, 4.2, 4.25, 4.3, 4.5)
LISTS = {"L5": L5, "L8": L8, "L9": L9, "L41": L41, "EDGE": EDGE}

# kind, N, tableau, control ("fixed": lock-step step(), "h_array": per-trajectory fixed steps, "adaptive"), t_end of the
# fractional lists, h, rtol, options (stage_path, k = events per launch, norm)
Row = namedtuple("Row", "kind n tab control tf h rtol opts")
ROWS = {
    "F1": Row("LORENZ63", 333, "RK4", "fixed", 0.5, 0.01, None, {}),
    "F1-harmonic": Row("HARMONIC2D", 64, "RKF45_REF", "fixed", 1.0, 0.01, None, {}),
    "F2": Row("LORENZ63", 640, "RKF45_REF", "fixed", 0.5, 0.01, None, {}),
    "F2-S0": Row("LORENZ63", 2048, "RK3", "fixed", 0.5, 0.01, None, {}),
    "F3": Row("LORENZ63", 2500, "RK4", "fixed", 0.5, 0.01, None, {}),
    "F4": Row("LORENZ63", 640, "RK4", "fixed", 0.5, 0.01, None, {"stage_path": True}),
    "F4-harmonic": Row("HARMONIC2D", 96, "RKF45_REF", "fixed", 1.0, 0.01, None, {"stage_path": True}),
    "C1": Row("VDP", 333, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {}),
    "C1-h": Row("VDP", 333, "RK4", "h_array", 1.0, None, None, {}),
    "C1-harmonic": Row("HARMONIC2D", 64, "RKF45_REF", "adaptive", 1.0, 0.01, 1e-7, {}),
    "C2": Row("VDP", 2500, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {}),
    "C2-640": Row("VDP", 640, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {}),
    "C3-linf": Row("VDP", 640, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {"norm": "LINF"}),
    "C3-h": Row("VDP", 2500, "RKF45_REF", "h_array", 1.0, None, None, {}),
    "C4": Row("VDP", 2500, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {"k": 1}),
    "C4-4096": Row("VDP", 4096, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {"k": 1}),
    "C5": Row("VDP", 640, "DOPRI5", "adaptive", 1.0, 1e-3, 1e-6, {"stage_path": True}),
    "C5-harmonic": Row("HARMONIC2D", 96, "RKF45_REF", "adaptive", 1.0, 0.01, 1e-7, {"stage_path": True}),
}
FAMILIES = ["F1", "F2", "F3", "F4", "C1", "C1-h", "C2", "C3-linf", "C3-h", "C4", "C5"]  # each kernel of the table once
ORACLE_CASES = ([(r, "L5") for r in ROWS] + [(r, lst) for r in FAMILIES for lst in ("L9", "L41")] +
                [(r, "L8") for r in ("F3", "C2", "C4")] + [(r, "EDGE") for r in ("F3", "C2", "C4", "C5")] )
LISTS["HARM_A"], LISTS["HARM_B"] = (0.0, 0.35, 0.5, 1.0), (0.0, 0.3, 0.55, 1.0)  # the lists of the HARMONIC2D cases, as they were

# a 3-stage tableau (Kutta's third-order method) from slices: no unrolled instantiation, so the staged kernel runs with S = 0
RK3 = (np.array([0.0, 0.0, 0.0, 0.5, 0.5, 0.0, -1.0, 2.0, 1.0]), np.array([1.0 / 6.0, 2.0 / 3.0, 1.0 / 6.0]), None, 3)
VDP_BODY = """
dx[0] = x[1];
dx[1] = (p[0] * (1.0 - x[0] * x[0])) * x[1] - x[0];
"""


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _times(row, lst):
    """The list in absolute times: fractional lists scale to the row's t_end (a power of two: exact)."""
    return [float(v) for v in LISTS[lst]] if lst in ("EDGE", "HARM_A", "HARM_B") else [float(v) * row.tf for v in LISTS[lst]]


def _inputs(vo, row):
    """(params AoS [N][np], x0 AoS [N][d], per-trajectory h or None)"""
    n = row.n
    if row.kind == "LORENZ63":
        return np.tile(vo.workloads.LORENZ_PARAMS, (n, 1)), vo.workloads.lorenz_x0(n), None
    if row.kind == "HARMONIC2D":
        rng = np.random.default_rng(5 if n == 64 else 11)
        return 0.5 + rng.random((n, 1)), rng.standard_normal((n, 2)), None
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n) + 0.01 * np.cos(np.arange(2 * n)).reshape(n, 2)
    return mu[:, None], x0, (np.linspace(0.004, 0.01, n) if row.control == "h_array" else None)


def _otab(oracle, row):
    return RK3 if row.tab == "RK3" else oracle.builtin_tableau(oracle.TABLEAU_ID[row.tab])


def _edge(row, lst):
    """EDGE runs with h = 0.1; adaptive runs also cap the step at 0.1, so slow trajectories walk the same grid."""
    return lst == "EDGE"


def _solver(vo, ctx, row, lst, snapshots=True, rhs=None, upto=None):
    """The solver of `row` on list `lst` (cut after entry `upto` if given), t_list and snapshots set, not yet stepped."""
    params, x0, h_arr = _inputs(vo, row)
    t_list = _times(row, lst)
    if upto is not None:
        t_list = t_list[:upto + 1]
    tab = vo.ButcherTableu.from_slices(*RK3) if row.tab == "RK3" else vo.ButcherTableu.builtin(row.tab)
    if rhs is None:
        rhs = vo.Rhs(ctx, row.kind, x0.shape[1])
        for q in range(params.shape[1]):
            rhs.set_param(q, params[:, q].copy() if row.kind != "LORENZ63" else float(params[0, q]))
    h = 0.1 if _edge(row, lst) else (row.h or 1e-3)
    s = vo.RK45Solver(rhs, 0.0, t_list[-1], vo.Ensemble.from_host(ctx, x0), h, tableau=tab)
    if row.rtol:
        s.with_tolerance(row.rtol, row.rtol)
        if _edge(row, lst):
            s.with_step_range(1e-6, 0.1).with_init_step(0.1)
    s.set_t_list(t_list)
    if row.opts.get("stage_path"):
        s.set_stage_path(True)
    if "k" in row.opts:
        s.set_events_per_launch(row.opts["k"])
    if "norm" in row.opts:
        s.with_norm(row.opts["norm"])
    if h_arr is not None:
        s.set_h_array(h_arr)
    if snapshots:
        s.enable_snapshots()
    return s, t_list


def _drive(s, row, call=False):
    """run() (fused events), or one step()/step_adaptive() per call until Done; returns the summed event counts."""
    adaptive = row.control == "adaptive"
    if not call:
        st = s.run(adaptive=adaptive)
        assert st.kind == "Done"
        return st.counts
    tot = dict(Step=0, Chkpt=0, Reject=0, End=0)
    for _ in range(100000):
        st = s.step_adaptive() if adaptive else s.step()
        for key in tot:
            tot[key] += st.counts[key]
        if st.kind == "Done":
            return tot
    raise AssertionError("no End")


@functools.lru_cache(maxsize=None)
def _oracle_refs(row_name, lst):
    """Oracle solves over t_list[:k+1] for every k: [k] -> dict(x, t, h, accepted, rejected)."""
    from oracle import oracle_lib as oracle
    import vecode_b200 as vo
    row = ROWS[row_name]
    params, x0, h_arr = _inputs(vo, row)
    t_list = _times(row, lst)
    kw = dict(n_threads=8)
    if row.control == "adaptive":
        kw.update(adaptive=True, rtol=row.rtol, atol=row.rtol, norm=row.opts.get("norm", "L2"))
        if _edge(row, lst):
            kw.update(max_dt=0.1)
    h = 0.1 if _edge(row, lst) else (row.h or 0.0)
    return [oracle.rk_ensemble(row.kind, params, _otab(oracle, row), 0.0, t_list[k], x0, h, h0_arr=h_arr, t_list=t_list[:k + 1], **kw)
            for k in range(len(t_list))]


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _h_close(got, ref, what):
    """h after an entry, adaptive. The controller's pow is correctly rounded on the device and comes from glibc in the oracle, which
    now and then rounds the other way. The next error estimate, a difference of two solutions that agree to about rtol, magnifies
    that one ulp of h by about 1/rtol: h then differs by ~1e-10 relative, up to 2.3e-7 over the 4.5 time units of EDGE, while states
    stay within 1e-12. A wrong h restored at a checkpoint is off by a factor (0.3 to 2 per controller step)."""
    rel = np.abs(got - ref) / np.abs(ref)
    print(f"{what}: h bit-identical for {np.mean(got == ref):.4f} of trajectories, max relative difference {rel.max():.2e}")
    assert rel.max() <= 1e-6, (what, rel.max())


def _check_against_oracle(s, counts, row, t_list, refs, h_at=None):
    n, L = row.n, len(t_list)
    full = refs[-1]
    stats = s.stats()
    assert counts["Chkpt"] == n * (L - 1) and counts["End"] == n
    assert counts["Step"] == int(full["accepted"].sum()) and counts["Reject"] == int(full["rejected"].sum())
    assert np.array_equal(stats["accepted"], full["accepted"]) and np.array_equal(stats["rejected"], full["rejected"])
    if row.control == "adaptive":
        for k in range(L):
            err = _rel(s.snapshot(k).to_host(), refs[k]["x"])
            assert err <= 1e-12, (k, err)
        assert np.all(np.abs(stats["t"] - t_list[-1]) <= EPS)
        _h_close(stats["h"], full["h"], "final h")
        for k, h in (h_at or {}).items():
            _h_close(h, refs[k]["h"], f"h after entry {k}")
    else:
        for k in range(L):
            assert np.array_equal(_bits(s.snapshot(k).to_host()), _bits(refs[k]["x"])), k
        assert np.array_equal(stats["t"], full["t"]) and np.array_equal(stats["h"], full["h"])
    assert np.array_equal(_bits(s.snapshot(L - 1).to_host()), _bits(s.current()[1].to_host()))


@pytest.mark.parametrize("row,lst", ORACLE_CASES)
def test_snapshots_against_the_oracle(vo, ctx, row, lst):
    """Snapshot k equals the oracle's solve over t_list[:k+1] (fixed: bit for bit; adaptive: 1e-12), with equal per-trajectory
    counts and event totals and the same h at the end. Adaptive lists up to 9 entries long also check the h restored at every entry: the final h of a
    device solve whose list stops there (its End restores prev_h as a Chkpt does)."""
    r = ROWS[row]
    s, t_list = _solver(vo, ctx, r, lst)
    counts = _drive(s, r)
    refs = _oracle_refs(row, lst)
    h_at = {}
    if r.control == "adaptive" and len(t_list) <= 9:
        for k in range(len(t_list) - 1):
            part = _solver(vo, ctx, r, lst, snapshots=False, upto=k)[0]
            _drive(part, r)
            h_at[k] = part.stats()["h"]
    _check_against_oracle(s, counts, r, t_list, refs, h_at)


def _outputs(s, L):
    """Everything a run leaves behind, for bit-for-bit comparisons of two runs."""
    st = s.stats()
    return [s.current()[1].to_host()] + [s.snapshot(k).to_host() for k in range(L)] + [st[k] for k in ("t", "h", "accepted", "rejected", "dx_norm", "status")]


def _same(a, b):
    assert len(a) == len(b)
    for i, (u, v) in enumerate(zip(a, b)):
        assert np.array_equal(_bits(u), _bits(v)), i


@pytest.mark.parametrize("row", ["F3", "C4"])
@pytest.mark.parametrize("lst", ["L9", "EDGE"])
def test_snapshot_equals_current_at_the_event(vo, ctx, row, lst):
    """One call at a time: whenever a trajectory sits on t_list[k], current() shows snapshot k bit for bit, and the h it shows
    after its Chkpt / End there (the second time it is seen on t_list[k], the third for the second of two equal entries: the
    first is after the step that lands there, later ones may follow rejected attempts) is the oracle's. Snapshot k read in
    mid-run keeps the rows of the trajectories that had passed entry k: rows are written once."""
    r = ROWS[row]
    s, t_list = _solver(vo, ctx, r, lst)
    L, n = len(t_list), r.n
    seen = np.zeros((L, n), dtype=bool)
    want = np.zeros((L, n, 2 if r.kind == "VDP" else 3))
    want_h = np.zeros((L, n))
    seen_at = np.zeros((L, n), dtype=int)  # calls after which the trajectory sat on t_list[k]
    rank = [1 + sum(t_list[j] == t_list[k] for j in range(k + 1)) for k in range(L)]
    kmid = L // 2
    early = None
    adaptive = r.control == "adaptive"
    def observe():
        st = s.stats()
        x = s.current()[1].to_host()
        for k, tk in enumerate(t_list):
            at = np.abs(st["t"] - tk) <= EPS
            want[k, at], seen[k, at] = x[at], True
            seen_at[k, at] += 1
            after = at & (seen_at[k] == rank[k])
            want_h[k, after] = st["h"][after]
        return st

    for _ in range(20000):
        st = observe()
        passed = st["t"] > t_list[kmid] + 1e-9
        if early is None and passed.any():  # the first call after which some trajectory is past entry kmid
            early = (passed, s.snapshot(kmid).to_host()[passed])
        if (s.step_adaptive() if adaptive else s.step()).kind == "Done":
            break
    observe()
    assert seen.all() and np.all(seen_at >= np.array(rank)[:, None])
    for k in range(L):
        assert np.array_equal(_bits(s.snapshot(k).to_host()), _bits(want[k])), k
    passed, rows = early
    assert np.array_equal(_bits(s.snapshot(kmid).to_host()[passed]), _bits(rows))
    if lst == "EDGE":
        assert np.array_equal(_bits(s.snapshot(4).to_host()), _bits(s.snapshot(5).to_host()))  # 4.2 twice
    refs = _oracle_refs(row, lst)
    for k in range(L):
        if adaptive:
            _h_close(want_h[k], refs[k]["h"], f"h after entry {k}")
        else:
            assert np.array_equal(want_h[k], refs[k]["h"]), k


@pytest.mark.parametrize("row", ["F3", "C2"])
@pytest.mark.parametrize("lst", ["L41", "EDGE"])
def test_fused_run_equals_single_calls(vo, ctx, row, lst):
    """run() fuses 16 (lock-step) or 8 (per-trajectory) events per launch, so checkpoints fall inside launches: the same bits as
    one step() / step_adaptive() per call."""
    r = ROWS[row]
    out = []
    for call in (False, True):
        s, t_list = _solver(vo, ctx, r, lst)
        counts = _drive(s, r, call=call)
        out.append((_outputs(s, len(t_list)), [counts[k] for k in ("Step", "Chkpt", "Reject", "End")]))
    _same(out[0][0], out[1][0])
    assert out[0][1] == out[1][1]


@pytest.mark.parametrize("row", ["F2", "F3", "C2-640", "C4"])
@pytest.mark.parametrize("lst", ["L41", "EDGE"])
def test_register_path_equals_stage_path(vo, ctx, row, lst):
    """The register-resident kernels against the stage path on the same ensemble: state, snapshots, t, h, counts and dx_norm."""
    out = []
    for stage_path in (False, True):
        r = ROWS[row]
        r = r._replace(opts={**r.opts, "stage_path": stage_path})
        s, t_list = _solver(vo, ctx, r, lst)
        _drive(s, r)
        out.append(_outputs(s, len(t_list)))
    _same(out[0], out[1])


@pytest.mark.parametrize("row", ["F3", "C4"])
def test_chained_step_many_equals_unchained_calls(vo, ctx, row):
    """vo_step_many round-robins two solvers with chained launches (the lock-step snapshot copies break the chain, the per-trajectory
    kernels write snapshots themselves): the bits of one unchained call at a time."""
    r = ROWS[row]
    adaptive = r.control == "adaptive"
    ref, t_list = _solver(vo, ctx, r, "L9")
    calls = 0
    while True:
        calls += 1
        if (ref.step_adaptive() if adaptive else ref.step()).kind == "Done":
            break
    pair = [_solver(vo, ctx, r, "L9")[0] for _ in range(2)]
    vo.step_many(pair, adaptive, calls // 2)
    vo.step_many(pair, adaptive, calls - calls // 2)
    for s in pair:
        _same(_outputs(s, len(t_list)), _outputs(ref, len(t_list)))


@pytest.mark.parametrize("lst", ["L5", "L9", "L41"])
def test_user_body_and_norm(vo, ctx, lst):
    """C6: run-time compiled modules. The VdP right-hand side as a user body gives the built-in kernels' bits, one event per launch
    (the module's two-trajectory control kernel) and through run() (its CFG 1 staged kernel); the 2-norm as a user norm (CFG 0)
    gives the built-in norm's bits. The body is also checked against the pure-Python restatement driving the same closure."""
    from oracle import vecode_oracle as po
    from oracle import oracle_lib as oracle
    for row in ("C4", "C2"):
        r = ROWS[row]
        params = _inputs(vo, r)[0]
        out = []
        for rhs in (None, vo.Rhs.custom(ctx, VDP_BODY, 2, [params[:, 0].copy()])):
            s, t_list = _solver(vo, ctx, r, lst, rhs=rhs)
            _drive(s, r)
            out.append((s, _outputs(s, len(t_list))))
        _same(out[0][1], out[1][1])
    s = out[1][0]
    ac, b, be, ns = oracle.builtin_tableau(2)
    _, x0, _ = _inputs(vo, r)
    stats = s.stats()
    for i in range(0, r.n, 499):
        p = po.RKSolver(po.rhs_vdp([float(params[i, 0])]), (list(ac), list(b), list(be), ns), 0.0, t_list[-1], [float(v) for v in x0[i]], 1e-3)
        p.with_tolerance(r.rtol, r.rtol)
        p.t_list = list(t_list)
        snaps = []
        while True:
            st = p.step_adaptive()
            if p.last_event in (po.CHKPT, po.END):
                snaps.append((list(p.x), p.h))
            if st != po.OK:
                break
        assert len(snaps) == len(t_list)
        assert (stats["accepted"][i], stats["rejected"][i]) == (p.n_accept, p.n_reject), i
        for k, (xk, hk) in enumerate(snaps):
            assert _rel(s.snapshot(k).to_host()[i], np.array(xk)) <= 1e-12, (i, k)
        _h_close(stats["h"][i:i + 1], np.array([hk]), f"trajectory {i}")
    r = ROWS["C2"]
    out = []
    for norm in ("L2", vo.NormFn(ctx, "m = e * e;", "sum", "r = sqrt(acc);")):
        s, t_list = _solver(vo, ctx, r, lst)
        s.with_norm(norm)
        _drive(s, r)
        out.append(_outputs(s, len(t_list)))
    _same(out[0], out[1])


def test_fixed_steps_then_adaptive_in_mid_list(vo, ctx, oracle):
    """Fixed steps through the first two entries (lock-step), then step_adaptive() to the end: the switch to per-trajectory control
    (materialize) in the middle of the list, on the register path and on the stage path, bit for bit. Up to entry 1 the snapshots
    are the fixed-step oracle's bits."""
    r = ROWS["C4"]
    out = []
    for stage_path in (False, True):
        s, t_list = _solver(vo, ctx, r._replace(opts={"k": 1, "stage_path": stage_path}), "L9")
        chk = 0
        while chk < 2 * r.n:
            chk += s.step().counts["Chkpt"]
        while s.step_adaptive().kind != "Done":
            pass
        out.append(_outputs(s, len(t_list)))
    _same(out[0], out[1])
    params, x0, _ = _inputs(vo, r)
    for k in (0, 1):
        ref = oracle.rk_ensemble("VDP", params, oracle.builtin_tableau(2), 0.0, t_list[k], x0, 1e-3, n_threads=8, t_list=t_list[:k + 1])
        assert np.array_equal(_bits(out[0][1 + k]), _bits(ref["x"])), k


@pytest.mark.parametrize("row", ["F3", "C3-h"])
def test_fast_arithmetic_fixed_steps(vo, row):
    """FAST arithmetic, fixed steps: lock-step F3 and per-trajectory steps on the staged control kernel (N = 2500, run()): every
    snapshot within 1e-12 relative of the STRICT oracle."""
    c = vo.Context(0, arith="fast")
    r = ROWS[row]
    s, t_list = _solver(vo, c, r, "L9")
    counts = _drive(s, r)
    refs = _oracle_refs(row, "L9")
    assert counts["Chkpt"] == r.n * (len(t_list) - 1) and counts["End"] == r.n
    for k in range(len(t_list)):
        err = _rel(s.snapshot(k).to_host(), refs[k]["x"])
        assert err <= 1e-12, (k, err)
    assert np.array_equal(s.stats()["accepted"], refs[-1]["accepted"])
    c.close()


HEAT = {"H1": (4099, False), "H2": (1 << 16, False), "H3": (4099, True)}


@pytest.mark.parametrize("row,lst", [(row, lst) for row in HEAT for lst in ("L5", "L9", "L41")] + [("H1", "EDGE")])
def test_heat_single_state_fixed(vo, ctx, oracle, row, lst):
    """H1-H3: one HEAT1D state, lock-step RK4 (h = 0.25 on [0, 2], EDGE with h = 0.1) through the plain stage kernel, the TMA
    stage kernel and the whole-step kernel: snapshots bit-identical to the oracle."""
    d, fused = HEAT[row]
    u0 = vo.workloads.heat_u0(d)
    t_list = list(EDGE) if lst == "EDGE" else [2.0 * float(v) for v in LISTS[lst]]
    h = 0.1 if lst == "EDGE" else 0.25
    s = vo.RK45Solver(vo.Rhs(ctx, "HEAT1D", d, [1.0]), 0.0, t_list[-1], vo.Ensemble.from_host(ctx, u0[None, :]), h, tableau=vo.ButcherTableu.builtin("RK4"))
    s.set_t_list(t_list).enable_snapshots()
    if fused:
        s.set_fused_step()
    st = s.run()
    assert st.kind == "Done" and st.counts["Chkpt"] == len(t_list) - 1 and st.counts["End"] == 1
    otab = oracle.builtin_tableau(1)
    for k in range(len(t_list)):
        rx, ro, _ = oracle.rk_solve("HEAT1D", [1.0], otab, 0.0, t_list[k], u0, h, t_list=t_list[:k + 1])
        assert np.array_equal(_bits(s.snapshot(k).to_host()[0]), _bits(rx)), k
    assert st.counts["Step"] == ro.n_accept and s.stats()["t"][0] == ro.t


@pytest.mark.parametrize("lst", ["L5", "L9", "L41"])
def test_heat_single_state_adaptive(vo, ctx, oracle, lst):
    """H4: one HEAT1D state, adaptive DOPRI5 with the controller on the host (tree-reduced norm on the device): accepted and
    rejected counts equal to the oracle's, snapshots within 1e-12 relative and the final h as _h_close allows."""
    d = 4096
    u0 = vo.workloads.heat_u0(d)
    t_list = [2.0 * float(v) for v in LISTS[lst]]
    s = vo.RK45Solver(vo.Rhs(ctx, "HEAT1D", d, [1.0]), 0.0, 2.0, vo.Ensemble.from_host(ctx, u0[None, :]), 0.01, tableau=vo.ButcherTableu.builtin("DOPRI5"))
    s.with_tolerance(1e-6, 1e-6).with_step_range(1e-6, 0.3).with_init_step(0.01)
    s.set_t_list(t_list).enable_snapshots()
    st = s.run(adaptive=True)
    assert st.kind == "Done" and st.counts["Chkpt"] == len(t_list) - 1
    otab = oracle.builtin_tableau(2)
    for k in range(len(t_list)):
        rx, ro, _ = oracle.rk_solve("HEAT1D", [1.0], otab, 0.0, t_list[k], u0, 0.01, adaptive=True, rtol=1e-6, atol=1e-6, max_dt=0.3, t_list=t_list[:k + 1])
        assert _rel(s.snapshot(k).to_host()[0], rx) <= 1e-12, k
    stats = s.stats()
    assert (stats["accepted"][0], stats["rejected"][0]) == (ro.n_accept, ro.n_reject)
    _h_close(stats["h"][:1], np.array([ro.h]), "final h")
    assert abs(stats["t"][0] - 2.0) <= EPS


def test_t_list_checkpoints(vo, ctx):
    """The HARMONIC2D / RKF45_REF cases with their original 4-entry lists: N = 64 on the register path (rk_fixed_kernel,
    rk_ctl_kernel) and N = 96 on the stage path, fixed and adaptive (rtol 1e-7), under the bars of the oracle test."""
    for row, lst in (("F1-harmonic", "HARM_A"), ("C1-harmonic", "HARM_A"), ("F4-harmonic", "HARM_B"), ("C5-harmonic", "HARM_B")):
        r = ROWS[row]
        s, t_list = _solver(vo, ctx, r, lst)
        counts = _drive(s, r)
        _check_against_oracle(s, counts, r, t_list, _oracle_refs(row, lst))


def test_refusals(vo, ctx):
    r = ROWS["C2-640"]

    def code(f, *a):
        with pytest.raises(vo.VecOdeError) as e:
            f(*a)
        return e.value.code

    s, t_list = _solver(vo, ctx, r, "L5", snapshots=False)
    assert code(s.snapshot, 0) == vo._cabi.VO_ERR_STATE  # snapshots off
    assert code(s.set_t_list, np.linspace(0.0, 1.0, 65536)) == vo._cabi.VO_ERR_UNSUPPORTED
    assert code(s.set_t_list, []) == vo._cabi.VO_ERR_BAD_ARG
    s.enable_snapshots()
    for k in (-1, len(t_list)):
        assert code(s.snapshot, k) == vo._cabi.VO_ERR_BAD_ARG
    s.step_adaptive()
    assert code(s.set_t_list, [0.0, 1.0]) == vo._cabi.VO_ERR_STATE  # per-trajectory stepping has begun
    assert s.run(adaptive=True).kind == "Done" and np.all(np.abs(s.stats()["t"] - 1.0) <= EPS)
