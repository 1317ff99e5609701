"""Runge-Kutta stepping path on the B200 against the CPU oracle (restatement of src/base/rk.rs + src/base/ode.rs).

Bars: fixed-step = BIT-EXACT in strict mode (same operations, same order, no FMA) and <= 1e-12 relative in fast mode;
adaptive = within the requested rtol at t_end, accepted/rejected counts compared and reported (the controller's
`powf` comes from different libms on the two sides, so step sequences may differ in the last bits).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TABLEAUX = ["RKF45_REF", "RK4", "DOPRI5"]


def _case(vo, name, n, seed=0):
    """(rhs kind, d, params AoS [n][np], x0 AoS [n][d])"""
    rng = np.random.default_rng(seed)
    if name == "LORENZ63":
        return name, 3, np.tile(vo.workloads.LORENZ_PARAMS, (n, 1)), vo.workloads.lorenz_x0(n)
    if name == "VDP":
        return name, 2, vo.workloads.vdp_mu(n)[:, None], vo.workloads.vdp_x0(n) + 0.01 * rng.standard_normal((n, 2))
    if name == "HARMONIC2D":
        return name, 2, 0.5 + rng.random((n, 1)), rng.standard_normal((n, 2))
    if name.startswith("DIAG"):
        d = int(name[4:])
        return "DIAG_LINEAR", d, -rng.random((n, d)) * 2.0, rng.standard_normal((n, d))
    raise KeyError(name)


def _make_rhs(vo, ctx, kind, d, params, per_traj=True):
    rhs = vo.Rhs(ctx, kind, d)
    for q in range(params.shape[1]):
        rhs.set_param(q, params[:, q].copy() if per_traj else float(params[0, q]))
    return rhs


@pytest.mark.parametrize("tab", TABLEAUX)
@pytest.mark.parametrize("case", ["LORENZ63", "VDP", "HARMONIC2D", "DIAG1", "DIAG2", "DIAG4"])
def test_try_step_stage_kernels_bit_exact(vo, ctx, oracle, tab, case):
    """One rk_step (rk.rs:90-155) through the stage kernels: next_x, x_err and every K_i equal the oracle's bits."""
    n = 257
    kind, d, params, x0 = _case(vo, case, n, seed=3)
    tableau = vo.ButcherTableu.builtin(tab)
    otab = oracle.builtin_tableau(oracle.TABLEAU_ID[tab])
    s = tableau.num_stages()
    rhs = _make_rhs(vo, ctx, kind, d, params)
    X0 = vo.Ensemble.from_host(ctx, x0)
    solver = vo.RK45Solver(rhs, 0.0, 1.0, X0, 0.01, tableau=tableau)
    nx, xe = vo.Ensemble(ctx, d, n), vo.Ensemble(ctx, d, n)
    K = [vo.Ensemble(ctx, d, n) for _ in range(s)]
    t, dt = 0.37, 0.0123
    solver.try_step(t, dt, nx, xe if otab[2] is not None else None, K)
    got_x, got_e = nx.to_host(), xe.to_host()
    got_K = [k.to_host() for k in K]
    for i in range(n):
        rx, re, rK = oracle.rk_step(kind, params[i], otab, t, dt, x0[i])
        assert np.array_equal(got_x[i], rx), (i, got_x[i], rx)
        if re is not None:
            assert np.array_equal(got_e[i], re)
        for j in range(s):
            assert np.array_equal(got_K[j][i], rK[j])


@pytest.mark.parametrize("stage_path", [False, True])
@pytest.mark.parametrize("tab,no_adaptive", [("RK4", False), ("RKF45_REF", False), ("RKF45_REF", True), ("DOPRI5", False)])
def test_fixed_step_lorenz_bit_exact(vo, ctx, oracle, tab, no_adaptive, stage_path):
    """Config 2 at a size the oracle finishes in seconds: N = 2048 Lorenz-63 trajectories, h = 1e-3, t in [0, 0.25]."""
    n = 2048
    kind, d, params, x0 = _case(vo, "LORENZ63", n)
    tableau = vo.ButcherTableu.builtin(tab)
    otab = oracle.builtin_tableau(oracle.TABLEAU_ID[tab])
    rhs = _make_rhs(vo, ctx, kind, d, params, per_traj=False)
    solver = vo.RK45Solver(rhs, 0.0, 0.25, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=tableau)
    if no_adaptive:
        solver.no_adaptive()
    solver.set_stage_path(stage_path)
    st = solver.run()
    assert st.kind == "Done"
    ref = oracle.rk_ensemble(kind, params, otab, 0.0, 0.25, x0, 1e-3, n_threads=8, no_adaptive=no_adaptive)
    (tmin, tmax), X = solver.current()
    assert tmin == tmax == ref["t"][0]
    assert st.counts["Step"] == int(ref["accepted"].sum())
    assert np.array_equal(X.to_host(), ref["x"])
    stats = solver.stats()
    assert np.array_equal(stats["accepted"], ref["accepted"])


def test_fixed_step_events_per_launch_and_step_calls(vo, ctx, oracle):
    """k events fused per launch give the same bits as k separate step() calls; the first call is a Chkpt (ode.rs:144-145)."""
    n = 1000
    kind, d, params, x0 = _case(vo, "LORENZ63", n)
    tableau = vo.ButcherTableu.builtin("RK4")
    rhs = _make_rhs(vo, ctx, kind, d, params, per_traj=False)
    a = vo.RK45Solver(rhs, 0.0, 0.05, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=tableau)
    first = a.step()
    assert first.kind == "Ok" and first.counts["Chkpt"] == n and first.counts["Step"] == 0
    calls = 1
    while a.step().is_ok:
        calls += 1
    b = vo.RK45Solver(rhs, 0.0, 0.05, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=tableau).set_events_per_launch(7)
    st = b.run()
    assert st.kind == "Done" and st.counts["Chkpt"] == n and st.counts["End"] == n
    assert np.array_equal(a.current()[1].to_host(), b.current()[1].to_host())
    ref = oracle.rk_ensemble(kind, params, oracle.builtin_tableau(1), 0.0, 0.05, x0, 1e-3, n_threads=4)
    assert np.array_equal(b.current()[1].to_host(), ref["x"])
    assert st.counts["Step"] == int(ref["accepted"].sum())
    assert calls + 1 == int(ref["accepted"][0]) + 2  # accepted + Chkpt + End


def test_reference_own_tests_golden(vo, ctx, oracle):
    """The reference's three smoke tests (src/impls/nalgebra.rs:52-107) as fixed by the oracle (SURVEY.md §4 table)."""
    import json, os
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "rk_known_answers.json")))
    # test_rk45_2: y' = (-y0, -2 y1), [0,2], h = 1e-4, step(), default constructor
    case = g["test_rk45_2"]
    rhs = vo.Rhs(ctx, "DIAG_LINEAR", 2, [-1.0, -2.0])
    s = vo.RK45Solver(rhs, 0.0, 2.0, vo.Ensemble.from_host(ctx, [[1.0, 1.0]]), 1e-4)
    st = s.run()
    assert st.counts["Step"] == case["accepted"]
    assert s.current()[1].to_host()[0].tolist() == case["x"]
    # same with .no_adaptive() (propagates X_b and shows the 2526 typo)
    case = g["test_rk45_2_no_adaptive"]
    s = vo.RK45Solver(rhs, 0.0, 2.0, vo.Ensemble.from_host(ctx, [[1.0, 1.0]]), 1e-4).no_adaptive()
    s.run()
    assert s.current()[1].to_host()[0].tolist() == case["x"]
    # test_rk45_1: complex Vector2 -> 4 real components, params (-1,-1,-2,-2)
    case = g["test_rk45_1_complex"]
    rhs4 = vo.Rhs(ctx, "DIAG_LINEAR", 4, [-1.0, -1.0, -2.0, -2.0])
    s = vo.RK45Solver(rhs4, 0.0, 2.0, vo.Ensemble.from_host(ctx, [[1.0, 0.0, 1.0, 0.0]]), 1e-4)
    s.run()
    got = s.current()[1].to_host()[0]
    assert np.array_equal(got, np.array(case["x"]))  # signed zeros compare equal
    # test_rk45_f64: scalar, with_tolerance(1e-10, 1e-10), step_adaptive()
    case = g["test_rk45_f64"]
    rhs1 = vo.Rhs(ctx, "DIAG_LINEAR", 1, [-1.0])
    s = vo.RK45Solver(rhs1, 0.0, 2.0, vo.Ensemble.from_host(ctx, [[1.0]]), 1e-4).with_tolerance(1e-10, 1e-10)
    st = s.run(adaptive=True)
    stats = s.stats()
    x = s.current()[1].to_host()[0, 0]
    assert abs(x - case["x"][0]) <= 1e-10
    assert abs(int(stats["accepted"][0]) - case["accepted"]) <= 4 and int(stats["rejected"][0]) == case["rejected"]


@pytest.mark.parametrize("rtol", [1e-6, 1e-8, 1e-10])
def test_config1_harmonic_adaptive(vo, ctx, oracle, rtol):
    """Config 1: adaptive RK45 (the reference's literal tableau) on x' = (v, -x), single trajectory."""
    otab = oracle.builtin_tableau(0)
    rx, ro, _ = oracle.rk_solve("HARMONIC2D", [1.0], otab, 0.0, 10.0, [1.0, 0.0], 1e-3, adaptive=True, rtol=rtol, atol=rtol)
    rhs = vo.Rhs(ctx, "HARMONIC2D", 2, [1.0])
    s = vo.RK45Solver(rhs, 0.0, 10.0, vo.Ensemble.from_host(ctx, [[1.0, 0.0]]), 1e-3).with_tolerance(rtol, rtol)
    st = s.run(adaptive=True)
    assert st.kind == "Done"
    x = s.current()[1].to_host()[0]
    stats = s.stats()
    print(f"rtol={rtol}: gpu accepted/rejected {stats['accepted'][0]}/{stats['rejected'][0]}  oracle {ro.n_accept}/{ro.n_reject}")
    assert abs(stats["t"][0] - 10.0) <= 1e-14 and abs(ro.t - 10.0) <= 1e-14
    # absolute-error controller (ode.rs:320): per-step error <= rtol; global error grows with the step count
    assert np.max(np.abs(x - rx)) <= rtol * 10
    assert abs(int(stats["accepted"][0]) - ro.n_accept) <= max(2, ro.n_accept // 500)


@pytest.mark.parametrize("tab", ["DOPRI5", "RKF45_REF"])
@pytest.mark.parametrize("stage_path", [False, True])
def test_config3_vdp_adaptive_ensemble(vo, ctx, oracle, tab, stage_path):
    """Config 3 at oracle size: N = 512 Van der Pol oscillators, mu sweep, per-trajectory step control on the device."""
    n, rtol, tf = 512, 1e-6, 20.0
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n)
    tableau = vo.ButcherTableu.builtin(tab)
    otab = oracle.builtin_tableau(oracle.TABLEAU_ID[tab])
    ref = oracle.rk_ensemble("VDP", mu[:, None], otab, 0.0, tf, x0, 1e-3, n_threads=8, adaptive=True, rtol=rtol, atol=rtol)
    rhs = vo.Rhs(ctx, "VDP", 2, [mu])
    s = vo.RK45Solver(rhs, 0.0, tf, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=tableau).with_tolerance(rtol, rtol)
    s.set_stage_path(stage_path)
    st = s.run(adaptive=True)
    assert st.kind == "Done" and st.counts["End"] == n
    x = s.current()[1].to_host()
    stats = s.stats()
    assert np.all(np.abs(stats["t"] - tf) <= 1e-13) and np.all(stats["status"] == 1)
    acc_g, acc_r = stats["accepted"].sum(), ref["accepted"].sum()
    rej_g, rej_r = stats["rejected"].sum(), ref["rejected"].sum()
    print(f"{tab} stage_path={stage_path}: accepted gpu/oracle {acc_g}/{acc_r}, rejected {rej_g}/{rej_r}, launches {st.counts['launches']}")
    assert st.counts["Step"] == acc_g and st.counts["Reject"] == rej_g
    assert abs(acc_g - acc_r) <= 0.01 * acc_r and abs(rej_g - rej_r) <= 0.02 * rej_r + 8
    # stiff-ish limit cycle: errors of a few hundred steps of size <= rtol each, amplified along the fast branches
    err = np.abs(x - ref["x"]).max(axis=1)
    assert np.quantile(err, 0.99) <= 200 * rtol, np.quantile(err, [0.5, 0.9, 0.99, 1.0])


@pytest.mark.parametrize("n,k_small", [(300, 5), (2500, 1), (2500, 5), (2500, 0)])
def test_small_and_stage_paths_agree_bitwise_adaptive(vo, ctx, n, k_small):
    """Same device libm on both paths, so the register-resident and the stage-granular kernels must agree bit for bit,
    step sequence included. n = 300 runs the one-trajectory-per-thread control kernel, n = 2500 the two-per-thread one
    (with a ragged tail of 2500 % 256 trajectories): one event per launch, five (the joint multi-event loop) and the
    automatic eight of vo_run."""
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n)
    out = []
    for stage_path in (False, True):
        rhs = vo.Rhs(ctx, "VDP", 2, [mu])
        s = vo.RK45Solver(rhs, 0.0, 5.0, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5"))
        s.with_tolerance(1e-6, 1e-6).set_stage_path(stage_path).set_events_per_launch(1 if stage_path else k_small)
        s.run(adaptive=True)
        out.append((s.current()[1].to_host(), s.stats()))
    assert np.array_equal(out[0][0], out[1][0])
    for k in ("accepted", "rejected", "t", "h", "dx_norm"):
        assert np.array_equal(out[0][1][k], out[1][1][k]), k


def test_fast_mode_within_1e12(vo, oracle):
    """FMA-contracted arithmetic with zero coefficients skipped: <= 1e-12 relative to the strict/oracle result."""
    n = 4096
    kind, d, params, x0 = _case(vo, "LORENZ63", n)
    ref = oracle.rk_ensemble(kind, params, oracle.builtin_tableau(1), 0.0, 0.25, x0, 1e-3, n_threads=8)
    c = vo.Context(0, arith="fast")
    rhs = _make_rhs(vo, c, kind, d, params, per_traj=False)
    s = vo.RK45Solver(rhs, 0.0, 0.25, vo.Ensemble.from_host(c, x0), 1e-3, tableau=vo.ButcherTableu.builtin("RK4"))
    s.run()
    x = s.current()[1].to_host()
    rel = np.abs(x - ref["x"]).max() / np.abs(ref["x"]).max()
    print("fast-mode max relative deviation:", rel)
    assert rel <= 1e-12


@pytest.mark.parametrize("d", [3, 1024, 1025, 4099, 1 << 16])
@pytest.mark.parametrize("tab", ["RK4", "RKF45_REF"])
def test_heat_stage_path_bit_exact(vo, ctx, oracle, d, tab):
    """Config 4 at oracle size: periodic 1-D heat equation, stage kernels with the stencil fused, ragged tile tails."""
    u0 = vo.workloads.heat_u0(d)
    otab = oracle.builtin_tableau(oracle.TABLEAU_ID[tab])
    steps = 6
    rx, ro, _ = oracle.rk_solve("HEAT1D", [1.0], otab, 0.0, 0.25 * steps, u0, 0.25)
    rhs = vo.Rhs(ctx, "HEAT1D", d, [1.0])
    s = vo.RK45Solver(rhs, 0.0, 0.25 * steps, vo.Ensemble.from_host(ctx, u0[None, :]), 0.25, tableau=vo.ButcherTableu.builtin(tab))
    st = s.run()
    assert st.kind == "Done" and st.counts["Step"] == ro.n_accept
    assert np.array_equal(s.current()[1].to_host()[0], rx)


def test_heat_adaptive_single_state(vo, ctx, oracle):
    """Large-state adaptive stepping: tree-reduced norm on the device, controller on the host (same libm as the oracle)."""
    d = 4096
    u0 = vo.workloads.heat_u0(d)
    otab = oracle.builtin_tableau(0)
    rx, ro, _ = oracle.rk_solve("HEAT1D", [1.0], otab, 0.0, 2.0, u0, 0.01, adaptive=True, rtol=1e-6, max_dt=0.3)
    rhs = vo.Rhs(ctx, "HEAT1D", d, [1.0])
    s = vo.RK45Solver(rhs, 0.0, 2.0, vo.Ensemble.from_host(ctx, u0[None, :]), 0.01).with_tolerance(1e-6, 1e-6)
    s.with_step_range(1e-6, 0.3).with_init_step(0.01)
    s.run(adaptive=True)
    stats = s.stats()
    print("heat adaptive accepted/rejected", stats["accepted"][0], stats["rejected"][0], "oracle", ro.n_accept, ro.n_reject)
    np.testing.assert_allclose(s.current()[1].to_host()[0], rx, atol=1e-6)
    assert abs(int(stats["accepted"][0]) - ro.n_accept) <= 3


def test_heat_ensemble_kernel(vo, ctx, oracle):
    n, d = 5, 96
    rng = np.random.default_rng(1)
    x0 = rng.standard_normal((n, d))
    otab = oracle.builtin_tableau(1)
    rhs = vo.Rhs(ctx, "HEAT1D", d, [0.7])
    s = vo.RK45Solver(rhs, 0.0, 0.5, vo.Ensemble.from_host(ctx, x0), 0.1, tableau=vo.ButcherTableu.builtin("RK4"))
    s.run()
    got = s.current()[1].to_host()
    for i in range(n):
        rx, _, _ = oracle.rk_solve("HEAT1D", [0.7], otab, 0.0, 0.5, x0[i], 0.1)
        assert np.array_equal(got[i], rx)


def test_per_trajectory_initial_step(vo, ctx, oracle):
    n = 128
    kind, d, params, x0 = _case(vo, "HARMONIC2D", n, seed=9)
    h0 = np.linspace(1e-3, 2e-2, n)
    otab = oracle.builtin_tableau(2)
    ref = oracle.rk_ensemble(kind, params, otab, 0.0, 1.0, x0, 0.0, h0_arr=h0, n_threads=2)
    rhs = _make_rhs(vo, ctx, kind, d, params)
    s = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5")).set_h_array(h0)
    st = s.run()
    assert st.kind == "Done"
    assert np.array_equal(s.current()[1].to_host(), ref["x"])
    assert np.array_equal(s.stats()["accepted"], ref["accepted"])


def test_error_behaviour(vo, ctx):
    rhs = vo.Rhs(ctx, "HARMONIC2D", 2)
    x0 = vo.Ensemble.from_host(ctx, [[1.0, 0.0]])
    s = vo.RK45Solver(rhs, 0.0, 1.0, x0, 1e-2)
    with pytest.raises(vo.VecOdeError) as e:
        s.with_tolerance(-1.0, 1e-3)  # ode.rs:299-301 panics
    assert "Invalid tolerances" in e.value.msg
    with pytest.raises(vo.VecOdeError) as e:
        s.with_step_range(1.0, 0.5)  # ode.rs:268-270
    assert "Invalid step range" in e.value.msg
    with pytest.raises(vo.VecOdeError):
        s.with_init_step(5.0)  # ode.rs:288-291: outside (min_dt, max_dt)
    s.no_adaptive()
    with pytest.raises(vo.VecOdeError) as e:
        s.step_adaptive()  # ode.rs:312 `.expect("adaptive step validation failed")`
    assert e.value.code == vo._cabi.VO_ERR_NOT_ADAPTIVE
    with pytest.raises(vo.VecOdeError):
        vo.RK45Solver(vo.Rhs(ctx, "LORENZ63", 3), 0.0, 1.0, x0, 1e-2)  # dimension mismatch
    with pytest.raises(vo.VecOdeError):
        vo.ButcherTableu.from_slices([0.0] * 4, [1.0], None, 2)


def test_with_step_range_sets_geometric_mean(vo, ctx, oracle):
    """with_step_range resets h to sqrt(min*max) (ode.rs:273-280)."""
    rhs = vo.Rhs(ctx, "DIAG_LINEAR", 1, [-1.0])
    s = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(ctx, [[1.0]]), 1e-4).with_step_range(1e-4, 1e-2)
    assert s.stats()["h"][0] == np.sqrt(1e-4 * 1e-2)


def test_nonfinite_and_stuck_flags(vo, ctx):
    """NaN error norms are accepted like the reference (ode.rs:321-330) but flagged; a trajectory rejected at min_dt is
    flagged STUCK and vo_run returns instead of spinning forever."""
    rhs = vo.Rhs(ctx, "DIAG_LINEAR", 1, [-1.0])
    s = vo.RK45Solver(rhs, 0.0, 0.01, vo.Ensemble.from_host(ctx, [[np.nan]]), 1e-2).set_events_per_launch(1000)
    st = s.run(adaptive=True)
    assert st.kind == "Done" and s.stats()["status"][0] & vo._cabi.TRAJ_NONFINITE
    # huge decay rate, rtol tiny, min_dt == max reachable: every attempt is rejected at h == min_dt
    rhs = vo.Rhs(ctx, "DIAG_LINEAR", 1, [-1.0e9])
    s = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(ctx, [[1.0]]), 1e-3).with_tolerance(1e-30, 1e-30)
    with pytest.raises(vo.VecOdeError):
        s.run(adaptive=True)
    assert s.stats()["status"][0] & vo._cabi.TRAJ_STUCK


def test_full_size_properties_lorenz(vo, ctx):
    """Config 2 at full size (N = 1e6): size-independent properties instead of an oracle run —
    (i) permutation equivariance: shuffled trajectories give shuffled results, bit for bit;
    (ii) splitting the ensemble into two shards (the multi-GPU decomposition) gives the same bits;
    (iii) a 2048-trajectory prefix equals the standalone 2048-trajectory run (which the oracle test covers)."""
    n = 1_000_000
    x0 = vo.workloads.lorenz_x0(n)
    tableau = vo.ButcherTableu.builtin("RK4")

    def run(x):
        rhs = vo.Rhs(ctx, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
        s = vo.RK45Solver(rhs, 0.0, 0.1, vo.Ensemble.from_host(ctx, x), 1e-3, tableau=tableau)
        st = s.run()
        assert st.kind == "Done"
        return s.current()[1].to_host()

    full = run(x0)
    assert np.all(np.isfinite(full))
    perm = np.random.default_rng(0).permutation(n)
    assert np.array_equal(run(x0[perm]), full[perm])
    half = n // 2
    assert np.array_equal(np.concatenate([run(x0[:half]), run(x0[half:])]), full)
    assert np.array_equal(run(x0[:2048]), full[:2048])


def test_step_many_and_chained_launches_bit_exact(vo, ctx, oracle):
    """vo_step_many round-robins several ensembles with no read-back; from the second round on every launch is CHAINED
    (CTA b waits only for CTA b of the solver's previous launch, not for the whole grid). Results must equal the oracle
    bit for bit — a missed dependency would show up as a torn state."""
    n, rounds = 20000, 40
    params = np.tile(vo.workloads.LORENZ_PARAMS, (n, 1))
    tableau = vo.ButcherTableu.builtin("RK4")
    rhs = vo.Rhs(ctx, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
    x0s = [vo.workloads.lorenz_x0(n, first=q * n) for q in range(3)]
    solvers = [vo.RK45Solver(rhs, 0.0, 1.0e9, vo.Ensemble.from_host(ctx, x), 1e-3, tableau=tableau) for x in x0s]
    vo.step_many(solvers, False, 1)        # the Chkpt at t0
    vo.step_many(solvers, False, rounds)   # `rounds` steps each, interleaved
    for x, s in zip(x0s, solvers):
        ref = oracle.rk_ensemble("LORENZ63", params, oracle.builtin_tableau(1), 0.0, 1.0e9, x, 1e-3, n_threads=8, max_calls=rounds + 1)
        assert np.array_equal(s.current()[1].to_host(), ref["x"])
        assert s.stats()["accepted"][0] == rounds
    # adaptive ensembles through the same entry point
    mu = vo.workloads.vdp_mu(n)
    rhs2 = vo.Rhs(ctx, "VDP", 2, [mu])
    a = [vo.RK45Solver(rhs2, 0.0, 1.0e9, vo.Ensemble.from_host(ctx, vo.workloads.vdp_x0(n)), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5"))
         .with_tolerance(1e-6, 1e-6) for _ in range(2)]
    vo.step_many(a, True, 31)
    b = vo.RK45Solver(rhs2, 0.0, 1.0e9, vo.Ensemble.from_host(ctx, vo.workloads.vdp_x0(n)), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5"))
    b.with_tolerance(1e-6, 1e-6)
    for _ in range(31):
        b.step_adaptive()              # one unchained launch per call
    for s in a:
        assert np.array_equal(s.current()[1].to_host(), b.current()[1].to_host())
        for k in ("accepted", "rejected", "t", "h"):
            assert np.array_equal(s.stats()[k], b.stats()[k]), k


def test_fast_mode_full_config2_within_1e12(vo, oracle):
    """Config 2's whole interval t in [0,1] (1000 steps + remainder) in FMA arithmetic: <= 1e-12 relative (north_star)."""
    n = 2048
    x0 = vo.workloads.lorenz_x0(n)
    params = np.tile(vo.workloads.LORENZ_PARAMS, (n, 1))
    ref = oracle.rk_ensemble("LORENZ63", params, oracle.builtin_tableau(1), 0.0, 1.0, x0, 1e-3, n_threads=8)
    c = vo.Context(0, arith="fast")
    rhs = vo.Rhs(c, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
    s = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(c, x0), 1e-3, tableau=vo.ButcherTableu.builtin("RK4"))
    st = s.run()
    assert st.counts["Step"] == int(ref["accepted"].sum())
    x = s.current()[1].to_host()
    rel = np.abs(x - ref["x"]).max() / np.abs(ref["x"]).max()
    print("fast-mode max relative deviation at t = 1:", rel)
    assert rel <= 1e-12


def test_full_size_properties_vdp_adaptive(vo, ctx, oracle):
    """Config 3 at full size (N = 1e6, t in [0, 20], per-trajectory control): size-independent properties —
    (i) every trajectory reaches t_end and is flagged done, none stuck / non-finite; (ii) the ensemble split into two
    shards (the multi-GPU decomposition, mu indexed by global trajectory number) gives the same bits; (iii) a strided
    sample of 256 trajectories agrees with the oracle within rtol-scale error and its step counts within 1 %."""
    n, tf, rtol = 1_000_000, 20.0, 1e-6
    mu = vo.workloads.vdp_mu(n)
    tableau = vo.ButcherTableu.builtin("DOPRI5")

    def run(mu_part):
        rhs = vo.Rhs(ctx, "VDP", 2, [mu_part])
        s = vo.RK45Solver(rhs, 0.0, tf, vo.Ensemble.from_host(ctx, vo.workloads.vdp_x0(len(mu_part))), 1e-3, tableau=tableau).with_tolerance(rtol, rtol)
        st = s.run(adaptive=True)
        assert st.kind == "Done" and st.counts["End"] == len(mu_part)
        return s.current()[1].to_host(), s.stats()

    x, stats = run(mu)
    assert np.all(stats["status"] == vo._cabi.TRAJ_DONE) and np.all(np.abs(stats["t"] - tf) <= 1e-12) and np.all(np.isfinite(x))
    half = 499_968  # not a multiple of the tile sizes
    xa, sa = run(mu[:half])
    xb, sb = run(mu[half:])
    assert np.array_equal(np.concatenate([xa, xb]), x)
    assert np.array_equal(np.concatenate([sa["accepted"], sb["accepted"]]), stats["accepted"])
    idx = np.arange(0, n, n // 256)[:256]
    ref = oracle.rk_ensemble("VDP", mu[idx, None], oracle.builtin_tableau(2), 0.0, tf, vo.workloads.vdp_x0(len(idx)), 1e-3, n_threads=8, adaptive=True,
                             rtol=rtol)
    assert np.quantile(np.abs(x[idx] - ref["x"]).max(axis=1), 0.99) <= 200 * rtol
    assert abs(int(stats["accepted"][idx].sum()) - int(ref["accepted"].sum())) <= 0.01 * ref["accepted"].sum()
    print("config 3 full size: attempts", int(stats["accepted"].sum() + stats["rejected"].sum()), "rejected fraction",
          float(stats["rejected"].sum() / (stats["accepted"].sum() + stats["rejected"].sum())))


def test_full_size_properties_heat(vo, ctx):
    """Config 4 at full size (d = 2^26): (i) the periodic stencil conserves the sum of u to rounding; (ii) linearity:
    solve(a*u0) == a*solve(u0) bit for bit when a is a power of two; (iii) the two analytic modes of u0 decay by the RK4
    amplification factor R(h*lambda_k) per step."""
    d, steps, h = 1 << 26, 8, 0.25
    u0 = vo.workloads.heat_u0(d)

    def run(u):
        rhs = vo.Rhs(ctx, "HEAT1D", d, [1.0])
        s = vo.RK45Solver(rhs, 0.0, h * steps, vo.Ensemble.from_host(ctx, u[None, :]), h, tableau=vo.ButcherTableu.builtin("RK4"))
        assert s.run().kind == "Done"
        return s.current()[1].to_host()[0]

    u = run(u0)
    assert abs(u.sum() - u0.sum()) <= 1e-6
    assert np.array_equal(run(4.0 * u0), 4.0 * u)
    j = np.arange(d, dtype=np.float64)
    expect = np.zeros(d)
    for kmode, amp in ((1, 1.0), (7, 0.5)):
        z = h * (2.0 * np.cos(2.0 * np.pi * kmode / d) - 2.0)
        R = 1.0 + z + z * z / 2.0 + z ** 3 / 6.0 + z ** 4 / 24.0
        expect += amp * (R ** steps) * np.sin(2.0 * np.pi * kmode * j / d)
    assert np.abs(u - expect).max() <= 1e-12


@pytest.mark.parametrize("n", [4096, 512])  # two-trajectory kernel / one-trajectory staged kernel
def test_fast_controller_agrees_with_reference_chain_within_ulps(vo, n):
    """FAST arithmetic evaluates handle_step_adaptive (ode.rs:311-334) as clamp(alpha * g^(-1/6)) with g = (dx_norm/rtol)^2
    instead of sqrt -> div -> powf. Feed both modes a bit-identical error estimate and compare the controller alone: a
    constant derivative dx = p, x0 = 0 and weights b = e_0, b_err = 0 make x_err = p*dt with one rounding in either mode."""
    s_ = 4
    ac = np.zeros((s_, s_))
    for i in range(1, s_):
        ac[i, i], ac[i, i - 1] = 0.5, 0.5
    tab = lambda: vo.ButcherTableu.from_slices(ac.ravel(), [1.0, 0, 0, 0], [0.0, 0, 0, 0], s_)
    rtol, h0 = 1e-6, 1e-3
    p = np.concatenate([10.0 ** np.linspace(-9.0, 3.0, n - 8), [0.0, 1e-200, 1e-14, 1e14, 1e160, 1e300, np.nan, rtol / h0]])
    out = {}
    for arith in ("strict", "fast"):
        c = vo.Context(0, arith=arith)
        rhs = vo.Rhs.custom(c, "dx[0] = p[0];", 1, [p])
        s = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(c, np.zeros((n, 1))), h0, tableau=tab()).with_tolerance(rtol, rtol)
        s.step_adaptive()  # Chkpt at t0
        s.step_adaptive()  # one attempt per trajectory
        out[arith] = s.stats()
        c.close()
    a, b = out["strict"], out["fast"]
    fin = np.isfinite(p) & (p < 1e150)
    ulp = np.abs(a["h"] - b["h"]) / np.spacing(np.abs(a["h"]))
    print("controller: max ulp distance of new h", ulp[fin].max(), "of dx_norm", (np.abs(a["dx_norm"] - b["dx_norm"]) / np.spacing(a["dx_norm"]))[fin & (p > 0)].max())
    assert ulp[fin].max() <= 8
    assert np.array_equal(a["h"][~fin], b["h"][~fin])  # clamped to 0.3 h either way (inf and NaN norms)
    f = rtol / (p * h0)
    sure = fin & (np.abs(f - 1.0) > 1e-12)
    assert np.array_equal(a["rejected"][sure], b["rejected"][sure]) and np.array_equal(a["accepted"][sure], b["accepted"][sure])
    nz = fin & (p > 1e-150)
    assert np.all(np.abs(a["dx_norm"][nz] - b["dx_norm"][nz]) <= 8 * np.spacing(a["dx_norm"][nz]))
    assert b["dx_norm"][p == 0.0][0] == 0.0 and np.isnan(b["dx_norm"][np.isnan(p)][0]) and np.isinf(b["dx_norm"][p == 1e300][0])
    assert (a["status"] == b["status"]).all()
    # STRICT against the reference's chain on the host C library (Rust's f64::powf is libm's pow): sqrt and the division are
    # IEEE-exact on both sides; pow(f, 1/3) is computed correctly rounded on the device, which glibc's pow also is except for
    # about one argument in a thousand
    import math
    ok = np.flatnonzero(fin & (p > 1e-150))
    h_ref, dxn_ref = np.zeros(len(ok)), np.zeros(len(ok))
    for k, i in enumerate(ok):
        e = p[i] * h0
        dxn_ref[k] = math.sqrt(e * e)
        f = rtol / dxn_ref[k]
        h_ref[k] = min(max(min(max(0.9 * math.pow(f, 1.0 / 3.0), 0.3), 2.0) * h0, 1e-6), 1.0)
    same = float(np.mean(h_ref == a["h"][ok]))
    print(f"strict controller: new h bit-identical to the libm chain on {same:.5f} of {len(ok)} inputs")
    assert np.array_equal(dxn_ref, a["dx_norm"][ok]) and same >= 0.995
    assert np.abs(h_ref - a["h"][ok]).max() <= 2 * np.spacing(h_ref).max()


def test_fast_mode_adaptive_config3_within_rtol(vo, oracle):
    """Config 3 in FAST arithmetic (FMA, lean controller): within the requested tolerance of the oracle at t_end, and
    the step sequences stay together (the controller differs from the reference chain by ulps only)."""
    n, rtol, tf = 2048, 1e-6, 20.0
    mu, x0 = vo.workloads.vdp_mu(n), vo.workloads.vdp_x0(n)
    ref = oracle.rk_ensemble("VDP", mu[:, None], oracle.builtin_tableau(2), 0.0, tf, x0, 1e-3, n_threads=8, adaptive=True, rtol=rtol, atol=rtol)
    c = vo.Context(0, arith="fast")
    s = vo.RK45Solver(vo.Rhs(c, "VDP", 2, [mu]), 0.0, tf, vo.Ensemble.from_host(c, x0), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5"))
    s.with_tolerance(rtol, rtol).set_events_per_launch(1)
    assert s.run(adaptive=True).kind == "Done"
    x, st = s.current()[1].to_host(), s.stats()
    same = np.mean((st["accepted"] == ref["accepted"]) & (st["rejected"] == ref["rejected"]))
    err = np.abs(x - ref["x"]).max(axis=1)
    print(f"fast adaptive: identical (accepted, rejected) on {same:.3f} of trajectories; accepted {st['accepted'].sum()}/{ref['accepted'].sum()}, "
          f"err quantiles {np.quantile(err, [0.5, 0.99, 1.0])}")
    assert abs(int(st["accepted"].sum()) - int(ref["accepted"].sum())) <= 0.01 * ref["accepted"].sum()
    assert np.quantile(err, 0.99) <= 200 * rtol and same >= 0.5
    c.close()


@pytest.mark.parametrize("d", [2048, 4099, (1 << 18) + 3])
@pytest.mark.parametrize("tab", ["RK4", "RKF45_REF", "DOPRI5"])
def test_heat_whole_step_kernel_bit_exact(vo, ctx, oracle, d, tab):
    """All stages of a step in one kernel (rk_heat_fused.cuh): same per-point operations in the same order as the stage
    path, so STRICT results are bit-identical to the oracle (fixed step, with and without the error estimate)."""
    u0 = vo.workloads.heat_u0(d)
    otab = oracle.builtin_tableau(oracle.TABLEAU_ID[tab])
    n_steps = 6
    rx, _, _ = oracle.rk_solve("HEAT1D", [1.0], otab, 0.0, 1.0e9, u0, 0.2, max_calls=n_steps + 1)
    s = vo.RK45Solver(vo.Rhs(ctx, "HEAT1D", d, [1.0]), 0.0, 1.0e9, vo.Ensemble.from_host(ctx, u0[None, :]), 0.2, tableau=vo.ButcherTableu.builtin(tab))
    s.set_fused_step()
    launches = 0
    for _ in range(n_steps + 1):
        launches += s.step().counts["launches"]
    assert launches == n_steps  # one kernel per step
    assert np.array_equal(s.current()[1].to_host()[0], rx)


def test_heat_whole_step_kernel_adaptive_and_fast(vo, ctx, oracle):
    d = 1 << 16
    u0 = vo.workloads.heat_u0(d)
    out = []
    for fused in (False, True):  # adaptive single state: x_err from the whole-step kernel feeds the same host controller
        s = vo.RK45Solver(vo.Rhs(ctx, "HEAT1D", d, [1.0]), 0.0, 2.0, vo.Ensemble.from_host(ctx, u0[None, :]), 0.01).with_tolerance(1e-6, 1e-6)
        s.with_step_range(1e-6, 0.3).with_init_step(0.01)
        if fused:
            s.set_fused_step()
        s.run(adaptive=True)
        out.append((s.current()[1].to_host()[0], s.stats()))
    assert np.array_equal(out[0][0], out[1][0])
    for k in ("accepted", "rejected", "t", "h", "dx_norm"):
        assert np.array_equal(out[0][1][k], out[1][1][k]), k
    cf = vo.Context(0, arith="fast")
    s = vo.RK45Solver(vo.Rhs(cf, "HEAT1D", d, [1.0]), 0.0, 1.0, vo.Ensemble.from_host(cf, u0[None, :]), 0.2, tableau=vo.ButcherTableu.builtin("RK4"))
    s.no_adaptive().set_fused_step()
    s.run()
    rx, _, _ = oracle.rk_solve("HEAT1D", [1.0], oracle.builtin_tableau(1), 0.0, 1.0, u0, 0.2, no_adaptive=True)
    assert np.abs(s.current()[1].to_host()[0] - rx).max() <= 1e-12 * np.abs(rx).max()
    with pytest.raises(vo.VecOdeError):
        vo.RK45Solver(vo.Rhs(ctx, "LORENZ63", 3), 0.0, 1.0, vo.Ensemble.from_host(ctx, vo.workloads.lorenz_x0(8)), 0.1).set_fused_step()
    cf.close()


# ---- round 2: chains that survive API calls, kernels that must not chain, the bench's kernels against the oracle ----------
def test_chain_survives_api_calls_bit_exact(vo, ctx, oracle):
    """The reference's driver loop `while let Ok(_) = solver.step() {}` (src/impls/nalgebra.rs:62): one launch per call. The
    CTA chain now stays alive from call to call (nothing else is enqueued on the ctx in between), so every launch after the
    first skips the grid-wide wait. Library calls that touch the state (here an in-place scale by 1.0 of the borrowed
    ensemble) and vo_ctx_fence break the chain for one launch. Bits must be the oracle's throughout."""
    n, calls = 20000, 160
    params = np.tile(vo.workloads.LORENZ_PARAMS, (n, 1))
    x0 = vo.workloads.lorenz_x0(n)
    rhs = vo.Rhs(ctx, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
    s = vo.RK45Solver(rhs, 0.0, 1.0e9, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin("RK4"))
    other = vo.RK45Solver(rhs, 0.0, 1.0e9, vo.Ensemble.from_host(ctx, x0[::-1].copy()), 1e-3, tableau=vo.ButcherTableu.builtin("RK4"))
    for k in range(calls + 1):  # the first call is the Chkpt at t0
        st = s.step()
        assert st.kind == "Ok"
        other.step()  # a second solver interleaved on the same ctx: its launches touch only its own state
        if k == 40:
            vo.LinearCombination.scale(s.current()[1], 1.0)  # library op on the solver's state: chain broken for one launch
        if k == 80:
            ctx.fence()
        if k == 120:
            ctx.sync()
    ref = oracle.rk_ensemble("LORENZ63", params, oracle.builtin_tableau(1), 0.0, 1.0e9, x0, 1e-3, n_threads=8, max_calls=calls + 1)
    assert np.array_equal(s.current()[1].to_host(), ref["x"])
    ref2 = oracle.rk_ensemble("LORENZ63", params, oracle.builtin_tableau(1), 0.0, 1.0e9, x0[::-1].copy(), 1e-3, n_threads=8, max_calls=calls + 1)
    assert np.array_equal(other.current()[1].to_host(), ref2["x"])


@pytest.mark.parametrize("max_calls", [9, 17, 41, 8 * 30 + 3])
def test_run_tail_launch_on_another_kernel_is_not_chained(vo, ctx, max_calls):
    """vo_run fuses 8 events per launch (one-trajectory kernel, 128-trajectory tiles) and ends a budget of 8 m + r calls with
    a launch of r events; r = 1 selects the two-trajectory kernel (256-trajectory tiles, another grid): that launch must not
    be chained to its predecessor, whose CTA b owned other trajectories. The stage path (no chaining at all) is the check."""
    n = 6144
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n)
    out = []
    for stage_path in (False, True):
        rhs = vo.Rhs(ctx, "VDP", 2, [mu])
        s = vo.RK45Solver(rhs, 0.0, 50.0, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5"))
        s.with_tolerance(1e-6, 1e-6).set_stage_path(stage_path)
        s.run(adaptive=True, max_calls=max_calls)
        s.run(adaptive=True, max_calls=max_calls)  # and again: 8-event launches follow the 1-event one
        out.append((s.current()[1].to_host(), s.stats()))
    assert np.array_equal(out[0][0], out[1][0])
    for k in ("accepted", "rejected", "t", "h", "dx_norm"):
        assert np.array_equal(out[0][1][k], out[1][1][k]), k
    assert int(out[0][1]["accepted"].sum() + out[0][1]["rejected"].sum()) == n * (2 * max_calls - 1)  # all but the Chkpt call


@pytest.mark.parametrize("prev_h", ["lazy", "every_attempt"])
@pytest.mark.parametrize("tab", ["DOPRI5", "RKF45_REF"])
def test_strict_one_event_control_kernel_against_oracle(vo, ctx, oracle, tab, prev_h):
    """The kernel bench.py times for config 3 — rk_ctl2w_staged_kernel<.., STRICT>, ONE event per launch, N >= 1024, with the
    lazy prev_h store and with mixed stepping (prev_h stored on every attempt) — straight against the oracle: same accepted /
    rejected counts per trajectory and the state within rtol. (The controller's powf is correctly rounded here and glibc's in
    the oracle, which rounds differently for about one argument in a thousand, so a step size may differ in its last bit now
    and then: states are compared to 1e-9, not bitwise.)"""
    n, rtol, tf = 2048, 1e-6, 4.0
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n)
    ref = oracle.rk_ensemble("VDP", mu[:, None], oracle.builtin_tableau(oracle.TABLEAU_ID[tab]), 0.0, tf, x0, 1e-3, n_threads=8, adaptive=True, rtol=rtol)
    rhs = vo.Rhs(ctx, "VDP", 2, [mu])
    s = vo.RK45Solver(rhs, 0.0, tf, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin(tab)).with_tolerance(rtol, rtol)
    s.set_events_per_launch(1).set_mixed_stepping(prev_h == "every_attempt")
    l0 = ctx.launch_count
    st = s.run(adaptive=True)
    assert st.kind == "Done"
    stats = s.stats()
    calls = int((ref["accepted"] + ref["rejected"]).max()) + 2
    assert ctx.launch_count - l0 >= calls  # one event per launch: at least as many launches as the slowest trajectory has events
    same = (stats["accepted"] == ref["accepted"]) & (stats["rejected"] == ref["rejected"])
    print(f"{tab}: per-trajectory counts equal for {same.mean() * 100:.2f} % of {n}; totals gpu {stats['accepted'].sum()}/{stats['rejected'].sum()}"
          f" oracle {ref['accepted'].sum()}/{ref['rejected'].sum()}")
    assert same.mean() >= 0.995
    assert abs(int(stats["accepted"].sum()) - int(ref["accepted"].sum())) <= 4 and abs(int(stats["rejected"].sum()) - int(ref["rejected"].sum())) <= 4
    x = s.current()[1].to_host()
    assert np.abs(x[same] - ref["x"][same]).max() <= 1e-9
    assert np.abs(x - ref["x"]).max() <= 50 * rtol


def test_strict_full_config2_bit_exact(vo, ctx, oracle):
    """Config 2's whole interval t in [0,1] (1000 steps + the remainder step) in strict arithmetic, through one launch per
    step() call and through vo_run's fused launches: bit-identical to the oracle."""
    n = 2048
    x0 = vo.workloads.lorenz_x0(n)
    params = np.tile(vo.workloads.LORENZ_PARAMS, (n, 1))
    ref = oracle.rk_ensemble("LORENZ63", params, oracle.builtin_tableau(1), 0.0, 1.0, x0, 1e-3, n_threads=8)
    rhs = vo.Rhs(ctx, "LORENZ63", 3, list(vo.workloads.LORENZ_PARAMS))
    a = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin("RK4"))
    calls = 0
    while a.step().is_ok:
        calls += 1
    b = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=vo.ButcherTableu.builtin("RK4"))
    st = b.run()
    assert st.counts["Step"] == int(ref["accepted"].sum()) and calls == int(ref["accepted"][0]) + 1
    assert np.array_equal(a.current()[1].to_host(), ref["x"])
    assert np.array_equal(b.current()[1].to_host(), ref["x"])


def test_shared_then_per_trajectory_parameters_same_kernel(vo, ctx, oracle):
    """The shared-memory size of a staged kernel depends on how many RHS parameters are per-trajectory arrays. A solver with
    shared parameters runs first, then one with per-trajectory parameters through the SAME kernel instantiation with a larger
    tile: the large-shared-memory opt-in and the occupancy must follow (they are cached per (device, kernel, size))."""
    n = 4096
    tab = vo.ButcherTableu.builtin("DOPRI5")
    x0 = vo.workloads.vdp_x0(n)
    for per_traj in (False, True):
        mu = vo.workloads.vdp_mu(n) if per_traj else np.full(n, 3.0)
        rhs = vo.Rhs(ctx, "VDP", 2, [mu if per_traj else 3.0])
        s = vo.RK45Solver(rhs, 0.0, 1.0, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=tab).with_tolerance(1e-6, 1e-6).set_events_per_launch(1)
        assert s.run(adaptive=True).kind == "Done"
        ref = oracle.rk_ensemble("VDP", mu[:, None], oracle.builtin_tableau(2), 0.0, 1.0, x0, 1e-3, n_threads=8, adaptive=True, rtol=1e-6)
        assert np.abs(s.current()[1].to_host() - ref["x"]).max() <= 1e-9
    rng = np.random.default_rng(5)
    lam, y0 = -rng.random((n, 4)) * 2.0, rng.standard_normal((n, 4))
    for per_traj in (False, True):
        p = lam if per_traj else np.tile(lam[0], (n, 1))
        rhs = _make_rhs(vo, ctx, "DIAG_LINEAR", 4, p, per_traj=per_traj)
        s = vo.RK45Solver(rhs, 0.0, 0.05, vo.Ensemble.from_host(ctx, y0), 1e-3, tableau=vo.ButcherTableu.builtin("RK4")).set_events_per_launch(1)
        assert s.run().kind == "Done"
        ref = oracle.rk_ensemble("DIAG_LINEAR", p, oracle.builtin_tableau(1), 0.0, 0.05, y0, 1e-3, n_threads=8)
        assert np.array_equal(s.current()[1].to_host(), ref["x"])


def test_mixed_step_and_step_adaptive(vo, ctx, oracle):
    """step() after step_adaptive() under per-trajectory control. The one-event adaptive kernels keep prev_h — read only by the
    Chkpt / End branch (ode.rs:192-195) — up to date only where a checkpoint comes next, so by default the mix is refused;
    with mixed stepping switched on they store it on every attempt (ode.rs:202-205) and the mix follows the oracle's rule:
    the step size a checkpoint restores is the one in force BEFORE the last adaptive attempt."""
    n = 2048
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n)
    tab = vo.ButcherTableu.builtin("DOPRI5")

    def make():
        rhs = vo.Rhs(ctx, "VDP", 2, [mu])
        s = vo.RK45Solver(rhs, 0.0, 0.5, vo.Ensemble.from_host(ctx, x0), 1e-3, tableau=tab).with_tolerance(1e-6, 1e-6)
        return s.set_events_per_launch(1).set_t_list([0.0, 0.05, 0.5])

    s = make()
    for _ in range(6):
        s.step_adaptive()
    with pytest.raises(vo.VecOdeError):
        s.step()
    s = make().set_mixed_stepping(True)
    for _ in range(6):
        s.step_adaptive()
    t = make().set_mixed_stepping(True)
    for _ in range(5):
        t.step_adaptive()
    h_before_last = t.stats()["h"].copy()
    # non-adaptive steps up to the checkpoint at 0.05: every trajectory then restores prev_h = the h before its last adaptive attempt
    passed = 0
    for _ in range(3000):
        passed += s.step().counts["Chkpt"]
        if passed == n:
            break
    assert passed == n
    assert np.array_equal(s.stats()["h"], h_before_last)


SWEEP_LISTS = {"": (0.0, 0.4, 1.0, 1.5), "-41": tuple(np.linspace(0.0, 1.5, 41))}  # 4 output times (inline) and 41 (device memory)


@pytest.mark.parametrize("n,t_list", [pytest.param(n, tl, id=f"{n}{key}") for key, tl in SWEEP_LISTS.items()
                                      for n in (1024, 1026, 2500, 8192, 40_000, 65_538)])
def test_one_event_sweep_equals_stage_path_bitwise(vo, n, t_list):
    """The one-event adaptive sweep of the register-resident path (rk_small2.cuh: rk_ctl2w_staged_kernel, its slow path and
    ragged tail through ctl_lane) against the stage path in strict arithmetic (FAST's reformulated controller exists only on
    the register path): every bit of the state, of the controller arrays and of the snapshots must agree — through
    checkpoints, snapshots, ragged tails (n % 256 != 0), reads in mid-run, a write to the borrowed ensemble, a parameter
    change and a switch to the 8-event kernel and back; with 4 output times (inline) and 41 (read from device memory). The public state layout is the only one: set_blocked(False) is
    accepted, set_blocked(True) refused."""
    c = vo.Context(0, arith="strict")
    mu = vo.workloads.vdp_mu(n)
    x0 = vo.workloads.vdp_x0(n) + 1e-3 * np.sin(np.arange(2 * n)).reshape(n, 2)
    out = []
    for stage_path in (False, True):
        rhs = vo.Rhs(c, "VDP", 2, [mu])
        s = vo.RK45Solver(rhs, 0.0, 1.5, vo.Ensemble.from_host(c, x0), 1e-3, tableau=vo.ButcherTableu.builtin("DOPRI5")).with_tolerance(1e-6, 1e-6)
        s.set_blocked(False).set_stage_path(stage_path).set_events_per_launch(1).set_t_list(t_list).enable_snapshots()
        with pytest.raises(vo.VecOdeError):
            s.set_blocked(True)
        for _ in range(25):
            s.step_adaptive()
        mid = s.stats()
        for _ in range(10):
            s.step_adaptive()
        vo.LinearCombination.scale(s.current()[1], 1.0 + 2.0 ** -30)   # the caller writes the borrowed state
        for _ in range(10):
            s.step_adaptive()
        rhs.set_param(0, mu * (1.0 + 2.0 ** -20))         # a parameter changes in mid-run
        for _ in range(10):
            s.step_adaptive()
        s.set_events_per_launch(8)
        s.run(adaptive=True, max_calls=24)                # the 8-event kernel on the register-resident path ...
        s.set_events_per_launch(1)
        st = s.run(adaptive=True)                         # ... and back to the one-event sweep until every trajectory is done
        assert st.kind == "Done"
        out.append((s.current()[1].to_host(), s.stats(), mid, [s.snapshot(k).to_host() for k in range(len(t_list))]))
    (xa, sa, ma, snapa), (xb, sb, mb, snapb) = out
    assert np.array_equal(xa, xb)
    for k in ("accepted", "rejected", "t", "h", "dx_norm", "status"):
        assert np.array_equal(sa[k], sb[k]), k
        assert np.array_equal(ma[k], mb[k]), "mid-run " + k
    for a, b in zip(snapa, snapb):
        assert np.array_equal(a, b)
    assert np.all(sa["status"] == 1) and np.all(sa["t"] == 1.5)
