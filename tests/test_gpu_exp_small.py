"""Exponential integrators for systems of 1 to 8 levels (exp_small_kernel: one system per thread, FP64 in registers) against
scipy expm, the CPU oracle, dense restatements and a closed form. Bars as for n >= 16: <= 1e-12 on states, unitarity to 1e-12."""
import numpy as np
import pytest

from oracle import split_oracle as so

pytestmark = pytest.mark.gpu


def _herm(rng, n):
    G = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    return (G + G.conj().T) / (2.0 * np.sqrt(n))


def _system(vo, n, N, seed=3):
    rng = np.random.default_rng(100 + n)
    k = np.arange(n)
    H0 = np.diag((k - (n - 1) / 2) * 0.3) + np.diag(np.full(n - 1, 0.5), 1) + np.diag(np.full(n - 1, 0.5), -1) if n > 1 else np.array([[0.4]])
    H1 = _herm(rng, n)
    gp = vo.workloads.schrodinger_drive(N)
    rng = np.random.default_rng(seed)
    psi0 = rng.standard_normal((N, n)) + 1j * rng.standard_normal((N, n))
    psi0 /= np.linalg.norm(psi0, axis=1, keepdims=True)
    return -1j * H0.astype(complex), -1j * H1, gp, psi0


def _map(vo, split, u, psi):
    import torch
    N, n = psi.shape
    x = torch.from_numpy(psi.view(np.float64).reshape(N, n, 2).copy()).cuda()
    y = torch.empty_like(x)
    split.map_exp(u, x.data_ptr(), y.data_ptr())
    torch.cuda.synchronize()
    return y.cpu().numpy().reshape(N, 2 * n).view(np.complex128)


@pytest.mark.parametrize("M", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6, 7, 8])
def test_map_exp_every_small_shape(vo, ctx, n, M):
    """map_exp against scipy expm per system, ragged batch, ||L||_1 up to ~6 (several sub-steps of the Taylor series)."""
    from scipy.linalg import expm
    N = 37
    rng = np.random.default_rng(10 * n + M)
    basis = np.stack([-1j * _herm(rng, n) for _ in range(M)])
    coef = (rng.uniform(-0.6, 0.6, (N, M)) + 0.1j * rng.uniform(-1, 1, (N, M))) * rng.choice([0.2, 1.0, 3.0, 6.0], (N, 1))
    psi = rng.standard_normal((N, n)) + 1j * rng.standard_normal((N, n))
    sp = vo.DenseBasisSplit(ctx, basis)
    got = _map(vo, sp, sp.exp(coef), psi)
    for i in range(N):
        ref = expm(np.einsum("m,mij->ij", coef[i], basis)) @ psi[i]
        assert np.abs(got[i] - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max()), (i, np.abs(got[i] - ref).max())


@pytest.mark.parametrize("name,ref", [("StrangSplit", so.strang), ("TripleJumpExpSplit", so.triple_jump)])
def test_map_exp_seq_through_composite_splits(vo, ctx, name, ref):
    """vo_map_exp_seq: a composite split's sequence of exponentials in one launch, n = 3, against the dense restatement."""
    n, N = 3, 21
    rng = np.random.default_rng(2)
    basis = np.stack([-1j * _herm(rng, n) for _ in range(3)])
    sp = vo.DenseBasisSplit(ctx, basis)
    psi = rng.standard_normal((N, n)) + 1j * rng.standard_normal((N, n))
    la, lb = rng.uniform(0.1, 0.9, (N, 2)) + 0j, rng.uniform(0.1, 0.9, (N, 1)) + 0j
    split = getattr(vo, name)(sp, [0, 1], [2])
    got = _map(vo, split, split.exp(vo.DirectSumL(la, lb)), psi)
    for i in range(N):
        want = ref(la[i, 0] * basis[0] + la[i, 1] * basis[1], lb[i, 0] * basis[2], psi[i])
        assert np.abs(got[i] - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (i, np.abs(got[i] - want).max())


def _solver(vo, ctx, scheme, B0, B1, gp, psi0, t1, h, **kw):
    if scheme == "magnus42":
        basis, cs = vo.with_commutator_slot(B0, B1)
        sp = vo.DenseBasisSplit(ctx, basis, commutator_structure=cs)
    else:
        basis, cs = np.stack([B0, B1]), None
        sp = vo.DenseBasisSplit(ctx, basis)
    cls = {"midpoint": "MidpointExpLinearSolver", "cfm4": "ExpCFMSolver", "magnus42": "MagnusExpLinearSolver"}[scheme]
    return getattr(vo, cls)(sp, gp, 0.0, t1, psi0, h, M_gen=2, **kw), basis, cs


@pytest.mark.parametrize("scheme", ["midpoint", "cfm4", "magnus42"])
@pytest.mark.parametrize("n", [2, 3, 8])
def test_fixed_step_schemes_match_oracle(vo, ctx, oracle, scheme, n):
    N = 40
    B0, B1, gp, psi0 = _system(vo, n, N)
    s, basis, cs = _solver(vo, ctx, scheme, B0, B1, gp, psi0, 2.0, 0.1)
    s.no_adaptive()
    ref = oracle.exp_ensemble(scheme, basis, gp, psi0, 0.0, 2.0, 0.1, M_gen=2, cs=cs, no_adaptive=True, n_threads=8)
    st = s.run()
    assert st.kind == "Done" and st.counts["Step"] == int(ref["accepted"].sum()) and st.counts["Chkpt"] == N
    (tmin, tmax), psi = s.current()
    assert tmin == tmax == ref["t"][0]
    assert np.abs(psi - ref["psi"]).max() <= 1e-12
    assert np.abs(np.linalg.norm(psi, axis=1) - 1.0).max() <= 1e-12


@pytest.mark.parametrize("scheme", ["cfm4", "magnus42"])
@pytest.mark.parametrize("n", [2, 4])
def test_adaptive_schemes_match_oracle(vo, ctx, oracle, scheme, n):
    N, rtol = 48, 1e-7
    B0, B1, gp, psi0 = _system(vo, n, N)
    s, basis, cs = _solver(vo, ctx, scheme, B0, B1, gp, psi0, 2.0, 0.05)
    s.with_tolerance(rtol, rtol)
    ref = oracle.exp_ensemble(scheme, basis, gp, psi0, 0.0, 2.0, 0.05, M_gen=2, cs=cs, adaptive=True, no_adaptive=False, rtol=rtol, n_threads=8)
    assert s.run(adaptive=True).kind == "Done"
    stats = s.stats()
    assert np.abs(stats["t"] - 2.0).max() <= 1e-13
    assert np.abs(s.current()[1] - ref["psi"]).max() <= 50 * rtol
    assert abs(int(stats["accepted"].sum()) - int(ref["accepted"].sum())) <= 0.02 * ref["accepted"].sum() + 2


def test_detuned_two_level_system_closed_form(vo, ctx):
    """H = (Omega sigma_x + Delta sigma_z) / 2 with a spread of Delta: constant L, so CFM4's two exponentials compose to exp(h L) and
    P1(t) = Omega^2 / (Omega^2 + Delta^2) sin^2(sqrt(Omega^2 + Delta^2) t / 2) for 10^4 systems."""
    N, Om, h, steps = 10_000, 1.3, 0.05, 40
    sx, sz = np.array([[0, 1], [1, 0]], complex), np.array([[1, 0], [0, -1]], complex)
    delta = np.linspace(-3.0, 3.0, N)
    gp = np.zeros((N, 1, 3))
    gp[:, 0, 0] = delta  # g_1(t) = Delta cos(0 t + 0)
    sp = vo.DenseBasisSplit(ctx, np.stack([-0.5j * Om * sx, -0.5j * sz]))
    psi0 = np.zeros((N, 2), complex)
    psi0[:, 0] = 1.0
    s = vo.ExpCFMSolver(sp, gp, 0.0, h * steps, psi0, h, M_gen=2).no_adaptive()
    assert s.run().kind == "Done"
    (_, t), psi = s.current()
    W = np.sqrt(Om ** 2 + delta ** 2)
    p1 = Om ** 2 / W ** 2 * np.sin(W * t / 2) ** 2
    assert np.abs(np.abs(psi[:, 1]) ** 2 - p1).max() <= 1e-12
    assert np.abs(np.linalg.norm(psi, axis=1) - 1.0).max() <= 1e-12


def _L3(B, gp3, i, t):
    return B[0] + gp3[i, 0, 0] * np.cos(gp3[i, 0, 1] * t + gp3[i, 0, 2]) * B[1] + gp3[i, 1, 0] * np.cos(gp3[i, 1, 1] * t + gp3[i, 1, 2]) * B[2]


def test_applied_commutator_magnus_on_generators_not_closed_under_commutation(vo, ctx):
    """magnus_42 with the commutator applied by products, three random generators at n = 3, large steps, against a dense restatement."""
    from scipy.linalg import expm
    n, N, h = 3, 21, 0.35
    B0, B1, gp, psi0 = _system(vo, n, N)
    B2 = -1j * _herm(np.random.default_rng(12), n)
    gp3 = np.concatenate([gp, gp * np.array([0.6, 1.7, 1.0]) + np.array([0.0, 0.0, 0.4])], axis=1)
    basis = np.stack([B0, B1, B2])
    a = vo.MagnusExpLinearSolver(vo.DenseBasisSplit(ctx, basis), gp3, 0.0, 1.05, psi0, h, applied_commutator=True).no_adaptive()
    assert a.run().kind == "Done"
    got = a.current()[1]
    assert np.abs(np.linalg.norm(got, axis=1) - 1.0).max() <= 1e-12
    c_mid = 0.288675134594812882254574390251
    for i in range(N):
        x, t = psi0[i].copy(), 0.0
        for dt in (h, h, h):
            l0, l1 = _L3(basis, gp3, i, t + dt / 2 - c_mid * dt), _L3(basis, gp3, i, t + dt / 2 + c_mid * dt)
            om = (l0 + l1) * (dt / 2) + (l0 @ l1 - l1 @ l0) * (dt * dt * -0.144337567297406441127287195125)
            x, t = expm(om) @ x, t + dt
        assert np.abs(got[i] - x).max() <= 1e-12, (i, np.abs(got[i] - x).max())


def test_tables_cfm_general_and_split_cfm(vo, ctx, oracle):
    """ExpCFMGeneralSolver with BLANES17_R4_J4 on the 6th-order Gauss nodes against the oracle, and ExpSplitCFMSolver against the
    dense restatement, n = 2."""
    n, N = 2, 24
    B0, B1, gp, psi0 = _system(vo, n, N)
    nodes = [0.5 - np.sqrt(15.0) / 10.0, 0.5, 0.5 + np.sqrt(15.0) / 10.0]
    alpha = vo.cfm_table("BLANES17_R4_J4")
    sp = vo.DenseBasisSplit(ctx, np.stack([B0, B1]))
    s = vo.ExpCFMGeneralSolver(sp, gp, 0.0, 2.0, psi0, 0.1, nodes, alpha)
    assert s.run().kind == "Done"
    ref = oracle.exp_ensemble("cfm_table", np.stack([B0, B1]), gp, psi0, 0.0, 2.0, 0.1, no_adaptive=True, tables=(nodes, alpha, None))
    assert np.abs(s.current()[1] - ref["psi"]).max() <= 1e-12 and np.array_equal(s.stats()["accepted"], ref["accepted"])
    c = list(vo.cfm_table("C_GAUSS_LEGENDRE_4")[0])
    rho, sigma = [[0.30, 0.20], [0.20, 0.30]], [[0.15, 0.05], [0.35, 0.25], [0.05, 0.15]]
    h, steps = 0.07, 3
    s = vo.ExpSplitCFMSolver(sp, [0], gp, 0.0, steps * h, psi0, h, c, rho, sigma)
    assert s.run().kind == "Done"
    got, acc = s.current()[1], s.stats()["accepted"]
    for i in range(N):
        y, t = psi0[i].copy(), 0.0
        for k in range(int(acc[i])):
            dt = h if k < steps else steps * h - t
            y = so.split_cfm_step(lambda tt: B0, lambda tt: gp[i, 0, 0] * np.cos(gp[i, 0, 1] * tt + gp[i, 0, 2]) * B1, t, y, dt, c, rho, sigma)
            t += dt
        assert np.abs(got[i] - y).max() <= 1e-12, (i, np.abs(got[i] - y).max())


COS_BODY = "g[1] = p[0] * cos(p[1] * t + p[2]);"


@pytest.mark.parametrize("scheme", ["cfm4", "midpoint", "magnus42"])
def test_user_generator_restating_the_cosine_family_gives_the_builtin_bits(vo, ctx, scheme):
    n, N = 3, 40
    B0, B1, gp, psi0 = _system(vo, n, N)
    out = []
    for custom in (False, True):
        s, _, _ = _solver(vo, ctx, scheme, B0, B1, gp, psi0, 1.0, 0.1)
        s.no_adaptive()
        if custom:
            s.set_generator(COS_BODY)
        assert s.run().kind == "Done"
        out.append(s.current()[1])
    assert np.array_equal(out[0].view(np.float64), out[1].view(np.float64))


def test_user_generator_gaussian_pulse_and_user_norm(vo, ctx):
    """A Gaussian pulse g(t) = a exp(-(t - t0)^2 / w^2) against CFM4 restated with dense exponentials; then a user norm (the 2-norm
    written as source) must give the built-in controller's bits on an adaptive run."""
    from scipy.linalg import expm
    n, N, h, steps = 2, 20, 0.1, 10
    B0, B1, _, psi0 = _system(vo, n, N)
    rng = np.random.default_rng(2)
    gp = np.stack([rng.uniform(0.5, 2.0, N), rng.uniform(0.2, 0.8, N), rng.uniform(0.3, 0.7, N)], axis=1)[:, None, :]
    sp = vo.DenseBasisSplit(ctx, np.stack([B0, B1]))
    s = vo.ExpCFMSolver(sp, gp, 0.0, h * steps, psi0, h, M_gen=2).no_adaptive()
    s.set_generator("g[1] = p[0] * exp(-(t - p[2]) * (t - p[2]) / (p[1] * p[1]));")
    assert s.run().kind == "Done"
    got = s.current()[1]
    c = (0.21132486540518711775, 0.78867513459481288225)
    a = ((0.53867513459481288225, -0.038675134594812882255), (-0.038675134594812882255, 0.53867513459481288225))
    for i in range(N):
        g = lambda t: gp[i, 0, 0] * np.exp(-(t - gp[i, 0, 2]) ** 2 / gp[i, 0, 1] ** 2)
        x, t = psi0[i].copy(), 0.0
        for _ in range(steps):
            L = [B0 + g(t + cq * h) * B1 for cq in c]
            for row in a:
                x = expm(h * (row[0] * L[0] + row[1] * L[1])) @ x
            t += h
        assert np.abs(got[i] - x).max() <= 1e-12, (i, np.abs(got[i] - x).max())
    gp2 = vo.workloads.schrodinger_drive(N)
    runs = []
    for norm in (None, vo.NormFn(ctx, "m = e * e + im * im;", "sum", "r = sqrt(acc);")):
        s = vo.ExpCFMSolver(sp, gp2, 0.0, 2.0, psi0, 0.05, M_gen=2).with_tolerance(1e-7, 1e-7)
        if norm is not None:
            s.with_norm(norm)
        assert s.run(adaptive=True).kind == "Done"
        runs.append((s.current()[1], s.stats()))
    assert np.array_equal(runs[0][1]["accepted"], runs[1][1]["accepted"]) and np.array_equal(runs[0][1]["rejected"], runs[1][1]["rejected"])
    assert np.abs(runs[0][0] - runs[1][0]).max() <= 1e-13


@pytest.mark.parametrize("scheme,adaptive", [("cfm4", False), ("cfm4", True), ("magnus42", True)])
def test_fused_events_equal_single_steps_bitwise(vo, ctx, scheme, adaptive):
    """vo_exp_run fuses several events per launch on this path: run(max_calls=k) must equal k calls of step() / step_adaptive()."""
    n, N, k = 3, 333, 23
    B0, B1, gp, psi0 = _system(vo, n, N)
    res = []
    for fused in (True, False):
        s, _, _ = _solver(vo, ctx, scheme, B0, B1, gp, psi0, 2.0, 0.05)
        if adaptive:
            s.with_tolerance(1e-7, 1e-7)
        else:
            s.no_adaptive()
        if fused:
            s.run(adaptive=adaptive, max_calls=k)
        else:
            for _ in range(k):
                s.step_adaptive() if adaptive else s.step()
        res.append((s.current()[1], s.stats()))
    (pa, sa), (pb, sb) = res
    assert np.array_equal(pa.view(np.float64), pb.view(np.float64))
    for key in ("t", "h", "accepted", "rejected", "dx_norm"):
        assert np.array_equal(sa[key], sb[key]), key


def test_dynamic_grouping_and_order_on_this_path(vo, ctx):
    """Every system runs its own Taylor plan here, so dynamic grouping is accepted and changes nothing (bit for bit), and a caller's
    permutation (group_similar -> vo_exp_set_order) keeps results and statistics in the caller's order."""
    n, N = 2, 301
    B0, B1, gp, psi0 = _system(vo, n, N)
    runs = []
    for dyn, grp in ((False, False), (True, False), (False, True)):
        s = vo.ExpCFMSolver(vo.DenseBasisSplit(ctx, np.stack([B0, B1])), gp, 0.0, 1.0, psi0, 0.1, M_gen=2, group_similar=grp).with_tolerance(1e-7, 1e-7)
        if dyn:
            s.dynamic_grouping()
        assert s.run(adaptive=True).kind == "Done"
        runs.append((s.current()[1], s.stats()))
    for psi, st in runs[1:]:
        assert np.array_equal(psi.view(np.float64), runs[0][0].view(np.float64))
        assert np.array_equal(st["accepted"], runs[0][1]["accepted"]) and np.array_equal(st["h"], runs[0][1]["h"])


def test_full_size_qubit_ensemble(vo, ctx):
    """2^22 driven qubits, CFM4, 10 steps: unitarity of every system, and the two halves run apart equal the whole, bit for bit."""
    N, h = 1 << 22, 0.1
    rng = np.random.default_rng(0)
    sx, sz = np.array([[0, 1], [1, 0]], complex), np.array([[1, 0], [0, -1]], complex)
    sp = vo.DenseBasisSplit(ctx, np.stack([-0.5j * sz, -0.5j * sz, -0.5j * sx]))
    gp = np.zeros((N, 2, 3))
    gp[:, 0, 0] = rng.uniform(-0.5, 0.5, N)                 # detuning spread (omega = 0: constant)
    gp[:, 1, 0], gp[:, 1, 1] = 1.0, 1.0 + rng.uniform(-0.1, 0.1, N)  # cosine drive on sigma_x
    psi0 = np.zeros((N, 2), complex)
    psi0[:, 0] = 1.0

    def run(lo, hi):
        s = vo.ExpCFMSolver(sp, gp[lo:hi], 0.0, 10 * h, psi0[lo:hi], h, M_gen=3).no_adaptive()
        assert s.run().kind == "Done"
        return s.current()[1]

    full = run(0, N)
    assert np.abs(np.linalg.norm(full, axis=1) - 1.0).max() <= 1e-13
    half = N // 2
    assert np.array_equal(np.concatenate([run(0, half), run(half, N)]).view(np.float64), full.view(np.float64))


def test_refusals(vo, ctx):
    for n in range(9, 16):
        with pytest.raises(vo.VecOdeError) as e:
            vo.DenseBasisSplit(ctx, np.zeros((2, n, n), dtype=complex))
        assert "1 <= n <= 8" in e.value.msg
    B0, B1, gp, psi0 = _system(vo, 4, 5)
    with pytest.raises(vo.VecOdeError):
        vo.MagnusExpLinearSolver(vo.DenseBasisSplit(ctx, np.stack([B0, B1])), gp, 0.0, 1.0, psi0, 0.1, dense_commutator=True)
