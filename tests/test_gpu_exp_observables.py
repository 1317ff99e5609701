"""Expectation values of user observables at every output time (vo_exp_set_observables, vo_exp_expectation): at each Chkpt / End event
the kernels compute e[j][i][k] = <psi| O_k |psi> from the state the snapshot keeps. Covered on all three kernels: exp_small_kernel
(n = 1 .. 8), exp_step_kernel (n = 16, 24, 32, 40, 48, 64) and magnus_dense_kernel (n = 16, dense commutator)."""
import numpy as np
import pytest

import _exp_tlist as tl

pytestmark = pytest.mark.gpu

T_LIST = [0.0, 0.13, 0.5, 0.77, 1.0]
COS_BODY = "g[1] = p[0] * cos(p[1] * t + p[2]);"
# kernel -> (n, extra solver options); "dense16" is magnus_42 with the per-system dense commutator
KERNELS = {f"small{n}": (n, {}) for n in range(1, 9)}
KERNELS.update({f"tile{n}": (n, {}) for n in (16, 24, 32, 40, 48, 64)})
KERNELS["dense16"] = (16, {"dense_commutator": True})


def _system(vo, n, N, seed=3):
    if n == 64:
        H0, H1 = vo.workloads.schrodinger_system(64)
    else:
        rng = np.random.default_rng(40 + n)
        k = np.arange(n)
        H0 = np.diag((k - (n - 1) / 2) * 0.3) + np.diag(np.full(n - 1, 0.5), 1) + np.diag(np.full(n - 1, 0.5), -1) if n > 1 else np.array([[0.4]])
        G = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
        H1 = (G + G.conj().T) / (2.0 * np.sqrt(n))
    gp = vo.workloads.schrodinger_drive(N)
    rng = np.random.default_rng(seed)
    psi0 = rng.standard_normal((N, n)) + 1j * rng.standard_normal((N, n))
    psi0 /= np.linalg.norm(psi0, axis=1, keepdims=True)
    return -1j * H0.astype(complex), -1j * H1, gp, psi0


def _ops(n, seed=7):
    """K = 3: a population-like diagonal, a random Hermitian and a random non-Hermitian operator."""
    rng = np.random.default_rng(seed + n)
    G = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    return np.stack([np.diag(np.arange(n, dtype=float)).astype(complex) / max(n - 1, 1), (G + G.conj().T) / 2.0,
                     rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))])


def _solver(vo, ctx, kernel, scheme, adaptive, N, tf=1.0, h=0.1, seed=3, gp=None, **kw):
    """The solver of `scheme` on `kernel` and the oracle's view of it: (solver, oracle basis, structure tensor, gp, psi0)."""
    n, extra = KERNELS[kernel]
    B0, B1, gp0, psi0 = _system(vo, n, N, seed)
    gp = gp0 if gp is None else gp
    basis3, cs = vo.with_commutator_slot(B0, B1)
    sp = vo.DenseBasisSplit(ctx, np.stack([B0, B1]))
    if scheme == "magnus42":
        s = vo.MagnusExpLinearSolver(sp, gp, 0.0, tf, psi0, h, M_gen=2, applied_commutator=not extra, **extra, **kw)
    else:
        s = getattr(vo, {"midpoint": "MidpointExpLinearSolver", "cfm4": "ExpCFMSolver"}[scheme])(sp, gp, 0.0, tf, psi0, h, M_gen=2, **kw)
    s.with_tolerance(1e-7, 1e-7) if adaptive else s.no_adaptive()
    return s, (basis3 if scheme == "magnus42" else np.stack([B0, B1])), (cs if scheme == "magnus42" else None), gp, psi0


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _expect(ops, snap):
    """e[j][i][k] = sum_r conj(psi_r) sum_c O_k[r][c] psi_c and its rounding scale sum_rc |O_rc| |psi_r| |psi_c|, snap [len][N][n]."""
    e = np.einsum("jir,krc,jic->jik", snap.conj(), ops, snap)
    scale = np.einsum("jir,krc,jic->jik", np.abs(snap), np.abs(ops), np.abs(snap))
    return e, scale


def _all(s, f, m):
    return np.stack([f(j) for j in range(m)])


@pytest.mark.parametrize("kernel", ["small2", "small4", "small8", "tile16", "tile64", "dense16"])
def test_observables_change_no_other_output(vo, ctx, kernel):
    """With observables on: state, snapshots, t, h, dx_norm, accepted / rejected counts and event counts bit-identical to the same run
    with them off, fixed and adaptive."""
    scheme = "magnus42" if kernel == "dense16" else "cfm4"
    n = KERNELS[kernel][0]
    for adaptive in (False, True):
        out = []
        for on in (False, True):
            s = _solver(vo, ctx, kernel, scheme, adaptive, 37, h=0.05 if adaptive else 0.1)[0]
            s.set_t_list(T_LIST).enable_snapshots()
            if on:
                s.set_observables(_ops(n))
            st = s.run(adaptive=adaptive)
            assert st.kind == "Done"
            out.append((s.current()[1], _all(s, s.snapshot, len(T_LIST)), s.stats(), st.counts))
        (pa, na, sa, ca), (pb, nb, sb, cb) = out
        assert np.array_equal(_bits(pa), _bits(pb)) and np.array_equal(_bits(na), _bits(nb))
        assert {k: v for k, v in ca.items() if k != "launches"} == {k: v for k, v in cb.items() if k != "launches"}
        for key in ("t", "h", "accepted", "rejected", "dx_norm"):
            assert np.array_equal(_bits(sa[key]), _bits(sb[key])), (adaptive, key)


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_expectations_equal_the_einsum_of_the_snapshots(vo, ctx, kernel):
    """K = 3 operators, one of them non-Hermitian: every expectation equals the einsum of the same run's snapshot within
    1e-13 sum_rc |O_rc| |psi_r| |psi_c|, at every n of the small kernel and every compiled tile n."""
    n = KERNELS[kernel][0]
    scheme = "magnus42" if kernel == "dense16" else "cfm4"
    s = _solver(vo, ctx, kernel, scheme, True, 45, h=0.05)[0]
    ops = _ops(n)
    s.set_t_list(T_LIST).enable_snapshots().set_observables(ops)
    assert s.run(adaptive=True).kind == "Done"
    got = _all(s, s.expectation, len(T_LIST))
    assert got.shape == (len(T_LIST), 45, 3)
    want, scale = _expect(ops, _all(s, s.snapshot, len(T_LIST)))
    assert np.all(np.abs(got - want) <= 1e-13 * scale + 1e-300), np.abs(got - want).max()
    assert np.abs(got[..., 2].imag).max() > 1e-3  # the non-Hermitian operator has a genuine imaginary part


ORACLE_CASES = [(k, "midpoint", False) for k in ("small2", "small8", "tile16", "tile64")] + \
               [(k, "cfm4", a) for k in ("small2", "small8", "tile16", "tile64") for a in (False, True)] + \
               [(k, "magnus42", True) for k in ("small2", "small8", "tile16", "tile64")] + \
               [("dense16", "magnus42", False), ("dense16", "magnus42", True)]


@pytest.mark.parametrize("kernel,scheme,adaptive", ORACLE_CASES)
def test_expectations_against_the_oracle(vo, ctx, oracle, kernel, scheme, adaptive):
    """Expectations of the oracle's snapshots (tl.exp_ensemble with the same list) within 1e-12, with the same per-system counts.
    magnus_42 runs with the applied commutator on the small kernel and the tiles, with the dense one on "dense16"."""
    N = 24
    h = 0.05 if adaptive else 0.1
    s, basis, cs, gp, psi0 = _solver(vo, ctx, kernel, scheme, adaptive, N, h=h)
    ops = _ops(KERNELS[kernel][0])
    s.set_t_list(T_LIST).set_observables(ops)
    assert s.run(adaptive=adaptive).kind == "Done"
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-7) if adaptive else dict(no_adaptive=True)
    ref = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 1.0, h, M_gen=2, cs=cs, t_list=T_LIST, snapshots=True, n_threads=8, **kw)
    want = _expect(ops, ref["snap"])[0]
    err = np.abs(_all(s, s.expectation, len(T_LIST)) - want).max()
    assert err <= 1e-12, err
    stats = s.stats()
    assert np.array_equal(stats["accepted"], ref["accepted"]) and np.array_equal(stats["rejected"], ref["rejected"])


def test_detuned_two_level_closed_form(vo, ctx):
    """H = (Omega sigma_x + Delta sigma_z) / 2 over 10^4 detunings from |0>: <sigma_z>(t) = 1 - 2 Omega^2 / W^2 sin^2(W t / 2),
    W^2 = Omega^2 + Delta^2, at 50 output times within 1e-10 (and a zero imaginary part)."""
    N, Om, h = 10_000, 1.3, 0.05
    sx, sz = np.array([[0, 1], [1, 0]], complex), np.array([[1, 0], [0, -1]], complex)
    delta = np.linspace(-3.0, 3.0, N)
    gp = np.zeros((N, 1, 3))
    gp[:, 0, 0] = delta
    sp = vo.DenseBasisSplit(ctx, np.stack([-0.5j * Om * sx, -0.5j * sz]))
    psi0 = np.zeros((N, 2), complex)
    psi0[:, 0] = 1.0
    t_list = np.linspace(0.0, 2.0, 50)
    s = vo.ExpCFMSolver(sp, gp, 0.0, 2.0, psi0, h, M_gen=2).no_adaptive()
    s.set_t_list(t_list).set_observables(sz)
    assert s.run().kind == "Done"
    W = np.sqrt(Om ** 2 + delta ** 2)
    for j, t in enumerate(t_list):
        e = s.expectation(j)[:, 0]
        want = 1.0 - 2.0 * Om ** 2 / W ** 2 * np.sin(W * t / 2) ** 2
        assert np.abs(e.real - want).max() <= 1e-10 and np.abs(e.imag).max() <= 1e-10, j


def test_fused_launches_give_the_expectations_of_single_steps(vo, ctx):
    """vo_exp_run fuses 16 events per launch of exp_small_kernel, so checkpoints fall mid-launch: run() gives the expectations of single
    step_adaptive() calls bit for bit on 1 000 qubits whose step counts differ widely."""
    N = 1000
    gp = vo.workloads.schrodinger_drive(N).copy()
    gp[:, 0, 0] *= np.linspace(0.2, 6.0, N)
    runs, launches, calls = [], 0, 0
    for fused in (True, False):
        s = _solver(vo, ctx, "small2", "cfm4", True, N, h=0.05, gp=gp)[0]
        s.set_t_list(T_LIST).set_observables(_ops(2))
        if fused:
            launches = s.run(adaptive=True).counts["launches"]
        else:
            calls = 1
            while s.step_adaptive().kind != "Done":
                calls += 1
        runs.append((_all(s, s.expectation, len(T_LIST)), s.stats()))
    assert 8 * launches < calls
    (ea, sa), (eb, sb) = runs
    assert np.unique(sa["accepted"]).size > 10
    assert np.array_equal(_bits(ea), _bits(eb))
    for key in ("t", "h", "accepted", "rejected"):
        assert np.array_equal(sa[key], sb[key]), key


@pytest.mark.parametrize("kernel", ["small4", "tile16", "dense16"])
def test_expectations_in_the_callers_order(vo, ctx, kernel):
    """Under group_similar (vo_exp_set_order) and, on the tiles, dynamic grouping, expectations come back in the caller's order within
    1e-13 of the plain-order run; the device view holds the host copy's bits."""
    N = 77
    scheme = "magnus42" if kernel == "dense16" else "cfm4"
    ops = _ops(KERNELS[kernel][0])
    variants = [{}, {"group_similar": True}] + ([{"dynamic": True}] if kernel == "tile16" else [])
    res = []
    for v in variants:
        s = _solver(vo, ctx, kernel, scheme, False, N, group_similar=v.get("group_similar", False))[0]
        if v.get("group_similar"):
            assert s._perm is not None and not np.array_equal(s._perm, np.arange(N))
        if v.get("dynamic"):
            s.dynamic_grouping()
        s.set_t_list(T_LIST).set_observables(ops)
        assert s.run().kind == "Done"
        res.append(_all(s, s.expectation, len(T_LIST)))
        for j in (1, 4):
            dev = s.expectation_ensemble(j).to_host().reshape(-1).view(np.complex128).reshape(N, 3)
            assert np.array_equal(_bits(dev), _bits(res[-1][j]))
    for other in res[1:]:
        assert np.abs(other - res[0]).max() <= 1e-13


@pytest.mark.parametrize("kernel", ["small2", "tile64"])
def test_user_generator_and_norm_expectations(vo, ctx, kernel):
    """The cosine drive written as a generator body gives the built-in family's expectation bits; a user norm (the 2-norm as source)
    gives the built-in controller's counts."""
    N = 40
    ops = _ops(KERNELS[kernel][0])
    out = []
    for custom in (False, True):
        s = _solver(vo, ctx, kernel, "cfm4", False, N)[0]
        if custom:
            s.set_generator(COS_BODY)
        s.set_t_list(T_LIST).set_observables(ops)
        assert s.run().kind == "Done"
        out.append(_all(s, s.expectation, len(T_LIST)))
    assert np.array_equal(_bits(out[0]), _bits(out[1]))
    runs = []
    for norm in (None, vo.NormFn(ctx, "m = e * e + im * im;", "sum", "r = sqrt(acc);")):
        s = _solver(vo, ctx, kernel, "cfm4", True, N, h=0.05)[0]
        if norm is not None:
            s.with_norm(norm)
        s.set_t_list(T_LIST).set_observables(ops)
        assert s.run(adaptive=True).kind == "Done"
        runs.append((_all(s, s.expectation, len(T_LIST)), s.stats()))
    assert np.array_equal(runs[0][1]["accepted"], runs[1][1]["accepted"]) and np.array_equal(runs[0][1]["rejected"], runs[1][1]["rejected"])
    assert np.abs(runs[0][0] - runs[1][0]).max() <= 1e-12


@pytest.mark.parametrize("kernel", ["small4", "tile16"])
def test_long_list_from_device_memory(vo, ctx, oracle, kernel):
    """A list longer than the inline part of the launch parameters (41 entries) is read from device memory."""
    N = 16
    s, basis, cs, gp, psi0 = _solver(vo, ctx, kernel, "cfm4", False, N)
    ops = _ops(KERNELS[kernel][0])
    t_list = np.linspace(0.0, 1.0, 41)
    s.set_t_list(t_list).set_observables(ops)
    st = s.run()
    assert st.kind == "Done" and st.counts["Chkpt"] == N * 40
    ref = tl.exp_ensemble("cfm4", basis, gp, psi0, 0.0, 1.0, 0.1, M_gen=2, t_list=t_list, snapshots=True, no_adaptive=True)
    want = _expect(ops, ref["snap"])[0]
    for j in range(41):
        assert np.abs(s.expectation(j) - want[j]).max() <= 1e-12, j


def test_observables_without_snapshots(vo, ctx):
    """Observables alone: snapshot() refuses with VO_ERR_STATE, expectation() works and gives the bits of the run with snapshots."""
    ops = _ops(4)
    res = []
    for snaps in (False, True):
        s = _solver(vo, ctx, "small4", "cfm4", False, 20)[0]
        s.set_t_list(T_LIST).set_observables(ops)
        if snaps:
            s.enable_snapshots()
        assert s.run().kind == "Done"
        if not snaps:
            with pytest.raises(vo.VecOdeError) as e:
                s.snapshot(0)
            assert e.value.code == vo._cabi.VO_ERR_STATE
        res.append(_all(s, s.expectation, len(T_LIST)))
    assert np.array_equal(_bits(res[0]), _bits(res[1]))


def test_refusals(vo, ctx):
    s = _solver(vo, ctx, "small2", "cfm4", False, 8)[0]
    lib = vo._cabi.lib()

    def code(f, *a):
        with pytest.raises(vo.VecOdeError) as e:
            f(*a)
        return e.value.code

    assert code(s.expectation, 0) == vo._cabi.VO_ERR_STATE  # observables off
    assert code(s.expectation_ensemble, 0) == vo._cabi.VO_ERR_STATE
    assert code(s.set_observables, np.zeros((3, 3))) == vo._cabi.VO_ERR_SHAPE  # n = 2
    assert code(s.set_observables, np.zeros((2, 2, 3))) == vo._cabi.VO_ERR_SHAPE
    assert code(s.set_observables, np.zeros((9, 2, 2))) == vo._cabi.VO_ERR_BAD_ARG  # K > VO_EXP_MAX_OBS
    assert lib.vo_exp_set_observables(s._h, -1, None) == vo._cabi.VO_ERR_BAD_ARG
    assert lib.vo_exp_set_observables(s._h, 2, None) == vo._cabi.VO_ERR_BAD_ARG
    s.set_observables(np.zeros((8, 2, 2)))  # K = 8 is accepted
    s.set_observables(None)  # K = 0: off
    assert code(s.expectation, 0) == vo._cabi.VO_ERR_STATE
    sz = np.diag([1.0, -1.0]).astype(complex)
    s.set_t_list(T_LIST).set_observables(sz)
    for bad in (np.empty((8, 1)), np.empty((8, 2), complex), np.empty((8, 2), complex)[:, :1]):  # dtype, shape, layout of `out`
        assert code(s.expectation, 0, bad) == vo._cabi.VO_ERR_SHAPE
    for j in (-1, len(T_LIST)):
        assert code(s.expectation, j) == vo._cabi.VO_ERR_BAD_ARG
        assert code(s.expectation_ensemble, j) == vo._cabi.VO_ERR_BAD_ARG
    s.step()
    assert code(s.set_observables, sz) == vo._cabi.VO_ERR_STATE  # stepping has begun
    assert code(s.set_observables, None) == vo._cabi.VO_ERR_STATE
    assert s.run().kind == "Done"
    done = _all(s, s.expectation, len(T_LIST))
    s.reset()  # keeps the contents until a run overwrites them
    assert np.array_equal(_bits(_all(s, s.expectation, len(T_LIST))), _bits(done))
    s.set_observables(np.stack([sz, -sz]))  # accepted again after reset
    s.set_t_list([0.0, 0.25, 0.5, 0.75, 1.0])  # re-allocates the [len][N][K] storage
    assert s.run().kind == "Done"
    e = s.expectation(4)
    assert e.shape == (8, 2) and np.abs(e[:, 0] + e[:, 1]).max() <= 1e-15 and np.abs(e[:, 0].real).max() > 0.0
