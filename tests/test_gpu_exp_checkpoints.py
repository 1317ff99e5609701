"""Output times and checkpoint snapshots of the exponential solvers (vo_exp_set_t_list, vo_exp_enable_snapshots, vo_exp_snapshot):
every system raises Chkpt at each entry of t_list before the last and End at the last, and the kernels keep the state it shows at
each of those events. Covered on all three kernels: exp_small_kernel (n = 2, 4), exp_step_kernel (n = 16, 64) and
magnus_dense_kernel (n = 16, dense commutator)."""
import numpy as np
import pytest

import _exp_tlist as tl

pytestmark = pytest.mark.gpu

# five entries, two of them (0.13, 0.77) off the grid of h = 0.1 and one (0.5) on it
T_LIST = [0.0, 0.13, 0.5, 0.77, 1.0]
COS_BODY = "g[1] = p[0] * cos(p[1] * t + p[2]);"
# kernel -> (n, extra solver options); "dense16" is magnus_42 with the per-system dense commutator
KERNELS = {"small2": (2, {}), "small4": (4, {}), "tile16": (16, {}), "tile64": (64, {}), "dense16": (16, {"dense_commutator": True})}


def _system(vo, n, N, seed=3):
    if n == 64:
        H0, H1 = vo.workloads.schrodinger_system(64)
    else:
        rng = np.random.default_rng(40 + n)
        k = np.arange(n)
        H0 = np.diag((k - (n - 1) / 2) * 0.3) + np.diag(np.full(n - 1, 0.5), 1) + np.diag(np.full(n - 1, 0.5), -1)
        G = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
        H1 = (G + G.conj().T) / (2.0 * np.sqrt(n))
    gp = vo.workloads.schrodinger_drive(N)
    rng = np.random.default_rng(seed)
    psi0 = rng.standard_normal((N, n)) + 1j * rng.standard_normal((N, n))
    psi0 /= np.linalg.norm(psi0, axis=1, keepdims=True)
    return -1j * H0.astype(complex), -1j * H1, gp, psi0


def _solver(vo, ctx, kernel, scheme, adaptive, N, tf=1.0, h=0.1, seed=3, gp=None, **kw):
    """The solver of `scheme` on `kernel` and the oracle's view of it: (solver, oracle basis, structure tensor)."""
    n, extra = KERNELS[kernel]
    B0, B1, gp0, psi0 = _system(vo, n, N, seed)
    gp = gp0 if gp is None else gp
    basis3, cs = vo.with_commutator_slot(B0, B1)  # the oracle's magnus_42 expands the commutator through a structure tensor
    sp = vo.DenseBasisSplit(ctx, np.stack([B0, B1]))
    if scheme == "magnus42":  # the GPU forms no structure tensor: applied by products, or dense per system on "dense16"
        s = vo.MagnusExpLinearSolver(sp, gp, 0.0, tf, psi0, h, M_gen=2, applied_commutator=not extra, **extra, **kw)
    else:
        s = getattr(vo, {"midpoint": "MidpointExpLinearSolver", "cfm4": "ExpCFMSolver"}[scheme])(sp, gp, 0.0, tf, psi0, h, M_gen=2, **kw)
    s.with_tolerance(1e-7, 1e-7) if adaptive else s.no_adaptive()
    return s, (basis3 if scheme == "magnus42" else np.stack([B0, B1])), (cs if scheme == "magnus42" else None), gp, psi0


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


@pytest.mark.parametrize("kernel", list(KERNELS))
def test_default_list_gives_the_bits_of_no_list(vo, ctx, kernel):
    """set_t_list([t0, tf]) and no call at all: identical state, t, h, counts and dx_norm, fixed and adaptive."""
    scheme = "magnus42" if kernel == "dense16" else "cfm4"
    for adaptive in (False, True):
        out = []
        for explicit in (False, True):
            s = _solver(vo, ctx, kernel, scheme, adaptive, 37, tf=0.95, h=0.07)[0]
            if explicit:
                s.set_t_list([0.0, 0.95])
            st = s.run(adaptive=adaptive)
            assert st.kind == "Done"
            out.append((s.current()[1], s.stats(), st.counts))
        (pa, sa, ca), (pb, sb, cb) = out
        assert np.array_equal(_bits(pa), _bits(pb)) and ca == cb
        for key in ("t", "h", "accepted", "rejected", "dx_norm"):
            assert np.array_equal(_bits(sa[key]), _bits(sb[key])), (adaptive, key)


ORACLE_CASES = [(k, "midpoint", False) for k in ("small2", "small4", "tile16", "tile64")] + \
               [(k, "cfm4", a) for k in ("small2", "small4", "tile16", "tile64") for a in (False, True)] + \
               [(k, "magnus42", True) for k in ("small2", "small4", "tile16", "tile64")] + \
               [("dense16", "magnus42", False), ("dense16", "magnus42", True)]


@pytest.mark.parametrize("kernel,scheme,adaptive", ORACLE_CASES)
def test_snapshots_against_the_oracle(vo, ctx, oracle, kernel, scheme, adaptive):
    """Snapshot k equals the oracle's solve whose list stops at entry k (<= 1e-12), with the same per-system counts; the run raises
    N (len - 1) Chkpt events and ends every system on the last entry."""
    N = 24
    s, basis, cs, gp, psi0 = _solver(vo, ctx, kernel, scheme, adaptive, N, h=0.05 if adaptive else 0.1)
    s.set_t_list(T_LIST).enable_snapshots()
    st = s.run(adaptive=adaptive)
    assert st.kind == "Done" and st.counts["Chkpt"] == N * (len(T_LIST) - 1) and st.counts["End"] == N
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-7) if adaptive else dict(no_adaptive=True)
    h = 0.05 if adaptive else 0.1
    for k in range(len(T_LIST)):
        ref = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 1.0, h, M_gen=2, cs=cs, t_list=T_LIST[:k + 1], n_threads=8, **kw)
        err = np.abs(s.snapshot(k) - ref["psi"]).max()
        assert err <= 1e-12, (k, err)
    stats = s.stats()  # `ref` is now the solve over the whole list
    assert np.array_equal(stats["accepted"], ref["accepted"]) and np.array_equal(stats["rejected"], ref["rejected"])
    assert np.all(np.abs(stats["t"] - 1.0) <= 2.0 ** -52)
    assert np.array_equal(_bits(s.snapshot(len(T_LIST) - 1)), _bits(s.current()[1]))


@pytest.mark.parametrize("kernel", ["small4", "tile16", "dense16"])
def test_snapshot_equals_current_at_the_event(vo, ctx, kernel):
    """Stepped one event at a time: whenever a system sits on t_list[k] (within 2^-52, the reference's rule), current() shows it;
    the last such state of every system is snapshot k, bit for bit. Adaptive, so systems reach each entry in different calls."""
    N = 40
    scheme = "magnus42" if kernel == "dense16" else "cfm4"
    s = _solver(vo, ctx, kernel, scheme, True, N, h=0.05)[0]
    s.set_t_list(T_LIST).enable_snapshots()
    seen = np.zeros((len(T_LIST), N), dtype=bool)
    want = np.zeros((len(T_LIST), N, KERNELS[kernel][0]), dtype=complex)
    calls = []
    for call in range(2000):
        t = s.stats()["t"]
        psi = s.current()[1]
        for k, tk in enumerate(T_LIST):
            at = np.abs(t - tk) <= 2.0 ** -52
            want[k, at], seen[k, at] = psi[at], True
            if at.any():
                calls.append((k, call))
        if s.step_adaptive().kind == "Done":
            break
    assert seen.all()
    for k in range(len(T_LIST)):
        assert np.array_equal(_bits(s.snapshot(k)), _bits(want[k])), k
    first = {k: min(c for kk, c in calls if kk == k) for k in range(1, len(T_LIST))}
    last = {k: max(c for kk, c in calls if kk == k) for k in range(1, len(T_LIST))}
    assert any(last[k] > first[k] + 1 for k in first)  # some entry was reached in different calls


def test_fused_launches_give_the_snapshots_of_single_steps(vo, ctx):
    """exp_small_kernel inside vo_exp_run runs 16 events per launch, so a checkpoint falls in the middle of a launch: snapshots of
    run() equal those of single step_adaptive() calls bit for bit, on an ensemble whose systems take very different step counts."""
    N = 1000
    gp = vo.workloads.schrodinger_drive(N).copy()
    gp[:, 0, 0] *= np.linspace(0.2, 6.0, N)  # weak to strong drive: the controller takes few to many steps
    runs, launches, calls = [], 0, 0
    for fused in (True, False):
        s = _solver(vo, ctx, "small2", "cfm4", True, N, h=0.05, gp=gp)[0]
        s.set_t_list(T_LIST).enable_snapshots()
        if fused:
            launches = s.run(adaptive=True).counts["launches"]
        else:
            calls = 1
            while s.step_adaptive().kind != "Done":
                calls += 1
        runs.append((s, s.stats()))
    assert 8 * launches < calls  # several events per launch
    (a, sa), (b, sb) = runs
    assert np.unique(sa["accepted"]).size > 10
    for k in range(len(T_LIST)):
        assert np.array_equal(_bits(a.snapshot(k)), _bits(b.snapshot(k))), k
    for key in ("t", "h", "accepted", "rejected"):
        assert np.array_equal(sa[key], sb[key]), key


@pytest.mark.parametrize("kernel", ["small4", "tile16", "dense16"])
def test_snapshots_in_the_callers_order(vo, ctx, kernel):
    """With a permutation (group_similar -> vo_exp_set_order) and, on the tiles, dynamic grouping, snapshots come back in the
    caller's order and equal the plain-order run to 1e-13; the device view holds the same rows as the host copy."""
    N = 77
    scheme = "magnus42" if kernel == "dense16" else "cfm4"
    variants = [{}, {"group_similar": True}] + ([{"dynamic": True}] if kernel == "tile16" else [])
    snaps = []
    for v in variants:
        s = _solver(vo, ctx, kernel, scheme, False, N, group_similar=v.get("group_similar", False))[0]
        if v.get("group_similar"):
            assert s._perm is not None and not np.array_equal(s._perm, np.arange(N))
        if v.get("dynamic"):
            s.dynamic_grouping()
        s.set_t_list(T_LIST).enable_snapshots()
        assert s.run().kind == "Done"
        snaps.append(np.stack([s.snapshot(k) for k in range(len(T_LIST))]))
        for k in (1, 3):
            dev = s.snapshot_ensemble(k).to_host().reshape(-1).view(np.complex128).reshape(N, -1)
            assert np.array_equal(_bits(dev), _bits(snaps[-1][k]))
    for other in snaps[1:]:
        assert np.abs(other - snaps[0]).max() <= 1e-13


@pytest.mark.parametrize("kernel", ["small2", "tile64"])
def test_user_generator_and_norm_snapshots(vo, ctx, kernel):
    """The cosine drive written as a generator body gives the built-in family's snapshot bits; a user norm (the 2-norm as source)
    gives the built-in controller's counts and its snapshots to 1e-13."""
    N = 40
    out = []
    for custom in (False, True):
        s = _solver(vo, ctx, kernel, "cfm4", False, N)[0]
        if custom:
            s.set_generator(COS_BODY)
        s.set_t_list(T_LIST).enable_snapshots()
        assert s.run().kind == "Done"
        out.append(np.stack([s.snapshot(k) for k in range(len(T_LIST))]))
    assert np.array_equal(_bits(out[0]), _bits(out[1]))
    runs = []
    for norm in (None, vo.NormFn(ctx, "m = e * e + im * im;", "sum", "r = sqrt(acc);")):
        s = _solver(vo, ctx, kernel, "cfm4", True, N, h=0.05)[0]
        if norm is not None:
            s.with_norm(norm)
        s.set_t_list(T_LIST).enable_snapshots()
        assert s.run(adaptive=True).kind == "Done"
        runs.append((np.stack([s.snapshot(k) for k in range(len(T_LIST))]), s.stats()))
    assert np.array_equal(runs[0][1]["accepted"], runs[1][1]["accepted"]) and np.array_equal(runs[0][1]["rejected"], runs[1][1]["rejected"])
    assert np.abs(runs[0][0] - runs[1][0]).max() <= 1e-13


def test_long_list_from_device_memory(vo, ctx, oracle):
    """A list longer than the inline part of the launch parameters (41 entries) is read from device memory."""
    N = 16
    s, basis, cs, gp, psi0 = _solver(vo, ctx, "small4", "cfm4", False, N)
    t_list = np.linspace(0.0, 1.0, 41)
    s.set_t_list(t_list).enable_snapshots()
    st = s.run()
    assert st.kind == "Done" and st.counts["Chkpt"] == N * 40
    ref = tl.exp_ensemble("cfm4", basis, gp, psi0, 0.0, 1.0, 0.1, M_gen=2, t_list=t_list, snapshots=True, no_adaptive=True)
    for k in range(0, 41, 8):
        assert np.abs(s.snapshot(k) - ref["snap"][k]).max() <= 1e-12, k


def test_refusals(vo, ctx):
    s = _solver(vo, ctx, "small2", "cfm4", False, 8)[0]

    def code(f, *a):
        with pytest.raises(vo.VecOdeError) as e:
            f(*a)
        return e.value.code

    assert code(s.set_t_list, np.linspace(0.0, 1.0, 65536)) == vo._cabi.VO_ERR_UNSUPPORTED
    assert code(s.set_t_list, []) == vo._cabi.VO_ERR_BAD_ARG
    assert code(s.snapshot, 0) == vo._cabi.VO_ERR_STATE  # snapshots off
    assert code(s.snapshot_ensemble, 0) == vo._cabi.VO_ERR_STATE
    s.set_t_list(T_LIST).enable_snapshots()
    for k in (-1, len(T_LIST)):
        assert code(s.snapshot, k) == vo._cabi.VO_ERR_BAD_ARG
        assert code(s.snapshot_ensemble, k) == vo._cabi.VO_ERR_BAD_ARG
    s.step()
    assert code(s.set_t_list, [0.0, 1.0]) == vo._cabi.VO_ERR_STATE  # stepping has begun
    s.reset()
    s.set_t_list([0.0, 0.5, 1.0])  # accepted again after reset
    assert s.run().kind == "Done" and np.all(np.abs(s.stats()["t"] - 1.0) <= 2.0 ** -52)
    assert s.snapshot(2).shape == (8, 2)
