"""Output times, checkpoint snapshots and expectation values of the exponential solvers (vo_exp_set_t_list, vo_exp_enable_snapshots,
vo_exp_snapshot, vo_exp_set_observables): every system raises Chkpt at each entry of t_list before the last and End at the last,
restores h = prev_h there (exp_event_finish), and the kernels keep the state it shows and <psi| O_k |psi> of that state.

Case table: the row, the kernel it reaches and the rule of exp.cu that selects it. N = 37 systems (77 for dynamic grouping, which
needs N >= 64): ragged, not a multiple of 16 on the tiles nor of 32 on the small kernel.

  row              kernel                          how it is reached
  S1..S8-cfm4a     exp_small_kernel<n, 2>          dispatch_exp: n <= VO_EXP_SMALL_MAX_N; CFM4 adaptive at every n = 1 .. 8: Taylor
                                                   terms on the assembled operator for n <= 4 (SmallOp::ASSEMBLE), per basis matrix above
  S5-cfm4          exp_small_kernel<5, 2>          CFM4 fixed steps
  S1-mid, S5-mid   exp_small_kernel<n, 2>          midpoint, fixed steps
  S3-mag(a)        exp_small_kernel<3, 2>          Magnus, vo_exp_set_applied_commutator, fixed / adaptive: Omega assembled (n <= 3)
  S4-, S7-mag(a)   exp_small_kernel<n, 2>          the same, Omega applied by products (n > 3)
  S2-, S6-M1       exp_small_kernel<n, 1>          M_gen = 1 (constant generator): per-basis branch (ASSEMBLE needs M > 1), fixed
  S3-, S8-M4a      exp_small_kernel<n, 4>          three cosine drives, CFM4 adaptive
  S3-blanes        exp_small_kernel<3, 2>          ExpCFMGeneralSolver with BLANES17_R4_J4 (three nodes, four exponentials), fixed
  T{n}x{M}         exp_step_kernel<n, M, 16>       VO_EXP_CASE of VO_EXP_SHAPES, each of the 16 shapes once, CFM4 fixed steps:
                                                   64x1 64x2 64x3 48x2 48x3 40x2 32x1 32x2 32x3 32x4 24x2 24x3 16x1 16x2 16x3 16x4
  T{n}x{M}-cfm4a   exp_step_kernel                 CFM4 adaptive at 16x2, 40x2, 64x3
  T{n}x{M}-maga    exp_step_kernel                 Magnus with the applied commutator (map_exp_tile_comm), adaptive, at 16x2, 40x2, 64x3
  T24x3-mid        exp_step_kernel<24, 3, 16>      midpoint, fixed steps
  T16x2-, T48x2-dyn exp_step_kernel, `order`       dynamic_grouping (exp_dynamic_order: N >= 64), CFM4 adaptive, tiles by tile_ctr
  D8 .. D64        magnus_dense_kernel<NB>         vo_exp_set_dense_commutator -> launch_magnus_dense, NB = n / 8 = 1 .. 8, fixed steps
  D8-, D24-, D64-a magnus_dense_kernel<NB>         the same, adaptive
  S5-gen, T40x2-gen  run-time compiled modules     the cosine family as a generator body (set_generator), CFM4 adaptive
  S5-norm          run-time compiled module        the 2-norm as a user norm (with_norm), CFM4 adaptive

Lists (absolute times): L5 (0, 0.13, 0.5, 0.77, 1), off the step grid; L8, 8 entries, the last one held inline; L9, 9 entries, the
shortest list read from device memory; L41, 41 entries; EDGE8 (inline) and EDGE (device memory) at h = 0.1: a first entry after t0
(the first call is a Step), 0.2 twice (two Chkpt with no step between them, inside one fused launch of exp_small_kernel), 4.2 /
4.25 / 4.3 closer together than h, and 3.0, 4.2, 4.5 reached by full steps that fall one ulp short (more than 2^-52), so that
exp_event_kind takes a clipped step of one ulp (tests/test_exp_tlist_oracle.py checks that it occurs); ONE, [1.0] alone: End at
entry 0, no Chkpt. Every row runs L5; S2-, S5-, S8-cfm4a, T16x2, T40x2, T64x3 (fixed and -cfm4a) and D16, D40 run every list.
Adaptive runs on EDGE8 / EDGE cap the step at 0.1 (with_step_range(1e-6, 0.1)), so slow systems walk the same grid. Every EDGE8 /
EDGE ensemble holds one system that starts at psi = 0: its embedded error is exactly 0, f = rtol / 0 = inf and the controller takes
pow() instead of pow_third_cr (step_size_mul).

Reference: the C++ oracle driven through the list (tests/_exp_tlist.py, exp_ensemble) on the same inputs; Magnus there expands the
commutator through a structure tensor on the basis closed by the pairwise commutators. Snapshot k of the oracle's run is the final
state of its solve whose list stops at entry k (test_exp_tlist_oracle.py, bit for bit); the final h of that stopped solve is the h
restored at entry k.
Bars, every (row, list): snapshots within 1e-12 of the oracle's; per-system accepted and rejected counts and the Chkpt / End
totals exact; every final t within 2^-52 of the last entry; fixed steps: t and h bit-identical; adaptive: h within 1e-6 relative
(_h_close); K = 3 expectation values (population, random Hermitian, non-Hermitian) within 1e-12 of the einsum of the oracle's
snapshots and within 1e-13 sum |O| |psi| |psi| of the einsum of the run's own; the zero-state system: snapshots and expectations
exactly 0, counts and h equal to the oracle's. GPU against GPU (one event at a time, fused launches, rows written once, caller's
order on the small and dense kernels): bit-identical; the caller's order on the tiles (other tile compositions): 1e-13.

The earlier cases of this file (after the table) keep their own inputs and bars.
"""
import functools
from collections import namedtuple

import numpy as np
import pytest

import _exp_tlist as tl

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
LISTS = {
    "L5": (0.0, 0.13, 0.5, 0.77, 1.0),
    "L8": (0.0, 0.0611, 0.1937, 0.3, 0.4226, 0.55, 0.7123, 1.0),
    "L9": (0.0, 0.0611, 0.1937, 0.3, 0.4226, 0.55, 0.7123, 0.8377, 1.0),
    "L41": tuple(float(v) for v in np.linspace(0.0, 1.0, 41)),
    "EDGE8": (0.2, 0.2, 3.0, 3.3, 4.2, 4.25, 4.3, 4.5),
    "EDGE": (0.2, 0.2, 3.0, 3.3, 4.2, 4.2, 4.25, 4.3, 4.5),
    "ONE": (1.0,),
}
EDGES = ("EDGE8", "EDGE")
ZERO_SYS = 5  # the system of an EDGE ensemble that starts at psi = 0
EDGE_H0 = float(np.sqrt(1e-6 * 0.1))  # the initial step vo_exp_with_step_range(1e-6, 0.1) sets
BLANES_C = np.array([0.5 - np.sqrt(15.0) / 10.0, 0.5, 0.5 + np.sqrt(15.0) / 10.0])
SHAPES = [(64, 1), (64, 2), (64, 3), (48, 2), (48, 3), (40, 2), (32, 1), (32, 2), (32, 3), (32, 4), (24, 2), (24, 3), (16, 1), (16, 2), (16, 3), (16, 4)]

# kind (small / tile / dense), n, M (= M_gen), scheme (midpoint / cfm4 / magnus42 / blanes), adaptive, options (dynamic, gen, norm)
Row = namedtuple("Row", "kind n M scheme adaptive opts")
ROWS = {}
for _n in range(1, 9):
    ROWS[f"S{_n}-cfm4a"] = Row("small", _n, 2, "cfm4", True, {})
ROWS["S5-cfm4"] = Row("small", 5, 2, "cfm4", False, {})
for _n in (1, 5):
    ROWS[f"S{_n}-mid"] = Row("small", _n, 2, "midpoint", False, {})
for _n in (3, 4, 7):
    ROWS[f"S{_n}-mag"] = Row("small", _n, 2, "magnus42", False, {})
    ROWS[f"S{_n}-maga"] = Row("small", _n, 2, "magnus42", True, {})
for _n in (2, 6):
    ROWS[f"S{_n}-M1"] = Row("small", _n, 1, "cfm4", False, {})
for _n in (3, 8):
    ROWS[f"S{_n}-M4a"] = Row("small", _n, 4, "cfm4", True, {})
ROWS["S3-blanes"] = Row("small", 3, 2, "blanes", False, {})
for _n, _m in SHAPES:
    ROWS[f"T{_n}x{_m}"] = Row("tile", _n, _m, "cfm4", False, {})
for _n, _m in ((16, 2), (40, 2), (64, 3)):
    ROWS[f"T{_n}x{_m}-cfm4a"] = Row("tile", _n, _m, "cfm4", True, {})
    ROWS[f"T{_n}x{_m}-maga"] = Row("tile", _n, _m, "magnus42", True, {})
ROWS["T24x3-mid"] = Row("tile", 24, 3, "midpoint", False, {})
for _n in (16, 48):
    ROWS[f"T{_n}x2-dyn"] = Row("tile", _n, 2, "cfm4", True, {"dynamic": True})
for _n in range(8, 65, 8):
    ROWS[f"D{_n}"] = Row("dense", _n, 2, "magnus42", False, {})
for _n in (8, 24, 64):
    ROWS[f"D{_n}-a"] = Row("dense", _n, 2, "magnus42", True, {})
ROWS["S5-gen"] = Row("small", 5, 2, "cfm4", True, {"gen": True})
ROWS["T40x2-gen"] = Row("tile", 40, 2, "cfm4", True, {"gen": True})
ROWS["S5-norm"] = Row("small", 5, 2, "cfm4", True, {"norm": True})
FAMILIES = ["S2-cfm4a", "S5-cfm4a", "S8-cfm4a", "T16x2", "T40x2", "T64x3", "T16x2-cfm4a", "T40x2-cfm4a", "T64x3-cfm4a", "D16", "D40"]
TABLE_CASES = [(r, "L5") for r in ROWS] + [(r, lst) for r in FAMILIES for lst in ("L8", "L9", "L41", "EDGE8", "EDGE", "ONE")]
COS_BODY = "g[1] = p[0] * cos(p[1] * t + p[2]);"
WORST = {}  # largest state error against the oracle per kernel family, largest relative h difference of adaptive runs


def _note(key, v):
    WORST[key] = max(WORST.get(key, 0.0), float(v))
    print(f"{key}: {v:.2e} (largest so far {WORST[key]:.2e})")


def _n_sys(row):
    return 77 if row.opts.get("dynamic") else 37


def _inputs(vo, row, lst, N=None):
    """(basis [M][n][n], gp [N][M-1][3], psi0 [N][n]): the system of the earlier cases (_system) for B_0, B_1, further random
    anti-Hermitian basis matrices and cosine drives for M > 2; on an edge list system ZERO_SYS starts at psi = 0."""
    N = _n_sys(row) if N is None else N
    B0, B1, gp, psi0 = _system(vo, row.n, N)
    mats = [B0, B1][:row.M]
    rng = np.random.default_rng(60 + row.n)
    drives = [gp[:, 0]]
    for _ in range(2, row.M):
        G = rng.standard_normal((row.n, row.n)) + 1j * rng.standard_normal((row.n, row.n))
        mats.append(-1j * (G + G.conj().T) / (2.0 * np.sqrt(row.n)))
        drives.append(np.stack([0.3 + 0.5 * rng.random(N), 0.5 + 1.5 * rng.random(N), 2.0 * np.pi * rng.random(N)], axis=1))
    gp = np.ascontiguousarray(np.stack(drives[:row.M - 1], axis=1)) if row.M > 1 else np.zeros((N, 0, 3))
    psi0 = psi0.copy()
    if lst in EDGES:
        psi0[ZERO_SYS] = 0.0
    return np.stack(mats), gp, psi0


def _closed(basis):
    """The basis closed by the pairwise commutators [B_a, B_b] (a < b) and its structure tensor: the oracle's Magnus expands
    [L(t1), L(t2)] on it (the GPU applies or forms the commutator itself)."""
    M = basis.shape[0]
    pairs = [(a, b) for a in range(M) for b in range(a + 1, M)]
    ext = np.concatenate([basis, np.stack([basis[a] @ basis[b] - basis[b] @ basis[a] for a, b in pairs])])
    cs = np.zeros((len(ext),) * 3)
    for j, (a, b) in enumerate(pairs):
        cs[a, b, M + j], cs[b, a, M + j] = 1.0, -1.0
    return ext, cs


def _h0(row, lst):
    return (EDGE_H0 if lst in EDGES else 0.05) if row.adaptive else 0.1


def _make(vo, ctx, row, lst, N=None, group_similar=False, dynamic=None):
    """The solver of `row` on list `lst` with snapshots and K = 3 observables on, not yet stepped: (solver, t_list, ops)."""
    basis, gp, psi0 = _inputs(vo, row, lst, N)
    t_list = list(LISTS[lst])
    sp = vo.DenseBasisSplit(ctx, basis)
    args = (sp, gp, 0.0, t_list[-1], psi0, _h0(row, lst))
    if row.scheme == "magnus42":
        s = vo.MagnusExpLinearSolver(*args, M_gen=row.M, group_similar=group_similar, applied_commutator=row.kind != "dense",
                                     dense_commutator=row.kind == "dense")
    elif row.scheme == "blanes":
        s = vo.ExpCFMGeneralSolver(*args, c=BLANES_C, alpha=vo.cfm_table("BLANES17_R4_J4"), M_gen=row.M, group_similar=group_similar)
    else:
        cls = vo.MidpointExpLinearSolver if row.scheme == "midpoint" else vo.ExpCFMSolver
        s = cls(*args, M_gen=row.M, group_similar=group_similar)
    if row.adaptive:
        s.with_tolerance(1e-7, 1e-7)
        if lst in EDGES:
            s.with_step_range(1e-6, 0.1)
    elif row.scheme != "blanes":
        s.no_adaptive()
    if row.opts.get("dynamic") if dynamic is None else dynamic:
        s.dynamic_grouping()
    if row.opts.get("gen"):
        s.set_generator(COS_BODY)
    if row.opts.get("norm"):
        s.with_norm(vo.NormFn(ctx, "m = e * e + im * im;", "sum", "r = sqrt(acc);"))
    ops = _ops(row.n)
    s.set_t_list(t_list).enable_snapshots().set_observables(ops)
    return s, t_list, ops


@functools.lru_cache(maxsize=None)
def _oracle(row_name, lst, upto=None, max_calls=0, N=None):
    """The oracle's run of the row on the list (cut after entry `upto` if given; `max_calls` calls per system if > 0), with snapshots
    and the event of every call."""
    import vecode_b200 as vo
    row = ROWS[row_name]
    basis, gp, psi0 = _inputs(vo, row, lst, N)
    t_list = list(LISTS[lst])
    if upto is not None:
        t_list = t_list[:upto + 1]
    cs, tables, scheme = None, None, row.scheme
    if scheme == "magnus42":
        basis, cs = _closed(basis)
    if scheme == "blanes":
        scheme, tables = "cfm_table", (BLANES_C, vo.cfm_table("BLANES17_R4_J4"), None)
    kw = dict(no_adaptive=True)
    if row.adaptive:
        kw = dict(adaptive=True, no_adaptive=False, rtol=1e-7, **(dict(min_dt=1e-6, max_dt=0.1) if lst in EDGES else {}))
    return tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, t_list[-1], _h0(row, lst), M_gen=row.M, cs=cs, t_list=t_list, snapshots=True,
                           events_cap=max_calls, max_calls=max_calls, tables=tables, n_threads=8, **kw)


def _ops(n, seed=7):
    """K = 3: a population-like diagonal, a random Hermitian and a random non-Hermitian operator (test_gpu_exp_observables.py's)."""
    rng = np.random.default_rng(seed + n)
    G = rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))
    return np.stack([np.diag(np.arange(n, dtype=float)).astype(complex) / max(n - 1, 1), (G + G.conj().T) / 2.0,
                     rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n))])


def _expect(ops, snap):
    """e[j][i][k] = sum_r conj(psi_r) sum_c O_k[r][c] psi_c and its rounding scale sum_rc |O_rc| |psi_r| |psi_c|, snap [len][N][n]."""
    e = np.einsum("jir,krc,jic->jik", snap.conj(), ops, snap)
    scale = np.einsum("jir,krc,jic->jik", np.abs(snap), np.abs(ops), np.abs(snap))
    return e, scale


def _h_close(got, ref, what):
    """h of an adaptive run. The controller's pow is correctly rounded on the device (pow_third_cr) and comes from libm in the oracle,
    which now and then rounds the other way; the next error estimate, a difference of two solutions that agree to about rtol,
    magnifies that ulp by about 1/rtol. A wrong h restored at an entry is off by a factor of 0.3 to 2."""
    rel = np.abs(got - ref) / np.abs(ref)
    print(f"{what}: h bit-identical for {np.mean(got == ref):.4f} of systems, max relative difference {rel.max():.2e}")
    _note("adaptive h, relative", rel.max())
    assert rel.max() <= 1e-6, (what, rel.max())


def _outputs(s, L):
    st = s.stats()
    return ([s.current()[1]] + [s.snapshot(k) for k in range(L)] + [s.expectation(k) for k in range(L)] +
            [st[k] for k in ("t", "h", "accepted", "rejected", "dx_norm")])


def _same(a, b):
    assert len(a) == len(b)
    for i, (u, v) in enumerate(zip(a, b)):
        assert np.array_equal(_bits(u), _bits(v)), i


def _check_against_the_oracle(s, counts, row, lst, t_list, ref, ops):
    N, L = s.N, len(t_list)
    stats = s.stats()
    assert counts["Chkpt"] == N * (L - 1) and counts["End"] == N
    assert counts["Step"] == int(ref["accepted"].sum()) and counts["Reject"] == int(ref["rejected"].sum())
    assert np.array_equal(stats["accepted"], ref["accepted"]) and np.array_equal(stats["rejected"], ref["rejected"])
    assert np.all(np.abs(stats["t"] - t_list[-1]) <= EPS)
    snaps = np.stack([s.snapshot(k) for k in range(L)])
    err = np.abs(snaps - ref["snap"]).max()
    _note(f"state error, {row.kind}", err)
    assert err <= 1e-12, err
    if row.adaptive:
        _h_close(stats["h"], ref["h"], "final h")
    else:
        assert np.array_equal(stats["t"], ref["t"]) and np.array_equal(stats["h"], ref["h"])
    assert np.array_equal(_bits(snaps[-1]), _bits(s.current()[1]))
    e = np.stack([s.expectation(j) for j in range(L)])
    err_e = np.abs(e - _expect(ops, ref["snap"])[0]).max()
    assert err_e <= 1e-12, err_e
    want, scale = _expect(ops, snaps)
    assert np.all(np.abs(e - want) <= 1e-13 * scale + 1e-300), np.abs(e - want).max()
    if lst in EDGES:
        z = ZERO_SYS
        assert np.all(snaps[:, z].view(np.float64) == 0.0) and np.all(e[:, z].view(np.float64) == 0.0)
        assert stats["h"][z] == ref["h"][z] and stats["t"][z] == ref["t"][z]


@pytest.mark.parametrize("row,lst", TABLE_CASES)
def test_table_against_the_oracle(vo, ctx, row, lst):
    """Every (row, list) of the table through run(): snapshots, counts, t, h and expectation values under the bars of the docstring."""
    r = ROWS[row]
    s, t_list, ops = _make(vo, ctx, r, lst)
    st = s.run(adaptive=r.adaptive)
    assert st.kind == "Done"
    _check_against_the_oracle(s, st.counts, r, lst, t_list, _oracle(row, lst), ops)


@pytest.mark.parametrize("row", ["S5-cfm4", "S5-cfm4a", "T40x2", "T40x2-cfm4a", "D24", "D24-a"])
def test_one_event_at_a_time_on_edge(vo, ctx, row):
    """EDGE one step() / step_adaptive() at a time: whenever a system sits on t_list[k], current() shows snapshot k bit for bit; the h it
    shows after its Chkpt / End there (the second time it is seen on t_list[k], the third for the second of two equal entries: the first
    is after the step that lands there, later ones may follow rejected attempts) is the final h of the oracle's solve whose list stops at
    entry k: bit for bit with fixed steps, within _h_close adaptive."""
    r = ROWS[row]
    s, t_list, ops = _make(vo, ctx, r, "EDGE")
    L, N = len(t_list), s.N
    want = np.zeros((L, N, r.n), dtype=complex)
    want_h = np.zeros((L, N))
    seen_at = np.zeros((L, N), dtype=int)
    rank = [1 + sum(t_list[j] == t_list[k] for j in range(k + 1)) for k in range(L)]

    def observe():
        st = s.stats()
        x = s.current()[1]
        for k, tk in enumerate(t_list):
            at = np.abs(st["t"] - tk) <= EPS
            want[k, at] = x[at]
            seen_at[k, at] += 1
            after = at & (seen_at[k] == rank[k])
            want_h[k, after] = st["h"][after]

    for _ in range(5000):
        observe()
        if (s.step_adaptive() if r.adaptive else s.step()).kind == "Done":
            break
    observe()
    assert np.all(seen_at >= np.array(rank)[:, None])
    for k in range(L):
        assert np.array_equal(_bits(s.snapshot(k)), _bits(want[k])), k
    assert np.array_equal(_bits(s.snapshot(4)), _bits(s.snapshot(5)))  # 4.2 twice
    for k in range(L):
        ref_h = _oracle(row, "EDGE", upto=k)["h"]
        if r.adaptive:
            _h_close(want_h[k], ref_h, f"h after entry {k}")
        else:
            assert np.array_equal(want_h[k], ref_h), k


@pytest.mark.parametrize("row", ["S5-cfm4", "T40x2", "D24"])
def test_rows_are_written_once(vo, ctx, row):
    """A fresh solver on EDGE with fixed steps, run(max_calls) in stages: after m calls the rows of the entries no system has reached
    are all-zero bytes, the rows reached equal the oracle stopped after the same m calls (1e-12), and rows written at an earlier
    stage keep their bits through the rest of the run."""
    r = ROWS[row]
    s, t_list, ops = _make(vo, ctx, r, "EDGE")
    L, done, kept = len(t_list), 0, {}
    for m in (1, 3, 4, 20, 36, 0):
        if m:
            s.run(max_calls=m - done)
            done = m
        else:
            assert s.run().kind == "Done"
        snaps = [s.snapshot(k) for k in range(L)]
        exps = [s.expectation(k) for k in range(L)]
        for k, (a, b) in kept.items():
            assert np.array_equal(_bits(snaps[k]), a) and np.array_equal(_bits(exps[k]), b), (m, k)
        if not m:
            break
        ref = _oracle(row, "EDGE", max_calls=m)
        ev = ref["events"][0]  # fixed steps: every system makes the same calls
        reached = int(np.sum((ev == tl.CHKPT) | (ev == tl.END)))
        assert np.all(ref["events"] == ev[None, :])
        assert np.array_equal(s.stats()["accepted"], ref["accepted"])
        assert np.abs(s.current()[1] - ref["psi"]).max() <= 1e-12
        for k in range(L):
            if k < reached:
                assert np.abs(snaps[k] - ref["snap"][k]).max() <= 1e-12, (m, k)
                assert np.abs(exps[k] - _expect(ops, ref["snap"][k:k + 1])[0][0]).max() <= 1e-12, (m, k)
                kept[k] = (_bits(snaps[k]).copy(), _bits(exps[k]).copy())
            else:
                assert not _bits(snaps[k]).any() and not _bits(exps[k]).any(), (m, k)
    assert set(kept) == {0, 1, 2}  # 0.2 twice and 3.0 reached by call 36: the rows the rest of the run must leave alone


@pytest.mark.parametrize("row", ["S2-cfm4a", "S7-cfm4a"])
def test_fused_run_equals_single_calls_on_edge(vo, ctx, row):
    """vo_exp_run fuses up to 16 events per launch of exp_small_kernel: the two Chkpt of the repeated entry 0.2 and the clipped one-ulp
    steps fall inside launches. Snapshots, expectations, state, t, h, counts, dx_norm and event totals: the bits of one
    step_adaptive() per call."""
    r = ROWS[row]
    out = []
    for fused in (True, False):
        s, t_list, _ = _make(vo, ctx, r, "EDGE")
        tot = dict(Step=0, Chkpt=0, Reject=0, End=0)
        launches = calls = 0
        while True:
            st = s.run(adaptive=True) if fused else s.step_adaptive()
            calls += 1
            launches += st.counts["launches"]
            for k in tot:
                tot[k] += st.counts[k]
            if st.kind == "Done":
                break
        out.append((_outputs(s, len(t_list)), tot, launches, calls))
    _same(out[0][0], out[1][0])
    assert out[0][1] == out[1][1]
    assert 4 * out[0][2] < out[1][3]  # several events per launch


@pytest.mark.parametrize("row", ["S5-cfm4", "T40x2", "D24"])
def test_callers_order_on_edge(vo, ctx, row):
    """group_similar (vo_exp_set_order) and, on the tiles, dynamic grouping, on EDGE with N = 77: snapshots, expectations, state and
    stats come back in the caller's order, equal to the plain-order run (bit for bit on the per-system kernels, 1e-13 on the tiles,
    whose tiles then hold other systems); the device views hold the host rows."""
    r = ROWS[row]
    N = 77
    variants = [(False, False), (True, False)] + ([(True, True), (False, True)] if r.kind == "tile" else [])
    res = []
    for gs, dyn in variants:
        s, t_list, _ = _make(vo, ctx, r, "EDGE", N=N, group_similar=gs, dynamic=dyn)
        if gs:
            assert s._perm is not None and not np.array_equal(s._perm, np.arange(N))
        assert s.run().kind == "Done"
        res.append(_outputs(s, len(t_list)))
        for k in (1, 4, 8):
            dev = s.snapshot_ensemble(k).to_host().reshape(-1).view(np.complex128).reshape(N, -1)
            assert np.array_equal(_bits(dev), _bits(s.snapshot(k)))
            dev = s.expectation_ensemble(k).to_host().reshape(-1).view(np.complex128).reshape(N, 3)
            assert np.array_equal(_bits(dev), _bits(s.expectation(k)))
    for other in res[1:]:
        if r.kind == "tile":
            for a, b in zip(other[:-5], res[0][:-5]):
                assert np.abs(a - b).max() <= 1e-13
            for a, b in zip(other[-5:-1], res[0][-5:-1]):  # t, h, accepted, rejected: fixed steps
                assert np.array_equal(a, b)
        else:
            _same(other, res[0])


@pytest.mark.parametrize("row", ["S3-cfm4a", "T16x2-cfm4a"])
def test_fixed_then_adaptive_in_mid_list(vo, ctx, row):
    """step() through entry 2 of L9, then run(adaptive=True) to the end: every snapshot within 1e-12 of the pure-Python restatement
    switched at the same call (_exp_tlist.solve(adaptive_from=...)), with equal accepted and rejected counts."""
    from oracle import exp_oracle as eo
    r = ROWS[row]
    s, t_list, _ = _make(vo, ctx, r, "L9")
    N = s.N
    chk = calls = 0
    while chk < 3 * N:
        chk += s.step().counts["Chkpt"]
        calls += 1
    assert s.run(adaptive=True).kind == "Done"
    basis, gp, psi0 = _inputs(vo, r, "L9")
    sp = eo.BasisSplit([[[(z.real, z.imag) for z in b_row] for b_row in B] for B in basis])
    stats = s.stats()
    snaps = np.stack([s.snapshot(k) for k in range(len(t_list))])
    for i in (range(N) if r.kind == "small" else (0, 12, 36)):
        py = tl.solve("cfm4", sp, [tuple(v) for v in gp[i]], r.M, [(z.real, z.imag) for z in psi0[i]], 0.0, 1.0, _h0(r, "L9"),
                      t_list=t_list, rtol=1e-7, adaptive_from=calls)
        assert (stats["accepted"][i], stats["rejected"][i]) == (py["accepted"], py["rejected"]), i
        for k in range(len(t_list)):
            want = np.array([complex(a, b) for a, b in py["snap"][k]])
            assert np.abs(snaps[k, i] - want).max() <= 1e-12, (i, k)


# ---- the earlier cases -------------------------------------------------------------------------------------------------------------

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
        H0 = np.diag((k - (n - 1) / 2) * 0.3) + np.diag(np.full(n - 1, 0.5), 1) + np.diag(np.full(n - 1, 0.5), -1) if n > 1 else np.array([[0.4]])
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
