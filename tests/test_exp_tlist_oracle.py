"""Output times (ODEData.t_list, ode.rs:89) in the two CPU restatements of the exponential integrators (tests/_exp_tlist.py): the
C++ oracle's solver loop and the pure-Python schemes of oracle/exp_oracle.py take a list in place of [t0, tf], clip steps to land on
every entry, raise Chkpt / End there and keep the state of each system at each of those events. They must agree bit for bit with each
other, and the default list must reproduce what the oracles compute without a list. Also: the device sources that carry the list
compile without a GPU."""
import importlib.util
import json
import os

import numpy as np
import pytest

import _exp_tlist as tl
from oracle import exp_oracle as eo

HERE = os.path.dirname(os.path.abspath(__file__))
# five entries, two of them (0.13, 0.77) off the grid of h = 0.1 and one (0.5) on it
T_LIST = [0.0, 0.13, 0.5, 0.77, 1.0]
STEP, CHKPT, REJECT, END = 0, 1, 2, 3


def _golden():
    spec = importlib.util.spec_from_file_location("make_golden_exp", os.path.join(HERE, "golden", "make_golden_exp.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, json.load(open(os.path.join(HERE, "golden", "exp_known_answers.json")))


def _case(scheme, n=4, seed=31):
    mod, _ = _golden()
    basis, gp, psi0 = mod.case(n, 2, seed)
    cs = None
    if scheme == "magnus42":  # a third basis slot holds [B_0, B_1]: the structure tensor closes magnus_42's one commutator
        basis = np.concatenate([basis, (basis[0] @ basis[1] - basis[1] @ basis[0])[None]])
        cs = np.zeros((3, 3, 3))
        cs[0, 1, 2], cs[1, 0, 2] = 1.0, -1.0
    return basis, gp, psi0, cs, mod.py_split(basis)


def _c(x):
    return np.array([complex(a, b) for a, b in x])


CASES = [("midpoint", False), ("cfm4", False), ("cfm4", True), ("magnus42", False), ("magnus42", True)]


@pytest.mark.parametrize("scheme,adaptive", CASES)
def test_tlist_cpp_equals_pure_python_bitwise(oracle, scheme, adaptive):
    """States, snapshots, (accepted, rejected) and the event of every call: the same bits from both restatements."""
    basis, gp, psi0, cs, sp = _case(scheme)
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-7) if adaptive else dict(no_adaptive=True)
    cap = 400
    ref = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 1.0, 0.1, M_gen=2, cs=cs, t_list=T_LIST, snapshots=True, events_cap=cap, **kw)
    for i in range(psi0.shape[0]):
        py = tl.solve(scheme, sp, [tuple(r) for r in gp[i]], 2, [(z.real, z.imag) for z in psi0[i]], 0.0, 1.0, 0.1, t_list=T_LIST,
                      adaptive=adaptive, rtol=1e-7, cs=None if cs is None else cs.tolist())
        assert np.array_equal(_c(py["x"]).view(np.float64), ref["psi"][i].view(np.float64)), i
        assert (py["accepted"], py["rejected"]) == (ref["accepted"][i], ref["rejected"][i])
        assert py["t"] == ref["t"][i] and py["h"] == ref["h"][i]
        ev = ref["events"][i]
        assert len(py["events"]) < cap and list(ev[:len(py["events"])]) == py["events"] and np.all(ev[len(py["events"]):] == -1)
        assert py["events"].count(CHKPT) == len(T_LIST) - 1 and py["events"][-1] == END
        if not adaptive:
            assert REJECT not in py["events"]
        for k in range(len(T_LIST)):
            assert np.array_equal(_c(py["snap"][k]).view(np.float64), ref["snap"][k, i].view(np.float64)), (i, k)
        assert np.array_equal(ref["snap"][0, i], psi0[i])  # entry 0 is t0: the initial state, before any step
    assert np.array_equal(ref["snap"][-1], ref["psi"])
    if adaptive:
        assert ref["rejected"].sum() > 0


@pytest.mark.parametrize("scheme,adaptive", CASES)
def test_snapshot_k_is_the_solve_that_stops_at_entry_k(oracle, scheme, adaptive):
    """Snapshot k of the 5-entry solve is the final state of the solve whose list ends at entry k, with the same counts up to there."""
    basis, gp, psi0, cs, _ = _case(scheme, n=3, seed=33)
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-7) if adaptive else dict(no_adaptive=True)
    full = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 1.0, 0.1, M_gen=2, cs=cs, t_list=T_LIST, snapshots=True, **kw)
    for k in range(1, len(T_LIST)):
        part = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 1.0, 0.1, M_gen=2, cs=cs, t_list=T_LIST[:k + 1], **kw)
        assert np.array_equal(part["psi"].view(np.float64), full["snap"][k].view(np.float64)), k
        assert np.all(np.abs(part["t"] - T_LIST[k]) <= 2.0 ** -52), k


@pytest.mark.parametrize("scheme,adaptive", CASES)
def test_default_list_is_unchanged(oracle, scheme, adaptive):
    """t_list = [t0, tf] given explicitly computes what the solvers computed without a list, in both restatements."""
    basis, gp, psi0, cs, sp = _case(scheme, n=3, seed=35)
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-6) if adaptive else dict(no_adaptive=True)
    a = oracle.exp_ensemble(scheme, basis, gp, psi0, 0.0, 0.9, 0.1, M_gen=2, cs=cs, **kw)
    b = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 0.9, 0.1, M_gen=2, cs=cs, t_list=[0.0, 0.9], snapshots=True, **kw)
    for key in ("psi", "t", "h", "accepted", "rejected"):
        assert np.array_equal(np.asarray(a[key]).view(np.uint8), np.asarray(b[key]).view(np.uint8)), key
    assert np.array_equal(b["snap"][0], psi0) and np.array_equal(b["snap"][1], b["psi"])
    if not adaptive:  # the pure-Python driver with the default list against its fixed-step loop
        for i in range(psi0.shape[0]):
            x0 = [(z.real, z.imag) for z in psi0[i]]
            py = tl.solve(scheme, sp, [tuple(r) for r in gp[i]], 2, x0, 0.0, 1.0e9, 0.1, max_calls=7, cs=None if cs is None else cs.tolist())
            fx = eo.solve_fixed(scheme, sp, [tuple(r) for r in gp[i]], 2, x0, 0.0, 0.1, 6, cs=None if cs is None else cs.tolist())
            assert py["x"] == fx and py["events"] == [CHKPT] + [STEP] * 6  # t0 is entry 0: the first call is its checkpoint


def test_default_list_reproduces_the_golden_fixture(oracle):
    """tests/golden/exp_known_answers.json through an explicit [t0, tf] list: the committed states, bit for bit."""
    mod, G = _golden()
    s15 = np.sqrt(15.0) / 10.0
    for key, e in G.items():
        if key.startswith("_"):
            continue
        basis, gp, psi0 = mod.case(e["n"], e["M"], e["seed"])
        cs, tables = None, None
        if e["scheme"] == "magnus42":
            basis = np.concatenate([basis, (basis[0] @ basis[1] - basis[1] @ basis[0])[None]])
            cs = np.zeros((3, 3, 3))
            cs[0, 1, 2], cs[1, 0, 2] = 1.0, -1.0
        if e["scheme"] == "cfm_table":
            tables = ([0.5 - s15, 0.5, 0.5 + s15], eo.BLANES17_R4_J4, None)
        ref = tl.exp_ensemble(e["scheme"], basis, gp, psi0, 0.0, 1.0e9, e["h"], M_gen=e["M"], cs=cs, no_adaptive=True, max_calls=e["steps"] + 1,
                              tables=tables, t_list=[0.0, 1.0e9], events_cap=e["steps"] + 2)
        want = np.array(e["psi"]).reshape(psi0.shape[0], e["n"], 2)
        assert np.array_equal(ref["psi"].view(np.float64).reshape(want.shape), want), key
        ev = ref["events"]
        assert np.all(ev[:, 0] == CHKPT) and np.all(ev[:, 1:e["steps"] + 1] == STEP) and np.all(ev[:, -1] == -1), key


@pytest.mark.parametrize("n", [2, 8, 16, 64])
def test_checkpoint_kernels_compile_without_a_gpu(vo, n):
    """The kernels that read the list and write the snapshots, compiled at run time with a user generator and with a user norm."""
    assert vo.ExpCFMSolver.check_generator("g[1] = p[0] * cos(p[1] * t + p[2]);", n, 2) > 5_000
    assert vo.NormFn.check_kernels("m = e * e + im * im;", "sum", "r = sqrt(acc);", exp_n=n, exp_M=2) > 5_000


# the edge lists of tests/test_gpu_exp_checkpoints.py, absolute times, h = 0.1: a first entry after t0, 0.2 twice, 4.2 / 4.25 / 4.3
# closer together than h, and 3.0 -> 3.3 -> 4.2, 4.3 -> 4.5 in full steps whose sum falls one ulp short of the entry (a clipped
# step of one ulp follows). EDGE8 (8 entries) is held inline in the launch parameters, EDGE (9) is read from device memory.
EDGE8 = [0.2, 0.2, 3.0, 3.3, 4.2, 4.25, 4.3, 4.5]
EDGE = [0.2, 0.2, 3.0, 3.3, 4.2, 4.2, 4.25, 4.3, 4.5]
ONE = [1.0]
EDGE_LISTS = {"EDGE8": EDGE8, "EDGE": EDGE, "ONE": ONE}
# adaptive runs on the edge lists: the step capped at h = 0.1 so that slow systems walk the same grid; the solvers' initial step is then
# sqrt(min_dt max_dt) (vo_exp_with_step_range, ode.rs:273-280)
EDGE_RANGE = dict(min_dt=1e-6, max_dt=0.1)
EDGE_H0 = float(np.sqrt(1e-6 * 0.1))


def _with_zero_state(psi0):
    """The ensemble plus one system that starts at psi = 0: its embedded error is exactly 0, so f = rtol / 0 = inf."""
    return np.concatenate([psi0, np.zeros((1, psi0.shape[1]), complex)])


@pytest.mark.parametrize("scheme,adaptive", CASES)
@pytest.mark.parametrize("lst", list(EDGE_LISTS))
def test_edge_lists_cpp_equals_pure_python_bitwise(oracle, scheme, adaptive, lst):
    """EDGE8, EDGE and ONE with a zero-state system: both restatements give the same bits of states, snapshots, t, h, counts and
    events. The zero-state system keeps exact zeros and, adaptive, takes the controller's largest growth at every step."""
    basis, gp, psi0, cs, sp = _case(scheme)
    psi0 = _with_zero_state(psi0)
    gp = np.concatenate([gp, gp[:1]])
    t_list = EDGE_LISTS[lst]
    kw = dict(adaptive=True, no_adaptive=False, rtol=1e-7, **EDGE_RANGE) if adaptive else dict(no_adaptive=True)
    h = EDGE_H0 if adaptive else 0.1
    cap = 2000
    ref = tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, t_list[-1], h, M_gen=2, cs=cs, t_list=t_list, snapshots=True, events_cap=cap, **kw)
    for i in range(psi0.shape[0]):
        py = tl.solve(scheme, sp, [tuple(r) for r in gp[i]], 2, [(z.real, z.imag) for z in psi0[i]], 0.0, t_list[-1], h, t_list=t_list,
                      adaptive=adaptive, rtol=1e-7, cs=None if cs is None else cs.tolist(), **(EDGE_RANGE if adaptive else {}))
        assert np.array_equal(_c(py["x"]).view(np.float64), ref["psi"][i].view(np.float64)), i
        assert (py["accepted"], py["rejected"]) == (ref["accepted"][i], ref["rejected"][i])
        assert py["t"] == ref["t"][i] and py["h"] == ref["h"][i]
        ev = ref["events"][i]
        assert len(py["events"]) < cap and list(ev[:len(py["events"])]) == py["events"]
        assert py["events"].count(CHKPT) == len(t_list) - 1 and py["events"].count(END) == 1 and py["events"][-1] == END
        assert py["events"][0] == STEP  # the first entry lies after t0
        for k in range(len(t_list)):
            assert np.array_equal(_c(py["snap"][k]).view(np.float64), ref["snap"][k, i].view(np.float64)), (i, k)
        assert abs(py["t"] - t_list[-1]) <= 2.0 ** -52
    z = ref["snap"][:, -1]
    assert np.all(z.view(np.float64) == 0.0) and np.all(ref["psi"][-1].view(np.float64) == 0.0)
    if lst != "ONE":
        assert np.array_equal(ref["snap"][0], ref["snap"][1])  # 0.2 twice: two Chkpt with no step between them
    if adaptive:
        assert ref["rejected"][-1] == 0 and ref["h"][-1] == 0.1  # f = inf: factor 2 at every step, up to max_dt


def test_edge_list_takes_one_ulp_steps():
    """On EDGE with fixed h = 0.1 the full steps to 3.0, 4.2 and 4.5 fall one ulp short: each of those entries is reached by a clipped step
    of less than 1e-14, directly before its Chkpt / End. Without these the edge list would not test the clipped step it claims to."""
    basis, gp, psi0, cs, sp = _case("cfm4")
    py = tl.solve("cfm4", sp, [tuple(r) for r in gp[0]], 2, [(z.real, z.imag) for z in psi0[0]], 0.0, 4.5, 0.1, t_list=EDGE)
    ev, dt = py["events"], py["dt"]
    tiny = [j for j in range(len(ev)) if ev[j] == STEP and 0.0 < dt[j] < 1e-14]
    assert len(tiny) >= 2, tiny
    assert all(ev[j + 1] in (CHKPT, END) for j in tiny)
    # the step before each is a full one
    assert all(dt[j - 1] == 0.1 for j in tiny)


@pytest.mark.parametrize("scheme", ["cfm4", "magnus42"])
def test_switch_to_adaptive_in_mid_list(oracle, scheme):
    """solve(adaptive_from=c): step() for the first c calls, step_adaptive() after. From call 0 it is the C++ adaptive run bit for bit,
    never (a switch past the last call) the fixed run; a switch after entry 2 of a 9-entry list keeps the fixed run's bits up to entry 2,
    then runs the controller (rejections, other step counts) to the end of the list."""
    basis, gp, psi0, cs, sp = _case(scheme)
    L9 = [0.0, 0.0611, 0.1937, 0.3, 0.4226, 0.55, 0.7123, 0.8377, 1.0]
    cap = 400
    ref = {a: tl.exp_ensemble(scheme, basis, gp, psi0, 0.0, 1.0, 0.1, M_gen=2, cs=cs, t_list=L9, snapshots=True, events_cap=cap,
                              **(dict(adaptive=True, no_adaptive=False, rtol=1e-7) if a else dict(no_adaptive=False)))
           for a in (False, True)}
    csl = None if cs is None else cs.tolist()
    for i in range(psi0.shape[0]):
        args = (scheme, sp, [tuple(r) for r in gp[i]], 2, [(z.real, z.imag) for z in psi0[i]], 0.0, 1.0, 0.1)
        fixed = tl.solve(*args, t_list=L9, rtol=1e-7, cs=csl)
        for c, a in ((0, True), (len(fixed["events"]) + 1, False)):
            py = tl.solve(*args, t_list=L9, rtol=1e-7, cs=csl, adaptive_from=c)
            r = ref[a]
            assert np.array_equal(_c(py["x"]).view(np.float64), r["psi"][i].view(np.float64)), (i, c)
            assert (py["accepted"], py["rejected"], py["t"], py["h"]) == (r["accepted"][i], r["rejected"][i], r["t"][i], r["h"][i])
            assert py["events"] == list(r["events"][i][:len(py["events"])])
        c = [j for j, e in enumerate(fixed["events"]) if e == CHKPT][2] + 1  # the call after entry 2's Chkpt
        py = tl.solve(*args, t_list=L9, rtol=1e-7, cs=csl, adaptive_from=c)
        assert py["events"][:c] == fixed["events"][:c]
        for k in range(3):
            assert py["snap"][k] == fixed["snap"][k], (i, k)
        assert py["events"].count(CHKPT) == len(L9) - 1 and py["events"][-1] == END
        assert py["accepted"] != fixed["accepted"] and abs(py["t"] - 1.0) <= 2.0 ** -52
