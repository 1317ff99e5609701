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
