"""Host-side mirror of vec-ode's exponential integrators (src/exp) over the C ABI.

  ExponentialSplit / Commutator / NormedExponentialSplit   src/exp/mod.rs:11-54   -> DenseBasisSplit
  MidpointExpLinearSolver                                  src/exp/magnus.rs:85-148
  MagnusExpLinearSolver                                    src/exp/magnus.rs:151-285
  ExpCFMSolver                                             src/exp/cfm.rs:102-224

The reference leaves exp / map_exp / commutator / norm to the user; `DenseBasisSplit` is the implementation this engine
ships: operators L_i = sum_m coef[i][m] B_m on M complex n x n matrices shared by the ensemble, exp lazy, map_exp a scaled
Taylor series applied to the state on the FP64 tensor cores. The generator closure `f(&[t]) -> Vec<L>` is replaced by the
built-in family L_i(t) = B_0 + sum_{m>=1} amp_im cos(omega_im t + phase_im) B_m (`gp[i][m-1] = (amp, omega, phase)`).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _cabi
from ._cabi import StepResult, check, lib
from .base import Context, ODEState, _np_ptr, _state_of

_vp = C.c_void_p


class DenseBasisSplit:
    """ExponentialSplit (+ Commutator, NormedExponentialSplit) for batched dense complex systems on a shared basis.

    `basis`: [M][n][n] complex, 1 <= M <= 4, with 1 <= n <= 8 (qubits, qutrits, few-qubit registers: one system per GPU thread in
    FP64 registers, each with its own Taylor plan; vo_exp_run fuses several events per launch) or n a multiple of 8 (16 to 64 on the
    FP64 tensor cores, by tiles of 16 systems). 9 <= n <= 15 is refused."""

    def __init__(self, ctx: Context, basis, commutator_structure=None, taylor_degree: int = 0):
        basis = np.ascontiguousarray(basis, dtype=np.complex128)
        self.M, self.n = basis.shape[0], basis.shape[1]
        self.norm1 = np.abs(basis).sum(axis=1).max(axis=1)  # induced 1-norm of each basis matrix (the bound behind the Taylor plan)
        self.ctx = ctx
        self.cs = None
        self._h = _vp()
        check(lib().vo_split_basis_create(ctx._h, self.n, self.M, _np_ptr(basis.view(np.float64)), C.byref(self._h)), ctx._h)
        if commutator_structure is not None:
            cs = np.ascontiguousarray(commutator_structure, dtype=np.float64)
            assert cs.shape == (self.M,) * 3
            check(lib().vo_split_set_commutator(self._h, _np_ptr(cs)), ctx._h)
            self.cs = cs
        if taylor_degree:
            check(lib().vo_split_set_taylor_degree(self._h, taylor_degree), ctx._h)

    # ExponentialSplit ---------------------------------------------------------------------------------------------
    def lin_zero(self, n_systems: int) -> np.ndarray:  # exp/mod.rs:20
        return np.zeros((n_systems, self.M), dtype=np.complex128)

    def exp(self, l: np.ndarray) -> np.ndarray:  # exp/mod.rs:23 — lazy: U is L
        return l

    def map_exp(self, u: np.ndarray, psi_dev_in: int, psi_dev_out: int):  # exp/mod.rs:25
        u = np.ascontiguousarray(u, dtype=np.complex128)
        check(lib().vo_map_exp(self._h, _np_ptr(u.view(np.float64)), u.shape[0], _vp(psi_dev_in), _vp(psi_dev_out)), self.ctx._h)

    def multi_exp(self, l: np.ndarray, k_arr):  # exp/mod.rs:28-34
        return [self.exp(l * k) for k in k_arr]

    # Commutator (exp/mod.rs:47-54) on coefficient vectors ---------------------------------------------------------------
    def commutator(self, la: np.ndarray, lb: np.ndarray) -> np.ndarray:
        la, lb = np.ascontiguousarray(la, dtype=np.complex128), np.ascontiguousarray(lb, dtype=np.complex128)
        out = np.empty_like(la)
        check(lib().vo_split_commutator(self._h, _np_ptr(la.view(np.float64)), _np_ptr(lb.view(np.float64)), la.shape[0], _np_ptr(out.view(np.float64))),
              self.ctx._h)
        return out

    # NormedExponentialSplit::norm (exp/mod.rs:37-45) -------------------------------------------------------------------
    def norm(self, psi_dev: int, n_systems: int) -> np.ndarray:
        out = np.empty(n_systems)
        check(lib().vo_split_norm(self._h, _vp(psi_dev), n_systems, _np_ptr(out)), self.ctx._h)
        return out

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().vo_split_destroy(self._h)
        except Exception:
            pass


class DenseSplit:
    """ExponentialSplit + Commutator + NormedExponentialSplit (src/exp/mod.rs:11-54) for GENERAL dense operators: every one of the
    N systems owns its n x n complex `L` and its explicit `U = exp(L)` (vo_split_dense_*). Operators are `Ensemble`s of one row of
    2 n^2 N doubles ([N][n][n] complex, row-major), so `LinearCombination` applies to them as to any other ensemble."""

    def __init__(self, ctx: Context, n: int, n_systems: int):
        self.ctx, self.n, self.N = ctx, n, n_systems
        self._h = _vp()
        check(lib().vo_split_dense_create(ctx._h, n, n_systems, C.byref(self._h)), ctx._h)

    def _new(self):
        from .base import Ensemble
        return Ensemble(self.ctx, 1, 2 * self.n * self.n * self.N)

    def operator(self, mats: np.ndarray):
        """[N][n][n] complex host array -> operator ensemble"""
        m = np.ascontiguousarray(mats, dtype=np.complex128)
        assert m.shape == (self.N, self.n, self.n)
        e = self._new()
        e.upload(m.view(np.float64).reshape(1, -1), "soa")
        return e

    def to_host(self, op) -> np.ndarray:
        return op.to_host("soa").reshape(-1).view(np.complex128).reshape(self.N, self.n, self.n)

    def lin_zero(self):  # exp/mod.rs:20
        from .base import Ensemble
        h = _vp()
        check(lib().vo_dense_lin_zero(self._h, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, 1, 2 * self.n * self.n * self.N, _handle=h)

    def from_basis(self, basis_split: "DenseBasisSplit", coef: np.ndarray):
        """L_i = sum_m coef[i][m] B_m as a dense operator ensemble (vo_dense_assemble)"""
        coef = np.ascontiguousarray(coef, dtype=np.complex128)
        out = self._new()
        check(lib().vo_dense_assemble(self._h, basis_split._h, _np_ptr(coef.view(np.float64)), out._h), self.ctx._h)
        return out

    def exp(self, l):  # exp/mod.rs:23 — explicit U
        u = self._new()
        check(lib().vo_dense_exp(self._h, l._h, u._h), self.ctx._h)
        return u

    def multi_exp(self, l, k_arr):  # exp/mod.rs:28-34
        ks = np.ascontiguousarray(k_arr, dtype=np.float64)
        us = [self._new() for _ in ks]
        hs = (C.c_void_p * len(us))(*[u._h.value for u in us])
        check(lib().vo_dense_multi_exp(self._h, l._h, _np_ptr(ks), len(us), hs), self.ctx._h)
        return us

    def map_exp(self, u, psi_dev_in: int, psi_dev_out: int):  # exp/mod.rs:25
        check(lib().vo_dense_map_exp(self._h, u._h, _vp(psi_dev_in), _vp(psi_dev_out)), self.ctx._h)

    def commutator(self, la, lb):  # exp/mod.rs:53
        out = self._new()
        check(lib().vo_dense_commutator(self._h, la._h, lb._h, out._h), self.ctx._h)
        return out

    def norm(self, psi_dev: int, n_systems: Optional[int] = None) -> np.ndarray:  # exp/mod.rs:37-45
        n_systems = self.N if n_systems is None else n_systems
        out = np.empty(n_systems)
        check(lib().vo_split_norm(self._h, _vp(psi_dev), n_systems, _np_ptr(out)), self.ctx._h)
        return out

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().vo_split_destroy(self._h)
        except Exception:
            pass


def with_commutator_slot(B0: np.ndarray, B1: np.ndarray):
    """Basis (B0, B1, [B0, B1]) and the structure tensor that closes ONE commutator of two generators from span{B0, B1}
    (all that magnus_42 takes, exp/magnus.rs:55)."""
    comm = B0 @ B1 - B1 @ B0
    cs = np.zeros((3, 3, 3))
    cs[0, 1, 2], cs[1, 0, 2] = 1.0, -1.0
    return np.stack([B0, B1, comm]), cs


def _checked_out(out, shape, what):
    """A caller's output buffer that the C ABI fills with shape[0] * shape[1] complex numbers: exactly that, contiguous."""
    if not isinstance(out, np.ndarray) or out.dtype != np.complex128 or out.shape != shape or not out.flags.c_contiguous:
        raise _cabi.VecOdeError(_cabi.VO_ERR_SHAPE, f"{what}: `out` must be a C-contiguous complex128 array of shape {shape}")
    return out


class _ExpSolver:
    SCHEME = None

    def __init__(self, sp: DenseBasisSplit, gp, t0: float, tf: float, psi0, h: float, M_gen: Optional[int] = None, group_similar: bool = False):
        """`group_similar`: hand the systems to the device ordered by drive amplitude. A tile of 16 systems runs the largest
        Taylor degree among them (the plan is tile-uniform), so tiles of similar ||L h|| waste fewer terms: ~5 % on config 5.
        The systems are independent, so the order is free; current() / stats() / reset() keep the caller's order
        (vo_exp_set_order: the reordering runs on the device; only `state_device_ptr` shows the device order)."""
        self.sp, self.ctx = sp, sp.ctx
        psi0 = np.ascontiguousarray(psi0, dtype=np.complex128)
        self.N, self.n = psi0.shape
        self.M_gen = sp.M if M_gen is None else M_gen
        gp = np.ascontiguousarray(gp, dtype=np.float64).reshape(self.N, max(self.M_gen - 1, 0), 3)
        self._perm = None
        self._n_obs = 0  # operators of set_observables
        if group_similar and self.M_gen > 1:
            key = (np.abs(gp[:, :, 0]) * sp.norm1[1:self.M_gen][None, :]).sum(axis=1)
            self._perm = np.ascontiguousarray(np.argsort(key, kind="stable"), dtype=np.int64)
            gp, psi0 = np.ascontiguousarray(gp[self._perm]), np.ascontiguousarray(psi0[self._perm])  # once, at construction
        self._h = _vp()
        check(lib().vo_exp_create(self.ctx._h, sp._h, _cabi.EXP_SCHEME[self.SCHEME], self.M_gen, _np_ptr(gp), self.N, t0, tf,
                                  _np_ptr(psi0.view(np.float64)), h, C.byref(self._h)), self.ctx._h)
        if self._perm is not None:  # from here on the C ABI speaks the caller's order (the reordering runs on the device)
            check(lib().vo_exp_set_order(self._h, _np_ptr(self._perm), self.N), self.ctx._h)

    def dynamic_grouping(self, on: bool = True):
        """Sort the systems by the norm bound of their exponent before every event, on the device, so that each 16-system tile runs the
        Taylor degree its systems need (vo_exp_set_dynamic_grouping)."""
        check(lib().vo_exp_set_dynamic_grouping(self._h, 1 if on else 0), self.ctx._h)
        return self

    def set_generator(self, body: str):
        """The generator closure itself (`FnMut(T) -> L`, exp/cfm.rs:54, exp/magnus.rs:12,32): CUDA C++ statements assigning
        `g[1] .. g[M_gen-1]` of L(t) = B_0 + sum_m g[m] B_m from `t` and this system's parameter row `p` (the 3 (M_gen - 1)
        doubles of `gp`); compiled at run time into the same tensor-core kernel (vo_exp_set_generator)."""
        check(lib().vo_exp_set_generator(self._h, body.encode()), self.ctx._h)
        return self

    @staticmethod
    def check_generator(body: str, n: int, M: int) -> int:
        """Compile `body` without a GPU; returns the cubin size or raises VecOdeError carrying the compiler log."""
        log = C.create_string_buffer(1 << 16)
        rc = lib().vo_exp_generator_check(body.encode(), n, M, log, len(log))
        if rc < 0:
            raise _cabi.VecOdeError(rc, log.value.decode("utf-8", "replace"))
        return rc

    def with_norm(self, norm_fn):
        """ExpCFMSolver's NormFn closure / NormedExponentialSplit::norm (exp/cfm.rs:105, 214-216, exp/mod.rs:37-45) as a
        user-defined base.NormFn: the DMMA kernel is re-compiled with it (vo_exp_set_norm_custom)."""
        check(lib().vo_exp_set_norm_custom(self._h, norm_fn._h), self.ctx._h)
        self._norm_fn = norm_fn
        return self

    def no_adaptive(self):  # exp/cfm.rs:157-161
        check(lib().vo_exp_no_adaptive(self._h), self.ctx._h)
        return self

    def with_tolerance(self, atol: float, rtol: float):
        check(lib().vo_exp_with_tolerance(self._h, atol, rtol), self.ctx._h)
        return self

    def with_step_range(self, dt_min: float, dt_max: float):
        check(lib().vo_exp_with_step_range(self._h, dt_min, dt_max), self.ctx._h)
        return self

    def set_t_list(self, t_list):
        """Output times (ODEData.t_list, ode.rs:89) in place of [t0, tf]: every system raises Chkpt at each entry before the last
        and End at the last (vo_exp_set_t_list). Before the first step, or after reset()."""
        tl = np.ascontiguousarray(t_list, dtype=np.float64).ravel()
        check(lib().vo_exp_set_t_list(self._h, _np_ptr(tl), tl.size), self.ctx._h)
        return self

    def enable_snapshots(self):
        """Keep every system's state at its Chkpt / End event for each entry of t_list (vo_exp_enable_snapshots)."""
        check(lib().vo_exp_enable_snapshots(self._h), self.ctx._h)
        return self

    def snapshot(self, k: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        """The states at t_list[k], [N][n] complex in the caller's order (vo_exp_snapshot)."""
        psi = np.empty((self.N, self.n), dtype=np.complex128) if out is None else _checked_out(out, (self.N, self.n), "snapshot")
        check(lib().vo_exp_snapshot(self._h, k, _np_ptr(psi.view(np.float64))), self.ctx._h)
        return psi

    def snapshot_ensemble(self, k: int):
        """Snapshot k as a device-side Ensemble view (one row of 2 n N doubles, the caller's order), for `Group.gather_placed`."""
        from .base import Ensemble, _TensorOwner
        h = _vp()
        check(lib().vo_exp_snapshot_device(self._h, k, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, 1, 2 * self.n * self.N, _handle=h, _owner=_TensorOwner(self))

    def set_observables(self, ops):
        """Expectation values <psi| O_k |psi> (complex, not normalised) of every system at each entry of t_list, computed in the
        kernels at the Chkpt / End event (vo_exp_set_observables). `ops`: one n x n matrix or [K][n][n], 1 <= K <= 8, shared by the
        ensemble; None turns them off. Before the first step, or after reset()."""
        if ops is None:
            check(lib().vo_exp_set_observables(self._h, 0, None), self.ctx._h)
            self._n_obs = 0
            return self
        a = np.asarray(ops, dtype=np.complex128)
        if a.ndim == 2:
            a = a[None]
        if a.ndim != 3 or a.shape[1:] != (self.n, self.n):
            raise _cabi.VecOdeError(_cabi.VO_ERR_SHAPE, f"set_observables: operators must be [K][{self.n}][{self.n}], got {a.shape}")
        a = np.ascontiguousarray(a)
        check(lib().vo_exp_set_observables(self._h, a.shape[0], _np_ptr(a.view(np.float64))), self.ctx._h)
        self._n_obs = a.shape[0]
        return self

    def expectation(self, j: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        """<psi| O_k |psi> at t_list[j], [N][K] complex in the caller's order (vo_exp_expectation)."""
        e = np.empty((self.N, max(self._n_obs, 1)), dtype=np.complex128) if out is None else _checked_out(out, (self.N, self._n_obs), "expectation")
        check(lib().vo_exp_expectation(self._h, j, _np_ptr(e.view(np.float64))), self.ctx._h)
        return e

    def expectation_ensemble(self, j: int):
        """Expectation values at t_list[j] as a device-side Ensemble view (one row of 2 K N doubles, the caller's order)."""
        from .base import Ensemble, _TensorOwner
        h = _vp()
        check(lib().vo_exp_expectation_device(self._h, j, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, 1, 2 * self._n_obs * self.N, _handle=h, _owner=_TensorOwner(self))

    def step(self) -> ODEState:
        res = StepResult()
        check(lib().vo_exp_step(self._h, C.byref(res)), self.ctx._h)
        return _state_of(res)

    def step_adaptive(self) -> ODEState:
        res = StepResult()
        check(lib().vo_exp_step_adaptive(self._h, C.byref(res)), self.ctx._h)
        return _state_of(res)

    def run(self, adaptive: bool = False, max_calls: int = 0) -> ODEState:
        res = StepResult()
        check(lib().vo_exp_run(self._h, 1 if adaptive else 0, max_calls, C.byref(res)), self.ctx._h)
        return _state_of(res)

    def current(self, out: Optional[np.ndarray] = None):
        tmin, tmax = C.c_double(), C.c_double()
        psi = np.empty((self.N, self.n), dtype=np.complex128) if out is None else out
        check(lib().vo_exp_current(self._h, C.byref(tmin), C.byref(tmax), _np_ptr(psi.view(np.float64))), self.ctx._h)
        return (tmin.value, tmax.value), psi

    def state_ensemble(self):
        """The states in the caller's order as a device-side Ensemble view (one row of 2 n N doubles), for `Group.gather_placed`."""
        from .base import Ensemble, _TensorOwner
        h = _vp()
        check(lib().vo_exp_current_device(self._h, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, 1, 2 * self.n * self.N, _handle=h, _owner=_TensorOwner(self))

    def stats(self) -> dict:
        n = self.N
        acc, rej, t, h, dxn = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n), np.zeros(n), np.zeros(n)
        check(lib().vo_exp_stats(self._h, _np_ptr(acc), _np_ptr(rej), _np_ptr(t), _np_ptr(h), _np_ptr(dxn)), self.ctx._h)
        return dict(accepted=acc, rejected=rej, t=t, h=h, dx_norm=dxn)

    def reset(self, psi0: Optional[np.ndarray] = None):
        p = None if psi0 is None else np.ascontiguousarray(psi0, dtype=np.complex128)
        check(lib().vo_exp_reset(self._h, None if p is None else _np_ptr(p.view(np.float64))), self.ctx._h)

    @property
    def state_device_ptr(self) -> int:
        return int(lib().vo_exp_state_device_ptr(self._h) or 0)

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().vo_exp_destroy(self._h)
        except Exception:
            pass


class MidpointExpLinearSolver(_ExpSolver):
    SCHEME = "midpoint"


class ExpCFMSolver(_ExpSolver):
    SCHEME = "cfm4"


def cfm_table(name: str) -> np.ndarray:
    """The reference's coefficient statics (src/dat/mod.rs:3-6, 66-81): 'C_GAUSS_LEGENDRE_4', 'CFM_R2_J1_GL', 'CFM_R4_J2_GL',
    'BLANES17_R4_J4', shaped [rows][nodes]."""
    r, k = C.c_int32(), C.c_int32()
    check(lib().vo_cfm_builtin_table(_cabi.CFM_TABLE[name], None, C.byref(r), C.byref(k)))
    out = np.zeros((r.value, k.value))
    check(lib().vo_cfm_builtin_table(_cabi.CFM_TABLE[name], _np_ptr(out), C.byref(r), C.byref(k)))
    return out


class ExpCFMGeneralSolver(_ExpSolver):
    """cfm_general (exp/cfm.rs:43-100) as a solver with the caller's tables — what ExpCFMSolver is once `c`, `alpha`, `alph_err`
    are arguments instead of the hard-wired CFM4 (cfm.rs:131-154): `c` [k] nodes, `alpha` [rows][k], `alph_err` [rows_err][k] | None."""
    SCHEME = "cfm_table"

    def __init__(self, sp, gp, t0, tf, psi0, h, c, alpha, alph_err=None, M_gen=None, group_similar=False):
        super().__init__(sp, gp, t0, tf, psi0, h, M_gen, group_similar)
        c = np.ascontiguousarray(c, dtype=np.float64).ravel()
        a = np.ascontiguousarray(alpha, dtype=np.float64)
        e = None if alph_err is None else np.ascontiguousarray(alph_err, dtype=np.float64)
        if a.ndim != 2 or a.shape[1] != c.size or (e is not None and (e.ndim != 2 or e.shape[1] != c.size)):
            raise _cabi.VecOdeError(_cabi.VO_ERR_SHAPE, "split_cfm: Incompatible array dimensions")  # cfm.rs:63
        check(lib().vo_exp_set_cfm_tables(self._h, _np_ptr(c), c.size, _np_ptr(a), a.shape[0], None if e is None else _np_ptr(e), 0 if e is None else e.shape[0]),
              self.ctx._h)
        if e is None:
            self.no_adaptive()


class MagnusExpLinearSolver(_ExpSolver):
    """exp/magnus.rs:151-285. `dense_commutator=True`: commutator(l0, l1) (magnus.rs:55) is formed densely per system on the
    tensor cores, so the generators need not be closed under commutation on the shared basis (vo_exp_set_dense_commutator).
    `applied_commutator=True`: the commutator is applied to the state by products inside the Taylor series and never formed
    (vo_exp_set_applied_commutator): no closure assumed either, and the work stays in the tiled shared-basis kernel."""
    SCHEME = "magnus42"

    def __init__(self, sp, gp, t0, tf, psi0, h, M_gen=None, group_similar=False, dense_commutator=False, applied_commutator=False):
        super().__init__(sp, gp, t0, tf, psi0, h, M_gen, group_similar)
        if dense_commutator:
            check(lib().vo_exp_set_dense_commutator(self._h, 1), self.ctx._h)
        if applied_commutator:  # Omega T = W1 T + b2 (L0 (L1 T) - L1 (L0 T)) inside the Taylor series: the commutator is never formed
            check(lib().vo_exp_set_applied_commutator(self._h, 1), self.ctx._h)

    def literal_norm(self, on: bool = True):
        """The reference's `norm()` as written (magnus.rs:274-276): the controller sees ||x0||, not the embedded error
        (vo_exp_set_literal_norm). Off by default."""
        check(lib().vo_exp_set_literal_norm(self._h, 1 if on else 0), self.ctx._h)
        return self
