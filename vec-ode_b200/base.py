"""Host-side mirror of vec-ode's integrator API for the time-stepping path, over the C ABI.

Names, argument meaning and error behaviour follow the reference crate (paths relative to its root):
  ButcherTableu                src/base/rk.rs:22-78
  RK45Solver                   src/base/rk.rs:158-320
  ODESolver / AdaptiveODESolver  src/base/ode.rs:208-344   (step, step_adaptive, current, with_* builders)
  ODEStep / ODEState / ODEError  src/base/ode.rs:13-76
  LinearCombination            src/lc.rs:7-55
  Normed                       src/base/ode.rs:9-11
What differs by design: `V` is an `Ensemble` of N independent states on one B200 (SoA [d][N]); the RHS closure is a
compiled-in device functor (`Rhs`); a panic in the reference is a `VecOdeError` here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _cabi
from ._cabi import StepResult, VecOdeError, check, lib

_vp = C.c_void_p


def _np_ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA device + one stream. `stream` may be a raw cudaStream_t (int), e.g. torch's current stream."""

    def __init__(self, device: int = 0, stream: Optional[int] = None, arith: str = "strict", urgency: int = 0):
        self._h = _vp()
        if urgency > 0 and not stream:  # its own stream, scheduled ahead of less urgent ones (vo_ctx_create_urgent)
            check(lib().vo_ctx_create_urgent(device, urgency, C.byref(self._h)))
        else:
            check(lib().vo_ctx_create(device, _vp(stream) if stream else None, C.byref(self._h)))
        self.device = device
        self.set_arith(arith)

    @classmethod
    def on_torch_stream(cls, device: int = 0, arith: str = "strict") -> "Context":
        import torch
        torch.cuda.set_device(device)
        # torch's default stream is the legacy NULL stream, whose handle 0 would mean "create your own" to vo_ctx_create:
        # name it by CUDA's explicit handle cudaStreamLegacy (0x1) so that torch.cuda.Event timing sees our kernels.
        return cls(device, torch.cuda.current_stream(device).cuda_stream or 1, arith)

    def set_arith(self, mode: str):
        """'strict': the reference's un-fused multiply/add order, bit-identical to the CPU restatement.
        'fast': FMA contraction and zero tableau coefficients skipped."""
        check(lib().vo_ctx_set_arith(self._h, {"strict": _cabi.ARITH_STRICT, "fast": _cabi.ARITH_FAST}[mode]), self._h)
        self.arith = mode

    def sync(self):
        check(lib().vo_ctx_sync(self._h), self._h)

    def fence(self):
        """Tell the library that the caller enqueued work of its own on this context's stream that touches solver state
        (vo_ctx_fence): the next launch of every solver waits for the whole stream instead of chaining to its predecessor."""
        check(lib().vo_ctx_fence(self._h), self._h)

    def wait_for(self, other: "Context"):
        """Order this context's stream after everything enqueued so far on `other` (vo_ctx_wait_for; no host wait)."""
        check(lib().vo_ctx_wait_for(self._h, other._h), self._h)

    @property
    def launch_count(self) -> int:
        return int(lib().vo_ctx_launch_count(self._h))

    @property
    def stream(self) -> int:
        return int(lib().vo_ctx_stream(self._h) or 0)

    def close(self):
        """Drain the stream. The native context itself is released when the last Ensemble / Rhs / solver that refers to
        it is gone (they hold a reference to this object), never while a child handle could still touch it."""
        if self._h:
            self.sync()

    def __del__(self):
        try:
            if self._h:
                lib().vo_ctx_destroy(self._h)
                self._h = _vp()
        except Exception:
            pass


class Ensemble:
    """The reference's `V`: N independent d-vectors, SoA on the device (component c of trajectory i at [c*N + i])."""

    def __init__(self, ctx: Context, d: int, n: int, _handle=None, _owner=None):
        self.ctx, self.d, self.n = ctx, int(d), int(n)
        self._owner = _owner  # keeps a wrapped torch tensor / parent solver alive
        self._borrowed = _handle is not None and _owner is not None and not isinstance(_owner, _TensorOwner)
        if _handle is None:
            self._h = _vp()
            check(lib().vo_ens_create(ctx._h, self.d, self.n, C.byref(self._h)), ctx._h)
        else:
            self._h = _handle

    @classmethod
    def from_host(cls, ctx: Context, a, layout: str = "aos") -> "Ensemble":
        """a: [N][d] (layout 'aos', one contiguous state per trajectory, as the reference holds them) or [d][N] ('soa')."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.ndim == 1:
            a = a.reshape(1, -1) if layout == "aos" else a.reshape(-1, 1)
        n, d = a.shape if layout == "aos" else a.shape[::-1]
        e = cls(ctx, d, n)
        e.upload(a, layout)
        return e

    @classmethod
    def wrap_tensor(cls, ctx: Context, t) -> "Ensemble":
        """Non-owning view of a CUDA float64 torch tensor of shape [d][N] (contiguous)."""
        assert t.is_cuda and t.is_contiguous() and t.dtype.itemsize == 8 and t.dim() == 2
        h = _vp()
        check(lib().vo_ens_wrap(ctx._h, _vp(t.data_ptr()), t.shape[0], t.shape[1], C.byref(h)), ctx._h)
        return cls(ctx, t.shape[0], t.shape[1], _handle=h, _owner=_TensorOwner(t))

    def upload(self, a: np.ndarray, layout: str = "aos"):
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.size != self.d * self.n:
            raise VecOdeError(_cabi.VO_ERR_SHAPE, "upload: host array has the wrong number of elements")
        check(lib().vo_ens_upload(self._h, _np_ptr(a), _cabi.LAYOUT_AOS if layout == "aos" else _cabi.LAYOUT_SOA), self.ctx._h)

    def to_host(self, layout: str = "aos", out: Optional[np.ndarray] = None) -> np.ndarray:
        shape = (self.n, self.d) if layout == "aos" else (self.d, self.n)
        if out is None:
            out = np.empty(shape, dtype=np.float64)
        check(lib().vo_ens_download(self._h, _np_ptr(out), _cabi.LAYOUT_AOS if layout == "aos" else _cabi.LAYOUT_SOA), self.ctx._h)
        return out

    def clone(self) -> "Ensemble":
        h = _vp()
        check(lib().vo_ens_clone(self._h, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, self.d, self.n, _handle=h)

    def copy_from(self, src: "Ensemble"):
        check(lib().vo_ens_copy(self._h, src._h), self.ctx._h)

    @property
    def device_ptr(self) -> int:
        return int(lib().vo_ens_device_ptr(self._h) or 0)

    def norm(self, kind="L2") -> np.ndarray:
        """Normed::norm (src/base/ode.rs:9-11) per trajectory: a built-in kind by name, or a NormFn."""
        out = np.empty(self.n)
        if isinstance(kind, NormFn):
            check(lib().vo_norm_custom(self._h, kind._h, _np_ptr(out)), self.ctx._h)
        else:
            check(lib().vo_norm(self._h, _cabi.NORM[kind], _np_ptr(out)), self.ctx._h)
        return out

    def __del__(self):
        try:
            if self._h and not self._borrowed and self.ctx._h:
                lib().vo_ens_destroy(self._h)
        except Exception:
            pass


class _TensorOwner:
    def __init__(self, t):
        self.t = t


class LinearCombination:
    """src/lc.rs:7-55 — static methods, like the trait. Element arithmetic is src/impls/ndarray.rs:14-32."""

    @staticmethod
    def scale(v: Ensemble, k: float):
        check(lib().vo_lc_scale(v._h, k), v.ctx._h)

    @staticmethod
    def scalar_multiply_to(v: Ensemble, k: float, target: Ensemble):
        check(lib().vo_lc_scalar_multiply_to(v._h, k, target._h), v.ctx._h)

    @staticmethod
    def add_scalar_mul(v: Ensemble, k: float, other: Ensemble):
        check(lib().vo_lc_add_scalar_mul(v._h, k, other._h), v.ctx._h)

    @staticmethod
    def add_assign_ref(v: Ensemble, other: Ensemble):
        check(lib().vo_lc_add_assign_ref(v._h, other._h), v.ctx._h)

    @staticmethod
    def delta(v: Ensemble, y: Ensemble):
        check(lib().vo_lc_delta(v._h, y._h), v.ctx._h)

    @staticmethod
    def linear_combination(v: Ensemble, v_arr: Sequence[Ensemble], k_arr: Sequence[float]):
        """lc.rs:20-35 in ONE pass. Empty input is an error (the reference panics)."""
        n = min(len(v_arr), len(k_arr))  # zip semantics of lc.rs:28-33
        hs = (C.c_void_p * max(n, 1))(*[e._h.value for e in v_arr[:n]])
        ks = (C.c_double * max(n, 1))(*[float(k) for k in k_arr[:n]])
        check(lib().vo_lc_linear_combination(v._h, hs, ks, n), v.ctx._h)

    @staticmethod
    def stage_combine(v: Ensemble, v_arr: Sequence[Ensemble], k_arr: Sequence[float], dt: float, x0: Ensemble):
        """rk.rs:121-124 fused: v = (sum k_j v_j) * dt + x0."""
        n = min(len(v_arr), len(k_arr))
        hs = (C.c_void_p * max(n, 1))(*[e._h.value for e in v_arr[:n]])
        ks = (C.c_double * max(n, 1))(*[float(k) for k in k_arr[:n]])
        check(lib().vo_lc_stage_combine(v._h, hs, ks, n, dt, x0._h), v.ctx._h)


class ComplexLinearCombination:
    """`LinearCombination<Complex<f64>, V>`: the same trait on vectors of interleaved (re, im) pairs with complex scalars (the element
    type of src/impls/ndarray.rs:8-33 is generic). `add_assign_ref` / `delta` are the real ones."""

    add_assign_ref = LinearCombination.add_assign_ref
    delta = LinearCombination.delta

    @staticmethod
    def scale(v: Ensemble, k: complex):
        k = complex(k)
        check(lib().vo_lc_scale_z(v._h, k.real, k.imag), v.ctx._h)

    @staticmethod
    def scalar_multiply_to(v: Ensemble, k: complex, target: Ensemble):
        k = complex(k)
        check(lib().vo_lc_scalar_multiply_to_z(v._h, k.real, k.imag, target._h), v.ctx._h)

    @staticmethod
    def add_scalar_mul(v: Ensemble, k: complex, other: Ensemble):
        k = complex(k)
        check(lib().vo_lc_add_scalar_mul_z(v._h, k.real, k.imag, other._h), v.ctx._h)

    @staticmethod
    def linear_combination(v: Ensemble, v_arr: Sequence[Ensemble], k_arr: Sequence[complex]):
        n = min(len(v_arr), len(k_arr))
        hs = (C.c_void_p * max(n, 1))(*[e._h.value for e in v_arr[:n]])
        flat = [c for k in k_arr[:n] for c in (complex(k).real, complex(k).imag)]
        ks = (C.c_double * max(2 * n, 2))(*flat)
        check(lib().vo_lc_linear_combination_z(v._h, hs, ks, n), v.ctx._h)


class ButcherTableu:
    """src/base/rk.rs:22-78 (the reference's spelling). `ac` is s*s row-major with c_i ON the diagonal."""

    def __init__(self, handle, s: int):
        self._h, self.s = handle, s

    @classmethod
    def from_slices(cls, ac, b, b_err, s: int) -> "ButcherTableu":
        ac = np.ascontiguousarray(ac, dtype=np.float64)
        b = np.ascontiguousarray(b, dtype=np.float64)
        be = None if b_err is None else np.ascontiguousarray(b_err, dtype=np.float64)
        if ac.size != s * s or b.size != s or (be is not None and be.size != s):
            raise VecOdeError(_cabi.VO_ERR_SHAPE, "ButcherTableu: slice lengths do not match s")  # rk.rs:35-39 panics
        h = _vp()
        check(lib().vo_tableau_create(_np_ptr(ac), _np_ptr(b), _np_ptr(be), s, C.byref(h)))
        return cls(h, s)

    from_vecs = from_slices  # rk.rs:44-53

    @classmethod
    def builtin(cls, name: str) -> "ButcherTableu":
        h = _vp()
        check(lib().vo_tableau_builtin(_cabi.TABLEAU[name], C.byref(h)))
        return cls(h, int(lib().vo_tableau_num_stages(h)))

    def num_stages(self) -> int:  # rk.rs:55-57
        return int(lib().vo_tableau_num_stages(self._h))

    def arrays(self):
        s = self.s
        ac, b, be, he = np.zeros(s * s), np.zeros(s), np.zeros(s), C.c_int32()
        check(lib().vo_tableau_get(self._h, _np_ptr(ac), _np_ptr(b), _np_ptr(be), C.byref(he)))
        return ac, b, (be if he.value else None), s

    def __del__(self):
        try:
            if self._h:
                lib().vo_tableau_destroy(self._h)
        except Exception:
            pass


class NormFn:
    """A user-defined norm, the reference's `Normed<T, V>` impl (src/base/ode.rs:9-11) or ExpCFMSolver's NormFn closure
    (src/exp/cfm.rs:105, 214-216), as source (vo_normfn_create):  norm(e) = finish(JOIN_i map(e_i, i)).
    `map_body` assigns `m` from `e` (`im`: imaginary part of a complex component), `i`, `n`; `join` is "sum" or "max"; `finish_body`
    assigns `r` from `acc`, `n`. `finish_py(acc, n)` is the optional host-side twin of `finish_body` for norms combined across
    ranks (domain.HeatSlabSolver)."""

    def __init__(self, ctx: Context, map_body: str, join: str = "sum", finish_body: str = "", finish_py=None):
        self.ctx, self.join, self.finish_py = ctx, join, finish_py
        self._h = _vp()
        check(lib().vo_normfn_create(ctx._h, map_body.encode(), {"sum": 0, "max": 1}[join], finish_body.encode(), C.byref(self._h)), ctx._h)

    @staticmethod
    def check_source(map_body: str, join: str = "sum", finish_body: str = "") -> int:
        """Compile only (NVRTC, no GPU): the cubin size, or VecOdeError with the compiler log."""
        log = C.create_string_buffer(8192)
        rc = lib().vo_normfn_check(map_body.encode(), {"sum": 0, "max": 1}[join], finish_body.encode(), log, len(log))
        if rc < 0:
            raise VecOdeError(rc, log.value.decode(errors="replace"))
        return rc

    @staticmethod
    def check_kernels(map_body: str, join: str = "sum", finish_body: str = "", rhs_kind: int = -1, d: int = 0, stages: int = 0, arith: str = "strict",
                      exp_n: int = 0, exp_M: int = 0) -> int:
        """Compile the solver kernels the functor goes INTO (vo_normfn_check_kernels; NVRTC, no GPU)."""
        log = C.create_string_buffer(8192)
        rc = lib().vo_normfn_check_kernels(map_body.encode(), {"sum": 0, "max": 1}[join], finish_body.encode(), rhs_kind, d, stages,
                                           _cabi.ARITH_STRICT if arith == "strict" else _cabi.ARITH_FAST, exp_n, exp_M, log, len(log))
        if rc < 0:
            raise VecOdeError(rc, log.value.decode(errors="replace"))
        return rc

    def finish_host(self, acc: float, n: int) -> float:
        if self.finish_py is None:
            raise ValueError("this NormFn has no finish_py: give the host-side twin of finish_body to combine the norm across ranks")
        return float(self.finish_py(acc, n))

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().vo_normfn_destroy(self._h)
        except Exception:
            pass


class Rhs:
    """Replaces the closure `FnMut(T, &V, &mut V) -> Result<(),()>` (src/base/rk.rs:97): a compiled-in device functor
    chosen by name, with parameters that are shared scalars or per-trajectory arrays."""

    def __init__(self, ctx: Context, kind: str, d: int, params=None, body: str | None = None, radius: int = 0):
        self.ctx, self.kind, self.d = ctx, kind, d
        self._h = _vp()
        if kind == "CUSTOM":
            n_params = 0 if params is None else len(params)
            check(lib().vo_rhs_create_custom(ctx._h, body.encode(), d, n_params, C.byref(self._h)), ctx._h)
        elif kind == "CUSTOM_STENCIL":
            n_params = 0 if params is None else len(params)
            check(lib().vo_rhs_create_custom_stencil(ctx._h, body.encode(), d, radius, n_params, C.byref(self._h)), ctx._h)
        else:
            check(lib().vo_rhs_create(ctx._h, _cabi.RHS[kind], d, C.byref(self._h)), ctx._h)
        self.num_params = int(lib().vo_rhs_num_params(self._h))
        if params is not None:
            for i, p in enumerate(params):
                self.set_param(i, p)

    @classmethod
    def custom(cls, ctx: Context, body: str, d: int, params=()):
        """The closure itself: `body` is CUDA C++ for the statements of `f(t, &x, &mut dx)` over `t`, `x[D]`, `dx[D]`, `p[NP]`;
        it is compiled at run time into the same fused kernels as the built-in families (vo_rhs_create_custom)."""
        return cls(ctx, "CUSTOM", d, list(params), body=body)

    @classmethod
    def custom_stencil(cls, ctx: Context, body: str, d: int, radius: int, params=()):
        """A user stencil on one periodic grid state of d points: `body` assigns `du` from `u[0 .. 2R]` (u[R] is the point itself),
        `t`, `j`, `d`, `p[NP]` (shared parameters); compiled at run time into the fused per-stage kernel (vo_rhs_create_custom_stencil)."""
        return cls(ctx, "CUSTOM_STENCIL", d, list(params), body=body, radius=radius)

    @staticmethod
    def check_stencil_source(body: str, radius: int, n_params: int, arith: str = "strict") -> int:
        log = C.create_string_buffer(1 << 16)
        rc = lib().vo_rhs_custom_stencil_check(body.encode(), radius, n_params, _cabi.ARITH_STRICT if arith == "strict" else _cabi.ARITH_FAST, log, len(log))
        if rc < 0:
            raise VecOdeError(rc, log.value.decode("utf-8", "replace"))
        return rc

    @staticmethod
    def check_source(body: str, d: int, n_params: int, stages: int = -1, arith: str = "strict") -> int:
        """Compile `body` without a GPU; returns the cubin size or raises VecOdeError carrying the compiler log."""
        log = C.create_string_buffer(1 << 16)
        rc = lib().vo_rhs_custom_check(body.encode(), d, n_params, stages, _cabi.ARITH_STRICT if arith == "strict" else _cabi.ARITH_FAST, log, len(log))
        if rc < 0:
            raise VecOdeError(rc, log.value.decode("utf-8", "replace"))
        return rc

    def set_param(self, idx: int, value):
        if np.ndim(value) == 0:
            check(lib().vo_rhs_set_param(self._h, idx, float(value)), self.ctx._h)
        else:
            a = np.ascontiguousarray(value, dtype=np.float64)
            check(lib().vo_rhs_set_param_array(self._h, idx, _np_ptr(a), a.size), self.ctx._h)

    def __call__(self, t: float, x: Ensemble, dx: Ensemble):
        check(lib().vo_rhs_eval(self._h, t, x._h, dx._h), self.ctx._h)

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().vo_rhs_destroy(self._h)
        except Exception:
            pass


# ---- ODEStep / ODEState / ODEError (src/base/ode.rs:13-76), aggregated over the ensemble ------------------------
@dataclass
class ODEError(Exception):
    msg: str


@dataclass(frozen=True)
class ODEStep:
    """`enum ODEStep<T>` (src/base/ode.rs:41-77) for ONE trajectory: kind in 'Step' | 'Chkpt' | 'Reject' | 'End' | 'Err', with the step
    size for 'Step' and the error for 'Err'. The device keeps one of these per trajectory in its status word; the host mirror is for
    callers that drive `try_step` themselves (rk.rs:287-293) or port code written against the enum."""
    kind: str
    dt: Optional[float] = None
    err: Optional["ODEError"] = None

    @staticmethod
    def Step(dt: float) -> "ODEStep":
        return ODEStep("Step", float(dt))

    def map_dt(self, f) -> "ODEStep":
        """ode.rs:53-61: run `f(dt)` on a Step; an ODEError it raises (Rust: returns) turns the step into Err, anything else passes."""
        if self.kind != "Step":
            return self
        try:
            f(self.dt)
        except ODEError as e:
            return ODEStep("Err", None, e)
        return self

    def unwrap_dt(self) -> float:  # ode.rs:63-68
        if self.kind != "Step":
            raise RuntimeError("ODEStep::unwrap_dt expected Step(T) in enum")
        return self.dt

    def unwrap_dt_or(self, dt2: float) -> float:  # ode.rs:70-75
        return self.dt if self.kind == "Step" else dt2


ODEStep.Chkpt, ODEStep.Reject, ODEStep.End = ODEStep("Chkpt"), ODEStep("Reject"), ODEStep("End")


def check_step(t0: float, tf: float, dt: float) -> Optional[float]:
    """src/base/ode.rs:389-399: None when tf - t0 is zero to `relative_eq` (approx 0.5: equal, or |rem| <= 2^-52), else the remainder if
    it is shorter than dt, else dt — the rule the kernels apply per trajectory (rk_small.cuh: ctl_lane)."""
    rem = tf - t0
    if rem == 0.0 or abs(rem) <= 2.220446049250313e-16:
        return None
    return rem if rem < dt else dt


@dataclass
class ODEState:
    """kind: 'Ok' while any trajectory still steps, 'Done' when all have emitted End, 'Err'. `counts` holds how many
    trajectories saw each ODEStep variant in this call (Step / Chkpt / Reject / End)."""
    kind: str
    counts: dict

    @property
    def is_ok(self):
        return self.kind == "Ok"


def _state_of(res: StepResult) -> ODEState:
    kind = {_cabi.STATE_OK: "Ok", _cabi.STATE_DONE: "Done", _cabi.STATE_ERR: "Err"}[res.state]
    return ODEState(kind, dict(Step=res.n_step, Chkpt=res.n_chkpt, Reject=res.n_reject, End=res.n_end, active=res.n_active,
                               launches=res.launches))


class RK45Solver:
    """RK45Solver (src/base/rk.rs:158-320) over an ensemble. `RK45Solver(f, t0, tf, x0, h)` hard-wires the reference's
    RKF45 tables exactly like `RK45Solver::new`; pass `tableau=` for any other ButcherTableu."""

    def __init__(self, f: Rhs, t0: float, tf: float, x0: Ensemble, h: float, tableau: Optional[ButcherTableu] = None):
        self.ctx, self.f, self.tableau = x0.ctx, f, tableau
        self._h = _vp()
        if tableau is None:
            check(lib().vo_rk45_create(self.ctx._h, f._h, t0, tf, x0._h, h, C.byref(self._h)), self.ctx._h)
        else:
            check(lib().vo_rk_create(self.ctx._h, tableau._h, f._h, t0, tf, x0._h, h, C.byref(self._h)), self.ctx._h)
        self.d, self.n = x0.d, x0.n

    # builders (consume-and-return like the reference) ------------------------------------------------------------
    def no_adaptive(self):  # rk.rs:233-237
        check(lib().vo_solver_no_adaptive(self._h), self.ctx._h)
        return self

    def with_tolerance(self, atol: float, rtol: float):  # ode.rs:298-306
        check(lib().vo_solver_with_tolerance(self._h, atol, rtol), self.ctx._h)
        return self

    def with_step_range(self, dt_min: float, dt_max: float):  # ode.rs:267-285
        check(lib().vo_solver_with_step_range(self._h, dt_min, dt_max), self.ctx._h)
        return self

    def with_init_step(self, h: float):  # ode.rs:287-296
        check(lib().vo_solver_with_init_step(self._h, h), self.ctx._h)
        return self

    def with_norm(self, kind):  # the user-supplied `Normed` impl (rk.rs:302): a built-in kind by name, or a NormFn
        if isinstance(kind, NormFn):
            check(lib().vo_solver_set_norm_custom(self._h, kind._h), self.ctx._h)
            self._norm_fn = kind  # keep the functor alive as long as the solver
        else:
            check(lib().vo_solver_set_norm(self._h, _cabi.NORM[kind]), self.ctx._h)
        return self

    def with_order_alpha(self, order: float, alpha: float):  # ode.rs:114-131
        check(lib().vo_solver_set_order_alpha(self._h, order, alpha), self.ctx._h)
        return self

    def set_t_list(self, t_list):  # pub field ODEData.t_list (ode.rs:89)
        a = np.ascontiguousarray(t_list, dtype=np.float64)
        check(lib().vo_solver_set_t_list(self._h, _np_ptr(a), a.size), self.ctx._h)
        return self

    def set_h_array(self, h):
        a = np.ascontiguousarray(h, dtype=np.float64)
        check(lib().vo_solver_set_h_array(self._h, _np_ptr(a), a.size), self.ctx._h)
        return self

    def set_events_per_launch(self, k: int):
        check(lib().vo_solver_set_events_per_launch(self._h, k), self.ctx._h)
        return self

    def set_record_dx_norm(self, on: bool = True):
        """Keep ODEAdaptiveData.dx_norm (ode.rs:104) of each trajectory's latest attempt (default) or skip that store."""
        check(lib().vo_solver_set_record_dx_norm(self._h, 1 if on else 0), self.ctx._h)
        return self

    def set_mixed_stepping(self, on: bool = True):
        """Allow step() after step_adaptive() under per-trajectory control: the adaptive kernels then store prev_h on every
        attempt (update_step_size, ode.rs:202-205) instead of only where a checkpoint comes next (vo_solver_set_mixed_stepping)."""
        check(lib().vo_solver_set_mixed_stepping(self._h, 1 if on else 0), self.ctx._h)
        return self

    def set_blocked(self, on: bool = True):
        """False: keep the public state layout, the only one (no-op). True raises: the tile-blocked copy of the state was
        removed as no faster (vo_solver_set_blocked)."""
        check(lib().vo_solver_set_blocked(self._h, 1 if on else 0), self.ctx._h)
        return self

    def set_fused_step(self, on: bool = True):
        """Whole-step path for a single HEAT1D state: every stage of a step in one kernel (vo_solver_set_path(s, 2))."""
        check(lib().vo_solver_set_path(self._h, 2 if on else 0), self.ctx._h)
        return self

    def set_stage_path(self, on: bool = True):
        check(lib().vo_solver_set_path(self._h, 1 if on else 0), self.ctx._h)
        return self

    # stepping ------------------------------------------------------------------------------------------------------
    def step(self) -> ODEState:  # ode.rs:249-253
        res = StepResult()
        check(lib().vo_step(self._h, C.byref(res)), self.ctx._h)
        return _state_of(res)

    def step_adaptive(self) -> ODEState:  # ode.rs:337-341
        res = StepResult()
        check(lib().vo_step_adaptive(self._h, C.byref(res)), self.ctx._h)
        return _state_of(res)

    def adaptive_try(self, lo: int, hi: int):
        """First half of step_adaptive (ode.rs:336-344) for a state held in pieces: try_step + the norm accumulator of this piece's
        components [lo, hi). Returns (acc, event, state): `state` is the finished ODEState when the event was Chkpt / End, else None
        (combine the pieces' accumulators, then call adaptive_handle with the global norm)."""
        acc, ev, res = C.c_double(), C.c_int32(), StepResult()
        check(lib().vo_adaptive_try(self._h, lo, hi, C.byref(acc), C.byref(ev), C.byref(res)), self.ctx._h)
        return acc.value, ev.value, (None if ev.value == 0 else _state_of(res))

    def adaptive_handle(self, dx_norm: float) -> ODEState:
        """Second half: handle_step_adaptive (ode.rs:311-334) with the global error norm, then apply_step."""
        res = StepResult()
        check(lib().vo_adaptive_handle(self._h, float(dx_norm), C.byref(res)), self.ctx._h)
        return _state_of(res)

    def run(self, adaptive: bool = False, max_calls: int = 0) -> ODEState:
        """`while let ODEState::Ok(_) = solver.step() {}` for the whole ensemble."""
        res = StepResult()
        check(lib().vo_run(self._h, 1 if adaptive else 0, max_calls, C.byref(res)), self.ctx._h)
        return _state_of(res)

    def state(self) -> "Ensemble":
        """The borrowed state ensemble alone (vo_current without the time range: nothing is read back, nothing synchronises)."""
        h = _vp()
        check(lib().vo_current(self._h, None, None, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, self.d, self.n, _handle=h, _owner=self)

    def current(self):  # ode.rs:216-218 -> ((t_min, t_max), borrowed Ensemble)
        tmin, tmax, h = C.c_double(), C.c_double(), _vp()
        check(lib().vo_current(self._h, C.byref(tmin), C.byref(tmax), C.byref(h)), self.ctx._h)
        return (tmin.value, tmax.value), Ensemble(self.ctx, self.d, self.n, _handle=h, _owner=self)

    def into_current(self):  # ode.rs:219-221: the state by value — a copy the solver no longer owns
        (t_min, t_max), x = self.current()
        return (t_min, t_max), x.clone()

    def validate_adaptive(self) -> None:  # ode.rs:263-265: the reference's default accepts every configuration
        return None

    def stats(self) -> dict:
        n = self.n
        acc, rej = np.zeros(n, np.int64), np.zeros(n, np.int64)
        t, h, dxn, st = np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n, np.int32)
        check(lib().vo_solver_stats(self._h, _np_ptr(acc), _np_ptr(rej), _np_ptr(t), _np_ptr(h), _np_ptr(dxn), _np_ptr(st)), self.ctx._h)
        return dict(accepted=acc, rejected=rej, t=t, h=h, dx_norm=dxn, status=st)

    def enable_snapshots(self):
        """Keep the state of every trajectory at each entry of t_list (its Chkpt / End events, ode.rs:165-176)."""
        check(lib().vo_solver_enable_snapshots(self._h), self.ctx._h)
        return self

    def snapshot(self, k: int) -> Ensemble:
        h = _vp()
        check(lib().vo_solver_snapshot(self._h, k, C.byref(h)), self.ctx._h)
        return Ensemble(self.ctx, self.d, self.n, _handle=h, _owner=_TensorOwner(self))  # view handle is ours, storage is the solver's

    def reset(self, x0: Ensemble):
        check(lib().vo_solver_reset(self._h, x0._h), self.ctx._h)

    def try_step(self, t: float, dt: float, next_x: Ensemble, x_err: Optional[Ensemble] = None, K: Optional[Sequence[Ensemble]] = None):
        """One bare rk_step (rk.rs:90-155) on the current x, without advancing."""
        ks = None
        if K is not None:
            ks = (C.c_void_p * len(K))(*[e._h.value for e in K])
        check(lib().vo_rk_try_step(self._h, t, dt, next_x._h, None if x_err is None else x_err._h, ks), self.ctx._h)

    def __del__(self):
        try:
            if self._h and self.ctx._h:
                lib().vo_solver_destroy(self._h)
        except Exception:
            pass


def step_many(solvers: Sequence[RK45Solver], adaptive: bool = False, rounds: int = 1):
    """Round-robin one launch per solver, `rounds` times, with no read-back (vo_step_many)."""
    hs = (C.c_void_p * len(solvers))(*[s._h.value for s in solvers])
    check(lib().vo_step_many(hs, len(solvers), 1 if adaptive else 0, rounds), solvers[0].ctx._h)
