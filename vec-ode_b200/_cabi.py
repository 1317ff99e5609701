"""ctypes binding of libvecode_b200.so (include/vecode_b200.h).

This is the only place the Python host touches native code. There is NO CPU fallback: if the shared object is
missing, or a context cannot be created because no CUDA device is present, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("VECODE_B200_SO") or os.path.join(_HERE, "libvecode_b200.so")  # the override selects an experimental build (tools/build_variant.sh)

# status codes (include/vecode_b200.h)
VO_OK = 0
VO_ERR_BAD_ARG, VO_ERR_SHAPE, VO_ERR_CUDA, VO_ERR_ALLOC = -1, -2, -3, -4
VO_ERR_NOT_ADAPTIVE, VO_ERR_UNSUPPORTED, VO_ERR_STATE, VO_ERR_NCCL = -5, -6, -7, -8
GROUP_ID_BYTES = 128
ARITH_STRICT, ARITH_FAST = 0, 1
LAYOUT_SOA, LAYOUT_AOS = 0, 1
NORM = {"L2": 0, "LINF": 1, "L1": 2, "HYPOT": 3}
TABLEAU = {"RKF45_REF": 0, "RK4": 1, "DOPRI5": 2}
RHS = {"DIAG_LINEAR": 0, "HARMONIC2D": 1, "LORENZ63": 2, "VDP": 3, "HEAT1D": 4, "CUSTOM": 5, "CUSTOM_STENCIL": 6}
EXP_SCHEME = {"midpoint": 0, "cfm4": 1, "magnus42": 2, "split_midpoint": 3, "cfm_table": 4, "split_cfm": 5}
CFM_TABLE = {"C_GAUSS_LEGENDRE_4": 0, "CFM_R2_J1_GL": 1, "CFM_R4_J2_GL": 2, "BLANES17_R4_J4": 3}
EV_STEP, EV_CHKPT, EV_REJECT, EV_END, EV_ERR = range(5)
STATE_OK, STATE_DONE, STATE_ERR = range(3)
TRAJ_DONE, TRAJ_NONFINITE, TRAJ_STUCK = 1, 2, 4

_ERR_NAMES = {-1: "BAD_ARG", -2: "SHAPE", -3: "CUDA", -4: "ALLOC", -5: "NOT_ADAPTIVE", -6: "UNSUPPORTED", -7: "STATE", -8: "NCCL"}


class VecOdeError(RuntimeError):
    """A non-zero status from the C ABI; `.msg` is what the reference puts in ODEError.msg or a panic message."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"vecode_b200: {_ERR_NAMES.get(code, code)}: {msg}")
        self.code, self.msg = code, msg


class StepResult(C.Structure):
    _fields_ = [("n_step", C.c_int64), ("n_chkpt", C.c_int64), ("n_reject", C.c_int64), ("n_end", C.c_int64),
                ("n_active", C.c_int64), ("state", C.c_int32), ("launches", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class GroupStats(C.Structure):
    _fields_ = [("accepted", C.c_int64), ("rejected", C.c_int64), ("n_traj", C.c_int64), ("n_done", C.c_int64),
                ("n_nonfinite", C.c_int64), ("n_stuck", C.c_int64), ("t_min", C.c_double), ("t_max", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_vp, _i32, _i64, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
_pvp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes): every entry point of include/vecode_b200.h
SIGNATURES = {
    "vo_ctx_create": (_i32, [_i32, _vp, _pvp]),
    "vo_ctx_create_urgent": (_i32, [_i32, _i32, _pvp]),
    "vo_ctx_destroy": (_i32, [_vp]),
    "vo_ctx_sync": (_i32, [_vp]),
    "vo_ctx_fence": (_i32, [_vp]),
    "vo_ctx_wait_for": (_i32, [_vp, _vp]),
    "vo_ctx_stream": (_vp, [_vp]),
    "vo_last_error": (C.c_char_p, [_vp]),
    "vo_version": (_i32, []),
    "vo_ctx_launch_count": (_i64, [_vp]),
    "vo_guard_enabled": (_i32, []),
    "vo_guard_check": (_i64, [C.POINTER(_i64)]),
    "vo_ctx_set_arith": (_i32, [_vp, _i32]),
    "vo_ens_create": (_i32, [_vp, _i64, _i64, _pvp]),
    "vo_ens_wrap": (_i32, [_vp, _vp, _i64, _i64, _pvp]),
    "vo_ens_clone": (_i32, [_vp, _pvp]),
    "vo_ens_copy": (_i32, [_vp, _vp]),
    "vo_ens_destroy": (_i32, [_vp]),
    "vo_ens_upload": (_i32, [_vp, _vp, _i32]),
    "vo_ens_download": (_i32, [_vp, _vp, _i32]),
    "vo_ens_dims": (_i32, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "vo_ens_device_ptr": (_vp, [_vp]),
    "vo_lc_scale": (_i32, [_vp, _f64]),
    "vo_lc_scalar_multiply_to": (_i32, [_vp, _f64, _vp]),
    "vo_lc_add_scalar_mul": (_i32, [_vp, _f64, _vp]),
    "vo_lc_add_assign_ref": (_i32, [_vp, _vp]),
    "vo_lc_delta": (_i32, [_vp, _vp]),
    "vo_lc_linear_combination": (_i32, [_vp, _pvp, C.POINTER(_f64), _i32]),
    "vo_lc_stage_combine": (_i32, [_vp, _pvp, C.POINTER(_f64), _i32, _f64, _vp]),
    "vo_lc_scale_z": (_i32, [_vp, _f64, _f64]),
    "vo_lc_scalar_multiply_to_z": (_i32, [_vp, _f64, _f64, _vp]),
    "vo_lc_add_scalar_mul_z": (_i32, [_vp, _f64, _f64, _vp]),
    "vo_lc_linear_combination_z": (_i32, [_vp, _pvp, C.POINTER(_f64), _i32]),
    "vo_norm": (_i32, [_vp, _i32, _vp]),
    "vo_tableau_create": (_i32, [_vp, _vp, _vp, _i32, _pvp]),
    "vo_tableau_builtin": (_i32, [_i32, _pvp]),
    "vo_tableau_num_stages": (_i32, [_vp]),
    "vo_tableau_get": (_i32, [_vp, _vp, _vp, _vp, C.POINTER(_i32)]),
    "vo_tableau_destroy": (_i32, [_vp]),
    "vo_rhs_create": (_i32, [_vp, _i32, _i32, _pvp]),
    "vo_rhs_create_custom": (_i32, [_vp, C.c_char_p, _i32, _i32, _pvp]),
    "vo_rhs_create_custom_stencil": (_i32, [_vp, C.c_char_p, _i64, _i32, _i32, _pvp]),
    "vo_rhs_custom_stencil_check": (_i32, [C.c_char_p, _i32, _i32, _i32, C.c_char_p, _i64]),
    "vo_rhs_custom_check": (_i32, [C.c_char_p, _i32, _i32, _i32, _i32, C.c_char_p, _i64]),
    "vo_rhs_num_params": (_i32, [_vp]),
    "vo_rhs_set_param": (_i32, [_vp, _i32, _f64]),
    "vo_rhs_set_param_array": (_i32, [_vp, _i32, _vp, _i64]),
    "vo_rhs_eval": (_i32, [_vp, _f64, _vp, _vp]),
    "vo_rhs_destroy": (_i32, [_vp]),
    "vo_rk_create": (_i32, [_vp, _vp, _vp, _f64, _f64, _vp, _f64, _pvp]),
    "vo_rk45_create": (_i32, [_vp, _vp, _f64, _f64, _vp, _f64, _pvp]),
    "vo_solver_destroy": (_i32, [_vp]),
    "vo_solver_no_adaptive": (_i32, [_vp]),
    "vo_solver_with_tolerance": (_i32, [_vp, _f64, _f64]),
    "vo_solver_with_step_range": (_i32, [_vp, _f64, _f64]),
    "vo_solver_with_init_step": (_i32, [_vp, _f64]),
    "vo_solver_set_t_list": (_i32, [_vp, _vp, _i32]),
    "vo_solver_set_order_alpha": (_i32, [_vp, _f64, _f64]),
    "vo_solver_set_norm": (_i32, [_vp, _i32]),
    "vo_solver_set_norm_custom": (_i32, [_vp, _vp]),
    "vo_normfn_create": (_i32, [_vp, C.c_char_p, _i32, C.c_char_p, _pvp]),
    "vo_normfn_destroy": (_i32, [_vp]),
    "vo_normfn_check": (_i32, [C.c_char_p, _i32, C.c_char_p, C.c_char_p, _i64]),
    "vo_normfn_check_kernels": (_i32, [C.c_char_p, _i32, C.c_char_p, _i32, _i32, _i32, _i32, _i32, _i32, C.c_char_p, _i64]),
    "vo_norm_custom": (_i32, [_vp, _vp, _vp]),
    "vo_exp_set_norm_custom": (_i32, [_vp, _vp]),
    "vo_solver_set_h_array": (_i32, [_vp, _vp, _i64]),
    "vo_solver_set_events_per_launch": (_i32, [_vp, _i32]),
    "vo_solver_set_path": (_i32, [_vp, _i32]),
    "vo_solver_set_record_dx_norm": (_i32, [_vp, _i32]),
    "vo_solver_set_mixed_stepping": (_i32, [_vp, _i32]),
    "vo_solver_set_blocked": (_i32, [_vp, _i32]),
    "vo_step": (_i32, [_vp, C.POINTER(StepResult)]),
    "vo_step_adaptive": (_i32, [_vp, C.POINTER(StepResult)]),
    "vo_adaptive_try": (_i32, [_vp, _i64, _i64, C.POINTER(_f64), C.POINTER(_i32), C.POINTER(StepResult)]),
    "vo_adaptive_handle": (_i32, [_vp, _f64, C.POINTER(StepResult)]),
    "vo_run": (_i32, [_vp, _i32, _i64, C.POINTER(StepResult)]),
    "vo_step_many": (_i32, [_pvp, _i32, _i32, _i64]),
    "vo_current": (_i32, [_vp, C.POINTER(_f64), C.POINTER(_f64), _pvp]),
    "vo_solver_enable_snapshots": (_i32, [_vp]),
    "vo_solver_snapshot": (_i32, [_vp, _i32, _pvp]),
    "vo_solver_stats": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vo_solver_reset": (_i32, [_vp, _vp]),
    "vo_rk_try_step": (_i32, [_vp, _f64, _f64, _vp, _vp, _pvp]),
    "vo_split_basis_create": (_i32, [_vp, _i32, _i32, _vp, _pvp]),
    "vo_split_destroy": (_i32, [_vp]),
    "vo_split_set_commutator": (_i32, [_vp, _vp]),
    "vo_split_set_taylor_degree": (_i32, [_vp, _i32]),
    "vo_split_norm": (_i32, [_vp, _vp, _i64, _vp]),
    "vo_split_commutator": (_i32, [_vp, _vp, _vp, _i64, _vp]),
    "vo_map_exp": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "vo_map_exp_seq": (_i32, [_vp, _vp, _i32, _i64, _vp, _vp]),
    "vo_split_dense_create": (_i32, [_vp, _i32, _i64, _pvp]),
    "vo_dense_lin_zero": (_i32, [_vp, _pvp]),
    "vo_dense_assemble": (_i32, [_vp, _vp, _vp, _vp]),
    "vo_dense_exp": (_i32, [_vp, _vp, _vp]),
    "vo_dense_multi_exp": (_i32, [_vp, _vp, _vp, _i32, _pvp]),
    "vo_dense_map_exp": (_i32, [_vp, _vp, _vp, _vp]),
    "vo_dense_commutator": (_i32, [_vp, _vp, _vp, _vp]),
    "vo_exp_set_dense_commutator": (_i32, [_vp, _i32]),
    "vo_exp_set_applied_commutator": (_i32, [_vp, _i32]),
    "vo_exp_set_literal_norm": (_i32, [_vp, _i32]),
    "vo_exp_set_split_mask": (_i32, [_vp, C.c_uint32]),
    "vo_exp_set_cfm_tables": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _i32]),
    "vo_exp_set_split_cfm_tables": (_i32, [_vp, _vp, _i32, _vp, _vp, _i32]),
    "vo_cfm_builtin_table": (_i32, [_i32, _vp, C.POINTER(_i32), C.POINTER(_i32)]),
    "vo_exp_create": (_i32, [_vp, _vp, _i32, _i32, _vp, _i64, _f64, _f64, _vp, _f64, _pvp]),
    "vo_exp_destroy": (_i32, [_vp]),
    "vo_exp_set_generator": (_i32, [_vp, C.c_char_p]),
    "vo_exp_set_order": (_i32, [_vp, _vp, _i64]),
    "vo_exp_set_dynamic_grouping": (_i32, [_vp, _i32]),
    "vo_exp_generator_check": (_i32, [C.c_char_p, _i32, _i32, C.c_char_p, _i64]),
    "vo_exp_no_adaptive": (_i32, [_vp]),
    "vo_exp_with_tolerance": (_i32, [_vp, _f64, _f64]),
    "vo_exp_with_step_range": (_i32, [_vp, _f64, _f64]),
    "vo_exp_step": (_i32, [_vp, C.POINTER(StepResult)]),
    "vo_exp_step_adaptive": (_i32, [_vp, C.POINTER(StepResult)]),
    "vo_exp_run": (_i32, [_vp, _i32, _i64, C.POINTER(StepResult)]),
    "vo_exp_current": (_i32, [_vp, C.POINTER(_f64), C.POINTER(_f64), _vp]),
    "vo_exp_current_device": (_i32, [_vp, _pvp]),
    "vo_exp_stats": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "vo_exp_reset": (_i32, [_vp, _vp]),
    "vo_exp_state_device_ptr": (_vp, [_vp]),
    "vo_exp_set_t_list": (_i32, [_vp, _vp, _i32]),
    "vo_exp_enable_snapshots": (_i32, [_vp]),
    "vo_exp_snapshot": (_i32, [_vp, _i32, _vp]),
    "vo_exp_snapshot_device": (_i32, [_vp, _i32, _pvp]),
    "vo_exp_set_observables": (_i32, [_vp, _i32, _vp]),
    "vo_exp_expectation": (_i32, [_vp, _i32, _vp]),
    "vo_exp_expectation_device": (_i32, [_vp, _i32, _pvp]),
    "vo_group_unique_id": (_i32, [_vp]),
    "vo_group_create_rank": (_i32, [_vp, _vp, _i32, _i32, _pvp]),
    "vo_group_create_local": (_i32, [_pvp, _i32, _pvp]),
    "vo_group_destroy": (_i32, [_vp]),
    "vo_group_world": (_i32, [_vp]),
    "vo_group_local_members": (_i32, [_vp]),
    "vo_group_member_rank": (_i32, [_vp, _i32]),
    "vo_group_last_error": (C.c_char_p, [_vp]),
    "vo_group_nccl_version": (_i32, []),
    "vo_group_shard_range": (_i32, [_i64, _i32, _i32, C.POINTER(_i64), C.POINTER(_i64)]),
    "vo_group_scatter": (_i32, [_vp, _vp, _i32, _i64, _i64, _i32, _pvp]),
    "vo_group_run": (_i32, [_vp, _pvp, _i32, _i64, C.POINTER(GroupStats)]),
    "vo_group_gather_device": (_i32, [_vp, _pvp, _i64, _i32, _pvp]),
    "vo_group_gather": (_i32, [_vp, _pvp, _i64, _i32, _vp, _i32]),
    "vo_group_gather_placed": (_i32, [_vp, _pvp, _i32, _vp, _vp, _vp, _i32, _i64]),
    "vo_group_gather_interleaved": (_i32, [_vp, _pvp, _i32, _i64, _i64, _vp, _i32, _i64]),
    "vo_group_sync": (_i32, [_vp]),
    "vo_group_reduce_stats": (_i32, [_vp, _pvp, C.POINTER(GroupStats)]),
    "vo_group_allreduce": (_i32, [_vp, _vp, _i32, _i32]),
}

_lib = None


def build(force: bool = False, jobs: int = 8) -> str:
    """Compile the CUDA sources in-tree with nvcc for sm_100a (csrc/Makefile)."""
    args = ["make", "-C", os.path.join(_HERE, "csrc"), f"-j{jobs}"]
    if force:
        args.append("-B")
    subprocess.check_call(args, stdout=subprocess.DEVNULL)
    return SO_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(vecode_b200 has no CPU fallback)")
        l = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError here = the .so is stale w.r.t. the header
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(code: int, ctx=None):
    if code != VO_OK:
        msg = lib().vo_last_error(ctx)
        if not msg and ctx is not None:
            msg = lib().vo_last_error(None)
        raise VecOdeError(code, (msg or b"").decode("utf-8", "replace"))
