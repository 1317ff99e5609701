/* vecode_b200.h — C ABI of the B200-native batched ODE time-stepping engine.
 *
 * Drop-in boundary for the time-stepping path of hmunozb/vec-ode. Each entry point names the reference
 * interface it replaces (paths relative to the crate root). Plain pointers and sizes only; every function
 * returns an int32 status (0 = ok, < 0 = error) and never aborts or throws across the boundary; the
 * message that the reference would put in `ODEError.msg` or a panic is available from vo_last_error().
 *
 * One `vo_ctx` = one CUDA device + one stream. Calls on a ctx are not re-entrant; different ctxs may be
 * driven from different threads / processes (one process per GPU is the multi-GPU model).
 *
 * Data model: an ensemble (`vo_ens`) is N independent state vectors of dimension d stored
 * structure-of-arrays, element (c, i) at `ptr[c * N + i]` (component c of trajectory i), f64. A single
 * large state is the N = 1 case. Where the reference owns one solver object per trajectory, a
 * `vo_solver` owns the whole ensemble and carries the per-trajectory controller state (t, h, prev_h,
 * tgt_t, counters) on the device.
 */
#ifndef VECODE_B200_H
#define VECODE_B200_H

#ifndef __CUDACC_RTC__ /* the run-time compiled RHS modules (vo_rhs_create_custom) get the fixed-width types from common.cuh */
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define VO_VERSION 100

/* ---- status codes ---------------------------------------------------------------------------- */
#define VO_OK 0
#define VO_ERR_BAD_ARG (-1)      /* precondition that panics in the reference (ode.rs:269,290,300; lc.rs:21-26) */
#define VO_ERR_SHAPE (-2)        /* mismatched ensemble shapes / stage counts (rk.rs:106-108) */
#define VO_ERR_CUDA (-3)
#define VO_ERR_ALLOC (-4)
#define VO_ERR_NOT_ADAPTIVE (-5) /* step_adaptive on a solver without x_err (ode.rs:312, rk.rs:317-319) */
#define VO_ERR_UNSUPPORTED (-6)
#define VO_ERR_STATE (-7)
#define VO_ERR_NCCL (-8)

typedef struct vo_ctx_s* vo_ctx;
typedef struct vo_ens_s* vo_ens;
typedef struct vo_tableau_s* vo_tableau;
typedef struct vo_rhs_s* vo_rhs;
typedef struct vo_solver_s* vo_solver;
typedef struct vo_split_s* vo_split;
typedef struct vo_expsolver_s* vo_expsolver;
typedef struct vo_group_s* vo_group;
typedef struct vo_normfn_s* vo_normfn;

/* ---- context ---------------------------------------------------------------------------------- */
/* device: CUDA ordinal. stream: a cudaStream_t to enqueue on (e.g. torch's current stream), or NULL to
 * let the ctx create its own non-blocking stream (use CUDA's cudaStreamLegacy handle, 0x1, to name the NULL stream). */
int32_t vo_ctx_create(int32_t device, void* stream, vo_ctx* out);
/* A ctx on a stream of its own whose pending thread blocks are scheduled ahead of those of less urgent streams (CUDA stream
 * priorities; urgency 0 = vo_ctx_create's default, higher = earlier, clamped to what the device offers). A solve cut into chunks
 * on several contexts (vec-ode_b200/pipeline.py) gives chunk q urgency parts - q, so the chunks FINISH one after the other and
 * the transfers of a finished chunk overlap the integration of the next instead of all chunks ending together. */
int32_t vo_ctx_create_urgent(int32_t device, int32_t urgency, vo_ctx* out);
int32_t vo_ctx_destroy(vo_ctx ctx);
int32_t vo_ctx_sync(vo_ctx ctx);
void* vo_ctx_stream(vo_ctx ctx);
/* Consecutive launches of one solver are chained CTA to CTA (a launch starts working on a tile as soon as the previous
 * launch has released that tile instead of waiting for the whole grid) — across API calls too, which is what makes the
 * reference's driver loop `while let Ok(_) = solver.step() {}` (src/impls/nalgebra.rs:62) run at the rate of vo_run. The
 * library knows about everything it enqueues itself. If the CALLER enqueues work on the ctx's stream that reads or writes a
 * solver's state (a kernel of its own on a borrowed device pointer, a framework op on a wrapped tensor), it calls
 * vo_ctx_fence afterwards: the next launch of every solver on the ctx then waits for the whole stream like an ordinary
 * launch. */
int32_t vo_ctx_fence(vo_ctx ctx);
/* Order everything enqueued on `waiter` from now on after everything enqueued on `other` so far (device-side, no host wait). */
int32_t vo_ctx_wait_for(vo_ctx waiter, vo_ctx other);
/* Message of the most recent failure on this ctx (NULL ctx: last failure of a create call on this thread).
 * Replaces ODEError.msg (src/base/ode.rs:13-30) and the reference's panic messages. */
const char* vo_last_error(vo_ctx ctx);
int32_t vo_version(void);
/* Number of kernels this ctx has launched since creation (bench.py's `gpu_launches`). */
int64_t vo_ctx_launch_count(vo_ctx ctx);

/* The library's own bounds check (compute-sanitizer's stand-in on pools where it is closed). With VECODE_GUARD=1 in the environment
 * when the library is loaded, every device block the library allocates lies between two 4 KiB guard zones filled with a byte
 * pattern. vo_guard_check synchronises, inspects the zones of every live block and returns the number of blocks found damaged since
 * load (blocks already freed were inspected when freed); *live_blocks (may be NULL) receives the number of blocks checked. Returns 0
 * and checks nothing when the switch is off (vo_guard_enabled() == 0). Diagnostics go to stderr. */
int32_t vo_guard_enabled(void);
int64_t vo_guard_check(int64_t* live_blocks);

/* Arithmetic mode of every kernel launched on the ctx.
 * VO_ARITH_STRICT: separate IEEE multiply and add in the reference's operation order, zero coefficients
 *   kept — bit-identical to rustc's un-fused f64 code (src/impls/ndarray.rs:14-32).
 * VO_ARITH_FAST: FMA contraction allowed and zero tableau coefficients skipped. */
#define VO_ARITH_STRICT 0
#define VO_ARITH_FAST 1
int32_t vo_ctx_set_arith(vo_ctx ctx, int32_t mode);

/* ---- ensembles (the `V` of the reference; `V: Clone`, src/base/ode.rs:79-80) ------------------- */
#define VO_LAYOUT_SOA 0 /* host buffer [d][N] */
#define VO_LAYOUT_AOS 1 /* host buffer [N][d] — one contiguous state per trajectory, as the reference holds them */
int32_t vo_ens_create(vo_ctx ctx, int64_t d, int64_t n, vo_ens* out); /* zero-filled */
int32_t vo_ens_wrap(vo_ctx ctx, void* device_ptr, int64_t d, int64_t n, vo_ens* out); /* non-owning view */
int32_t vo_ens_clone(vo_ens src, vo_ens* out);                          /* V::clone */
int32_t vo_ens_copy(vo_ens dst, vo_ens src);                            /* V::clone_from */
int32_t vo_ens_destroy(vo_ens e);
int32_t vo_ens_upload(vo_ens e, const double* host, int32_t layout);    /* synchronous on return */
int32_t vo_ens_download(vo_ens e, double* host, int32_t layout);        /* synchronous on return */
int32_t vo_ens_dims(vo_ens e, int64_t* d, int64_t* n);
void* vo_ens_device_ptr(vo_ens e);

/* ---- LinearCombination (src/lc.rs:7-55; element arithmetic of src/impls/ndarray.rs:14-32) ------ */
int32_t vo_lc_scale(vo_ens v, double k);                                /* lc.rs:10  v *= k            */
int32_t vo_lc_scalar_multiply_to(vo_ens v, double k, vo_ens target);    /* lc.rs:12  target = k*v      */
int32_t vo_lc_add_scalar_mul(vo_ens v, double k, vo_ens u);             /* lc.rs:14  v = v + (k*u)     */
int32_t vo_lc_add_assign_ref(vo_ens v, vo_ens u);                       /* lc.rs:16  v += u            */
int32_t vo_lc_delta(vo_ens v, vo_ens y);                                /* lc.rs:18  v -= y            */
/* lc.rs:20-54: v = k0*v0, then v = v + (ki*vi) left to right — ONE fused pass (n <= VO_MAX_TERMS).
 * n == 0 returns VO_ERR_BAD_ARG (the reference panics / returns Err(())). v may alias none of v_arr. */
#define VO_MAX_TERMS 16
int32_t vo_lc_linear_combination(vo_ens v, const vo_ens* v_arr, const double* k_arr, int32_t n);
/* Fused RK stage argument (rk.rs:121-124): v = (sum_j k_j v_j) * dt + x0, same operation order. */
int32_t vo_lc_stage_combine(vo_ens v, const vo_ens* v_arr, const double* k_arr, int32_t n, double dt, vo_ens x0);
/* LinearCombination<Complex<f64>, V> — the same trait with the scalar type of a complex vector space (src/impls/ndarray.rs:8-33 is
 * generic over the element type; the exponential integrators' states and dense operators are such vectors). v, u, target: ensembles
 * whose rows hold interleaved (re, im) pairs (n even), e.g. the view vo_exp_current_device hands out or the operator ensembles of vo_split_dense_*. Arithmetic as
 * num-complex writes it (Mul: re = a.re b.re - a.im b.im, im = a.re b.im + a.im b.re), un-fused in strict mode. add_assign_ref and
 * delta are vo_lc_add_assign_ref / vo_lc_delta unchanged. k_arr of the n-term reducer: [n][2] (re, im). */
int32_t vo_lc_scale_z(vo_ens v, double k_re, double k_im);                                 /* lc.rs:10 */
int32_t vo_lc_scalar_multiply_to_z(vo_ens v, double k_re, double k_im, vo_ens target);     /* lc.rs:12 */
int32_t vo_lc_add_scalar_mul_z(vo_ens v, double k_re, double k_im, vo_ens u);              /* lc.rs:14 */
int32_t vo_lc_linear_combination_z(vo_ens v, const vo_ens* v_arr, const double* k_arr, int32_t n);  /* lc.rs:20-54 */

/* ---- Normed (src/base/ode.rs:9-11): per-trajectory norm over the d components ------------------ */
#define VO_NORM_L2 0    /* sqrt(sum_c e_c^2), left-to-right for d <= 64, tree-reduced above that */
#define VO_NORM_LINF 1  /* max_c |e_c| */
#define VO_NORM_L1 2
#define VO_NORM_HYPOT 3 /* complex scalar stored as (re, im): hypot (rk.rs:209-214) */
#define VO_NORM_CUSTOM 4 /* a vo_normfn (below); set through vo_solver_set_norm_custom / vo_exp_set_norm_custom */
int32_t vo_norm(vo_ens e, int32_t kind, double* out_host /* [N] */);
/* User-defined norms. `Normed<T, V>` is the USER's trait impl (ode.rs:9-11; RK45Solver::norm, rk.rs:302-304) and ExpCFMSolver takes
 * a NormFn closure (exp/cfm.rs:105, 214-216). Like the RHS closure it crosses the C ABI as SOURCE, in the shape
 *     norm(e) = finish( JOIN_i map(e_i, i) ),   JOIN = VO_NORM_JOIN_SUM or VO_NORM_JOIN_MAX:
 * `map_body`: CUDA C++ statements assigning `double m` (>= 0) from `const double e` (component i; the real part of a complex
 * component), `const double im` (its imaginary part, 0 for real states), `const int i`, `const int n` (number of components);
 * `finish_body`: statements assigning `double r` from `const double acc`, `const int n` (NULL or "": r = acc).
 * E.g. a weighted RMS norm: map "m = (e * e) / (1.0 + i);", SUM, finish "r = sqrt(acc / n);".
 * The functor is compiled at run time (NVRTC, sm_100a) into the same kernels that hold the built-in norms: the register-resident
 * control kernels, the exponential-integrator kernel and the reduction kernels of the stage path. */
#define VO_NORM_JOIN_SUM 0
#define VO_NORM_JOIN_MAX 1
int32_t vo_normfn_create(vo_ctx ctx, const char* map_body, int32_t join, const char* finish_body, vo_normfn* out);
int32_t vo_normfn_destroy(vo_normfn f);
/* Compile the functor without a ctx or a GPU (NVRTC only): cubin size (> 0), or VO_ERR_* with the compiler log in `log`. */
int32_t vo_normfn_check(const char* map_body, int32_t join, const char* finish_body, char* log, int64_t log_cap);
/* The same for the solver kernels the functor is compiled INTO: rhs_kind >= 0 compiles the register-resident kernels of that
 * compiled-in family (d components, `stages`-stage tableau, VO_ARITH_* mode) with the norm; exp_n > 0 compiles
 * exp_step_kernel<exp_n, exp_M> with it. Sum of the cubin sizes, or VO_ERR_* with the log. No ctx, no GPU. */
int32_t vo_normfn_check_kernels(const char* map_body, int32_t join, const char* finish_body, int32_t rhs_kind, int32_t d, int32_t stages, int32_t arith,
                                int32_t exp_n, int32_t exp_M, char* log, int64_t log_cap);
int32_t vo_norm_custom(vo_ens e, vo_normfn f, double* out_host /* [N] */);  /* Normed::norm on its own */

/* ---- ButcherTableu (src/base/rk.rs:22-78) ------------------------------------------------------ */
#define VO_MAX_STAGES 16
/* Same argument meaning as ButcherTableu::from_slices (rk.rs:31-42): ac is s*s row-major with a_ij below
 * the diagonal and c_i ON the diagonal; b_err may be NULL. */
int32_t vo_tableau_create(const double* ac, const double* b, const double* b_err, int32_t s, vo_tableau* out);
#define VO_TABLEAU_RKF45_REF 0 /* RK45_AC/B/BERR literally as in src/dat/mod.rs:9-27 (incl. -3544./2526.) */
#define VO_TABLEAU_RK4 1
#define VO_TABLEAU_DOPRI5 2    /* 4th-order weights in b, 5th-order in b_err (local extrapolation under rk.rs:142-146) */
int32_t vo_tableau_builtin(int32_t which, vo_tableau* out);
int32_t vo_tableau_num_stages(vo_tableau t);                            /* rk.rs:55-57 */
int32_t vo_tableau_get(vo_tableau t, double* ac, double* b, double* b_err, int32_t* has_err);
int32_t vo_tableau_destroy(vo_tableau t);

/* ---- right-hand sides: replace the closure `FnMut(T, &V, &mut V) -> Result<(),()>` (rk.rs:97) ---- */
#define VO_RHS_DIAG_LINEAR 0 /* dx_c = p_c * x_c                      params: d                     */
#define VO_RHS_HARMONIC2D 1  /* dx = v ; dv = -(k*x)                  params: k                     */
#define VO_RHS_LORENZ63 2    /* sigma, rho, beta                      params: 3                     */
#define VO_RHS_VDP 3         /* dx = v ; dv = (mu*(1-x*x))*v - x      params: mu                    */
#define VO_RHS_HEAT1D 4      /* du_j = kappa*((u_{j-1}+u_{j+1}) - 2u_j), periodic in j; params: kappa */
#define VO_RHS_CUSTOM 5      /* vo_rhs_create_custom */
#define VO_RHS_CUSTOM_STENCIL 6 /* vo_rhs_create_custom_stencil */
int32_t vo_rhs_create(vo_ctx ctx, int32_t kind, int32_t d, vo_rhs* out);
/* User-defined right-hand side, the closest a C ABI gets to the reference's closure: `body` is CUDA C++ source for the
 * statements of f(t, &x, &mut dx). It sees `const double t`, `const double (&x)[D]`, `double (&dx)[D]`,
 * `const double (&p)[NP]` (D = d <= 32, NP = n_params <= 8, parameters shared or per-trajectory like the built-ins) and
 * must assign every dx[c]. It is compiled at run time with NVRTC for sm_100a INTO the fused register-resident kernels
 * (one module per stage count and arithmetic mode, cached): VO_ARITH_STRICT compiles with -fmad=false, so plain `a*b+c`
 * in the body stays an un-fused multiply and add like the reference's Rust. Compile errors come back through
 * vo_last_error. d <= 8 runs on both kernel paths (register-resident and stage path) like a built-in family; 9 <= d <= 32
 * runs on the stage path (one fused kernel per stage, the d components of a trajectory in one thread's registers). */
int32_t vo_rhs_create_custom(vo_ctx ctx, const char* body, int32_t d, int32_t n_params, vo_rhs* out);
/* Compile `body` exactly as vo_rhs_create_custom / the first step would, without a ctx or a GPU (NVRTC only): `stages` is the
 * tableau's stage count (-1 = the stage-path module), `arith` a VO_ARITH_* mode. Returns the size of the sm_100a cubin
 * (> 0), or a VO_ERR_* code with the compiler log copied to `log` (NUL-terminated, at most log_cap bytes; may be NULL). */
int32_t vo_rhs_custom_check(const char* body, int32_t d, int32_t n_params, int32_t stages, int32_t arith, char* log, int64_t log_cap);
/* User-defined STENCIL right-hand side for one large periodic grid state (N == 1; `V = Array1<f64>`, src/impls/ndarray.rs:8-33):
 * dx_j = f(t, x_{j-R} .. x_{j+R}). `body`: CUDA C++ statements assigning `double du` from `const double (&u)[2 * R + 1]` (u[R] is the
 * grid point itself, indices wrap periodically), `const double t`, `const long long j` (grid index), `const long long d` (grid size),
 * `const double (&p)[NP]` (shared parameters, vo_rhs_set_param). 1 <= radius <= 8. Compiled at run time into the fused per-stage
 * kernel of the stage path (rk_stage_stencil.cuh); fixed-step, adaptive (single-state controller) and domain-decomposed runs work
 * as for the compiled-in heat equation, whose body would be "du = p[0] * ((u[0] + u[2]) - 2.0 * u[1]);" with radius 1 (the same
 * bits in VO_ARITH_STRICT). */
int32_t vo_rhs_create_custom_stencil(vo_ctx ctx, const char* body, int64_t d, int32_t radius, int32_t n_params, vo_rhs* out);
int32_t vo_rhs_custom_stencil_check(const char* body, int32_t radius, int32_t n_params, int32_t arith, char* log, int64_t log_cap);
int32_t vo_rhs_num_params(vo_rhs r);
int32_t vo_rhs_set_param(vo_rhs r, int32_t idx, double value);                            /* shared by all trajectories */
int32_t vo_rhs_set_param_array(vo_rhs r, int32_t idx, const double* host, int64_t n);     /* one value per trajectory */
int32_t vo_rhs_eval(vo_rhs r, double t, vo_ens x, vo_ens dx);                             /* f(t, &x, &mut dx) */
int32_t vo_rhs_destroy(vo_rhs r);

/* ---- solver: RK45Solver + ODESolver + AdaptiveODESolver (rk.rs:158-320, ode.rs:208-344) --------- */
/* ODEStep (ode.rs:42-48) */
#define VO_EV_STEP 0
#define VO_EV_CHKPT 1
#define VO_EV_REJECT 2
#define VO_EV_END 3
#define VO_EV_ERR 4
/* ODEState (ode.rs:34-38), aggregated over the ensemble: OK while any trajectory is still Ok. */
#define VO_STATE_OK 0
#define VO_STATE_DONE 1
#define VO_STATE_ERR 2
/* per-trajectory status bits (vo_solver_stats) */
#define VO_TRAJ_DONE 1
#define VO_TRAJ_NONFINITE 2   /* a non-finite error norm was seen (the reference accepts such steps, ode.rs:321-330) */
#define VO_TRAJ_STUCK 4       /* rejected at h == min_dt: the reference would loop forever here */

typedef struct vo_step_result {
    int64_t n_step;    /* trajectories whose event was Step (accepted) in this call */
    int64_t n_chkpt;
    int64_t n_reject;
    int64_t n_end;     /* trajectories that emitted End in this call */
    int64_t n_active;  /* trajectories not Done after this call */
    int32_t state;     /* VO_STATE_* */
    int32_t launches;  /* kernels launched by this call */
} vo_step_result;

/* RK45Solver::new_with_lc (rk.rs:248-262) with the tableau as an argument; x0 is cloned. Defaults as the
 * reference: x_err = Some, order 3.0, alpha 0.9, atol 1e-6, rtol 1e-4, min_dt 1e-6, max_dt 1.0,
 * t_list = [t0, tf], tgt_t = 0. */
int32_t vo_rk_create(vo_ctx ctx, vo_tableau tableau, vo_rhs rhs, double t0, double tf, vo_ens x0, double h,
                     vo_solver* out);
/* RK45Solver::new (rk.rs:229-231): the hard-wired RKF45 tables. */
int32_t vo_rk45_create(vo_ctx ctx, vo_rhs rhs, double t0, double tf, vo_ens x0, double h, vo_solver* out);
int32_t vo_solver_destroy(vo_solver s);
int32_t vo_solver_no_adaptive(vo_solver s);                                  /* rk.rs:233-237 */
int32_t vo_solver_with_tolerance(vo_solver s, double atol, double rtol);     /* ode.rs:298-306 */
int32_t vo_solver_with_step_range(vo_solver s, double dt_min, double dt_max);/* ode.rs:267-285 */
int32_t vo_solver_with_init_step(vo_solver s, double h);                     /* ode.rs:287-296 */
int32_t vo_solver_set_t_list(vo_solver s, const double* t_list, int32_t n);  /* pub field ODEData.t_list, ode.rs:89 */
int32_t vo_solver_set_order_alpha(vo_solver s, double order, double alpha);  /* ODEAdaptiveData::new / with_alpha, ode.rs:114-131 */
int32_t vo_solver_set_norm(vo_solver s, int32_t norm_kind);                  /* the user `Normed` impl, rk.rs:302 */
/* ... as a user-defined functor (any RHS, compiled-in family or custom: the solver's control kernels are re-compiled at run time
 * with the norm in them). `f` must outlive the solver. */
int32_t vo_solver_set_norm_custom(vo_solver s, vo_normfn f);
int32_t vo_solver_set_h_array(vo_solver s, const double* h_host, int64_t n); /* one initial step per trajectory */
/* Events (calls of step()/step_adaptive()) fused per kernel launch on the register-resident path. 0 (default) =
 * automatic: one per launch for vo_step, vo_step_adaptive and vo_step_many, which expose every event; 16 (lock-step) or 8 (per-trajectory
 * control) inside vo_run, which only promises the final state. k >= 1 forces k everywhere. */
int32_t vo_solver_set_events_per_launch(vo_solver s, int32_t k);
/* 0 = whole-attempt register-resident kernel when the RHS/tableau allow it (default), 1 = force the
 * stage-granular path (one fused kernel per RK stage over the K buffers), 2 = whole-step path for a single HEAT1D state
 * (N = 1; 4, 6 or 7 stages): all stages of a step in one kernel, the state read and written once (16 B per grid point instead
 * of 104 B for RK4); the same per-point operations in the same order as the stage path. */
int32_t vo_solver_set_path(vo_solver s, int32_t path);
/* ODEAdaptiveData.dx_norm (ode.rs:104, written at ode.rs:319 and read by nothing in the crate): 1 (default) keeps the error
 * norm of every trajectory's latest attempt for vo_solver_stats; 0 drops that 8-byte store per attempted trajectory-step. */
int32_t vo_solver_set_record_dx_norm(vo_solver s, int32_t on);
/* The reference sets prev_h = h on every adaptive attempt (update_step_size, ode.rs:202-205) and reads it in one place, the
 * Chkpt / End branch (checkpoint_update, ode.rs:192-195). The one-event adaptive kernels therefore write prev_h only for a
 * trajectory whose next event is a checkpoint (8 bytes per attempt less). That is invisible as long as a solver under
 * per-trajectory control is only ever stepped adaptively; a non-adaptive step() after step_adaptive() could reach a
 * checkpoint with a prev_h that was never written, so it returns VO_ERR_STATE unless mixed stepping was switched on (1)
 * before the first adaptive step — the kernels then store prev_h on every attempt like the reference. Default 0. */
int32_t vo_solver_set_mixed_stepping(vo_solver s, int32_t on);
/* The solver's state has one layout, the public one (SoA ensemble + per-trajectory controller arrays). 0 selects it and does
 * nothing else; any other value returns VO_ERR_UNSUPPORTED: the tile-blocked private copy of the state that 1 once selected for
 * the one-event adaptive sweep was removed, having measured no faster (the sweep moves 92-96 B per attempt and sits at 85 % of
 * the HBM copy rate on either layout). */
int32_t vo_solver_set_blocked(vo_solver s, int32_t on);

/* ODESolver::step (ode.rs:249-253) / AdaptiveODESolver::step_adaptive (ode.rs:337-341) applied to every
 * trajectory: ONE state-machine event per trajectory per call. res may be NULL. */
int32_t vo_step(vo_solver s, vo_step_result* res);
int32_t vo_step_adaptive(vo_solver s, vo_step_result* res);
/* step_adaptive (ode.rs:336-344) in its two halves, for ONE state vector held in pieces by several solvers (grid slabs with
 * ghost zones on several GPUs; single state N == 1, stage path). vo_adaptive_try runs step_size_of + try_step (rk.rs:90-155)
 * and returns the norm ACCUMULATOR of this piece's components [lo, hi) of x_err — sum of squares (VO_NORM_L2), sum of
 * magnitudes (L1) or maximum (LINF) — and the event; a Chkpt / End event is complete on return. After a Step event the caller
 * combines the pieces' accumulators (sum / max over ranks, with vo_group_allreduce or any communicator), finishes the norm
 * (square root for L2) and gives the SAME value to every piece: vo_adaptive_handle = handle_step_adaptive (ode.rs:311-334)
 * + apply_step (ode.rs:402-428). */
int32_t vo_adaptive_try(vo_solver s, int64_t lo, int64_t hi, double* acc, int32_t* event, vo_step_result* res /* filled for Chkpt / End */);
int32_t vo_adaptive_handle(vo_solver s, double dx_norm, vo_step_result* res);
/* `while let ODEState::Ok(_) = solver.step() {}` for the whole ensemble. max_calls <= 0: until Done.
 * res accumulates the event counts of all calls. */
int32_t vo_run(vo_solver s, int32_t adaptive, int64_t max_calls, vo_step_result* res);
/* Round-robin stepping of several independent ensembles ("batches") that share one ctx: `rounds` times, each solver
 * in turn advances by one launch (its events-per-launch calls of step()/step_adaptive()). Nothing is read back and
 * nothing synchronises; counts and states are picked up later by vo_run / vo_solver_stats / vo_current. */
int32_t vo_step_many(const vo_solver* solvers, int32_t n, int32_t adaptive, int64_t rounds);
/* ODESolver::current (ode.rs:216-218): borrowed view of x (valid until the next step) and the time range. */
int32_t vo_current(vo_solver s, double* t_min, double* t_max, vo_ens* x);
/* Checkpoint output (pub field ODEData.t_list + the Chkpt / End events, ode.rs:89-90, 165-176, 192-195): keep, for every
 * entry k of t_list, the state each trajectory shows through current() at its Chkpt / End event for t_list[k]. With
 * per-trajectory control the trajectories pass a checkpoint in different calls; the snapshot is complete once every
 * trajectory has passed it (vo_solver_stats' status / t tell). vo_solver_snapshot returns a non-owning ensemble view
 * (destroy it with vo_ens_destroy; the storage belongs to the solver). */
int32_t vo_solver_enable_snapshots(vo_solver s);
int32_t vo_solver_snapshot(vo_solver s, int32_t k, vo_ens* out);
/* Per-trajectory controller state; any pointer may be NULL. Host arrays of length N. */
int32_t vo_solver_stats(vo_solver s, int64_t* accepted, int64_t* rejected, double* t, double* h, double* dx_norm,
                        int32_t* status);
/* Reset to (t0, x0, h) for another run (re-clones x0 like the constructor). */
int32_t vo_solver_reset(vo_solver s, vo_ens x0);
/* One bare rk_step (rk.rs:90-155) at (t, dt) on the solver's current x: writes next_x, x_err (NULL to skip)
 * and the s stage derivatives K (NULL to skip) WITHOUT advancing. For kernel-level parity tests. */
int32_t vo_rk_try_step(vo_solver s, double t, double dt, vo_ens next_x, vo_ens x_err, vo_ens* K);

/* ---- exponential integrators (src/exp) ---------------------------------------------------------- */
/* ExponentialSplit / Commutator / NormedExponentialSplit (exp/mod.rs:11-54) for batched dense complex
 * systems on a shared basis: an operator L_i = sum_m coef[i][m] * B_m with M complex n x n matrices B_m
 * shared by the ensemble; `L` values are coefficient ensembles, exp(L) is lazy and map_exp applies the
 * scaled Taylor series of exp(L) to the state without forming U. States: complex n-vectors, AoS
 * [N][n] interleaved (re, im). n is 1 <= n <= 8 (one system per thread, FP64 in registers, a Taylor plan per system) or a
 * multiple of 8 (the solvers run n in {16, 24, 32, 40, 48, 64} on the FP64 tensor cores, by 16-system tiles); 9 <= n <= 15 and
 * other sizes return VO_ERR_BAD_ARG. 1 <= M <= 4. */
int32_t vo_split_basis_create(vo_ctx ctx, int32_t n, int32_t M, const double* basis /* [M][n][n] (re,im) */,
                              vo_split* out);
int32_t vo_split_destroy(vo_split sp);
/* structure constants for Commutator::commutator (exp/mod.rs:53): [B_a, B_b] = sum_c cs[a][b][c] B_c */
int32_t vo_split_set_commutator(vo_split sp, const double* cs /* [M][M][M] */);
int32_t vo_split_set_taylor_degree(vo_split sp, int32_t deg); /* 0 = automatic from theta = ||L||_1 bound */
/* map_exp(&exp(L), &x) (exp/mod.rs:23-25) for every system: coef [N][M] complex (host), psi device [N][n] complex. */
int32_t vo_map_exp(vo_split sp, const double* coef_host, int64_t N, void* psi_in_dev, void* psi_out_dev);
/* Compositions of exponentials — what the split combinators of exp/split_exp.rs:24-517 (CommutativeExpSplit, StrangSplit,
 * SemiComplexO4ExpSplit, TripleJumpExpSplit, RKNR4ExpSplit) reduce to once the two user splits A and B are disjoint index
 * sets of one basis: psi <- map_exp(exp(L_K-1), ... map_exp(exp(L_0), psi)) with K coefficient sets coef [K][N][M],
 * in ONE launch (the state never leaves registers between the K exponentials). */
int32_t vo_map_exp_seq(vo_split sp, const double* coef_host, int32_t K, int64_t N, void* psi_in_dev, void* psi_out_dev);

/* NormedExponentialSplit::norm (exp/mod.rs:37-45): 2-norm of each of the N states psi_dev [N][n] complex -> out_host[N]. */
int32_t vo_split_norm(vo_split sp, const void* psi_dev, int64_t N, double* out_host);
/* Commutator::commutator (exp/mod.rs:47-54) on operators given as coefficient vectors la, lb, out: [N][M] complex (host). */
int32_t vo_split_commutator(vo_split sp, const double* la, const double* lb, int64_t N, double* out);

/* ---- the same traits for GENERAL dense operators: every system owns its n x n complex L and U (no shared basis, no closure
 * under commutation assumed). An operator ensemble is a vo_ens of one row of 2 n^2 N doubles ([N][n][n] complex, row-major,
 * interleaved), so LinearCombination on operators is vo_lc_* on those ensembles; n % 8 == 0, n <= 64. Products run on the FP64
 * tensor cores (DMMA), one CTA per system with both operands in shared memory. -------------------------------------------------- */
int32_t vo_split_dense_create(vo_ctx ctx, int32_t n, int64_t N, vo_split* out);
int32_t vo_dense_lin_zero(vo_split sp, vo_ens* out);                                     /* lin_zero, exp/mod.rs:20 */
/* L_i = sum_m coef[i][m] B_m: operators of a shared-basis split (coef [N][M] complex, host) as dense operators */
int32_t vo_dense_assemble(vo_split sp, vo_split basis, const double* coef_host, vo_ens L);
/* exp (exp/mod.rs:23): explicit U = exp(L) by scaling and squaring — L / 2^s with ||.||_1 <= 1/2, Taylor series to 2^-53, s
 * squarings: (degree + s) complex GEMMs of 8 n^3 flops per system. */
int32_t vo_dense_exp(vo_split sp, vo_ens L, vo_ens U);
int32_t vo_dense_multi_exp(vo_split sp, vo_ens L, const double* k_arr, int32_t K, const vo_ens* U_out); /* exp(k l) for every k, exp/mod.rs:28-34 */
int32_t vo_dense_map_exp(vo_split sp, vo_ens U, const void* psi_in_dev, void* psi_out_dev); /* map_exp, exp/mod.rs:25: y_i = U_i x_i */
int32_t vo_dense_commutator(vo_split sp, vo_ens La, vo_ens Lb, vo_ens out);              /* commutator, exp/mod.rs:53: La Lb - Lb La */
/* vo_split_norm (NormedExponentialSplit::norm) takes a dense split as well. */

/* Generator family replacing the closures of exp/magnus.rs:12,32 and exp/cfm.rs:54:
 *   L_i(t) = B_0 + sum_{m=1}^{M_gen-1} amp_im * cos(omega_im * t + phase_im) * B_m ,  gp = [N][M_gen-1][3]. */
#define VO_EXP_MIDPOINT 0 /* MidpointExpLinearSolver, exp/magnus.rs:85-148 */
#define VO_EXP_CFM4 1     /* ExpCFMSolver, exp/cfm.rs:102-224 */
#define VO_EXP_MAGNUS42 2 /* MagnusExpLinearSolver, exp/magnus.rs:151-285 */
#define VO_EXP_SPLIT_MIDPOINT 3 /* ExpSplitMidpointSolver, exp/split_exp.rs:520-562, 613-685 (literal: f at t, both splits by dt/2) */
#define VO_EXP_CFM_TABLE 4      /* cfm_general (exp/cfm.rs:43-100) with the caller's nodes and weights: vo_exp_set_cfm_tables */
#define VO_EXP_SPLIT_CFM 5      /* split_cfm (exp/split_exp.rs:568-609), the BAB commutator-free split: vo_exp_set_split_cfm_tables */
int32_t vo_exp_create(vo_ctx ctx, vo_split sp, int32_t scheme, int32_t M_gen, const double* gp_host, int64_t N,
                      double t0, double tf, const double* psi0_host /* [N][n] (re,im) */, double h, vo_expsolver* out);
int32_t vo_exp_destroy(vo_expsolver s);
/* The generator closure itself (`FnMut(T) -> L`, exp/cfm.rs:54, exp/magnus.rs:12,32) in place of the compiled-in cosine family:
 * `body` is CUDA C++ for statements that assign `g[1] .. g[M_gen-1]`, the real coefficients of L(t) = B_0 + sum_m g[m] B_m,
 * from `const double t` and `const double* p` (this system's 3 (M_gen - 1) parameters as handed to vo_exp_create). It is
 * compiled at run time (NVRTC, sm_100a) into the same tensor-core kernel the built-in family runs in; compile errors come
 * back through vo_last_error. vo_exp_generator_check compiles without a ctx or a GPU (1 <= n <= 8, or n a multiple of 8 up to
 * 64; M basis matrices) and returns the cubin size (> 0) or a VO_ERR_* code with the compiler log in `log`. */
int32_t vo_exp_set_generator(vo_expsolver s, const char* body);
/* The systems are independent, so their order on the device is free — and it matters: a tile of 16 systems runs the largest
 * Taylor degree among them. After vo_exp_set_order(s, perm, N) the solver treats device slot j as the caller's system perm[j]:
 * vo_exp_reset / vo_exp_current / vo_exp_stats speak the caller's order (the reordering runs on the device). The psi0 and gp
 * handed to vo_exp_create are in device order; call this right after creating the solver. */
int32_t vo_exp_set_order(vo_expsolver s, const int64_t* perm, int64_t n);
/* Dynamic grouping: before every event the systems are sorted on the device by the 1-norm bound of their exponent at the coming
 * step (one small kernel + a radix sort of N keys, ~1 % of a step of config 5) and the kernel forms its 16-system tiles in that
 * order. A tile runs the Taylor degree of its largest theta, so tiles of equal theta execute what their systems need and no more
 * (static grouping by drive amplitude cannot follow the phases). Results are those of any other order to rounding; buffers and
 * statistics stay in the caller's order. Compiled-in generator family only (a run-time compiled generator keeps the static order).
 * For 1 <= n <= 8 every system runs its own Taylor plan and there are no tiles to group: the switch is accepted and does nothing. */
int32_t vo_exp_set_dynamic_grouping(vo_expsolver s, int32_t on);
int32_t vo_exp_generator_check(const char* body, int32_t n, int32_t M, char* log, int64_t log_cap);
/* The arguments `c`, `alpha`, `alph_err` of cfm_general (exp/cfm.rs:47-52): k <= 4 nodes, alpha [rows][k] with rows <= 8
 * exponentials per step, alph_err [rows_err][k] (rows_err <= min(rows, 4)) or NULL for no embedded solution. A step is
 *   x <- exp(dt sum_q alpha[rows-1][q] L(t + c_q dt)) ... exp(dt sum_q alpha[0][q] L(t + c_q dt)) x
 * with every exponent formed by cfm_exp's operations in its order (cfm.rs:31-37). Mismatched shapes return VO_ERR_SHAPE with the
 * reference's panic message. VO_EXP_CFM4 solvers are created with C_GAUSS_LEGENDRE_4 / CFM_R4_J2_GL / CFM_R2_J1_GL already set. */
int32_t vo_exp_set_cfm_tables(vo_expsolver s, const double* c, int32_t k, const double* alpha, int32_t rows, const double* alpha_err, int32_t rows_err);
/* split_cfm's `c`, `rho` [stages][k], `sigma` [stages + 1][k] (split_exp.rs:571-573): per step B(sigma_0) A(rho_0) B(sigma_1) ...
 * A(rho_{stages-1}) B(sigma_stages), A and B being the two index sets of vo_exp_set_split_mask. 2 stages + 1 <= 8. */
int32_t vo_exp_set_split_cfm_tables(vo_expsolver s, const double* c, int32_t k, const double* rho, const double* sigma, int32_t stages);
/* The coefficient tables of src/dat/mod.rs:3-6, 66-81 (quad::C_GAUSS_LEGENDRE_4, cfqm::*) as the reference spells them. */
#define VO_CFM_C_GAUSS_LEGENDRE_4 0
#define VO_CFM_R2_J1_GL 1
#define VO_CFM_R4_J2_GL 2
#define VO_CFM_BLANES17_R4_J4 3
int32_t vo_cfm_builtin_table(int32_t which, double* out /* [rows][cols], nullable */, int32_t* rows, int32_t* cols);
/* VO_EXP_SPLIT_MIDPOINT: bit m of a_mask set <=> basis matrix m belongs to split A (the rest form split B). */
int32_t vo_exp_set_split_mask(vo_expsolver s, uint32_t a_mask);
/* VO_EXP_MAGNUS42 on generators that are NOT closed under commutation on the shared basis: 1 makes magnus_42 (exp/magnus.rs:28-83)
 * assemble L(t) at its two nodes per system and form commutator(l0, l1) (magnus.rs:55) densely on the tensor cores — two
 * n x n complex products per system and step — instead of expanding it through vo_split_set_commutator's structure tensor.
 * n % 8 == 0, n <= 64; compiled-in generator family only. */
int32_t vo_exp_set_dense_commutator(vo_expsolver s, int32_t on);
/* ... or never formed at all: with L0, L1 the generator at the two Gauss nodes, a Taylor term of exp(Omega) needs only
 * Omega T = b1 (L0 + L1) T + b2 (L0 (L1 T) - L1 (L0 T)) — three passes over the shared basis per term, each M tile products on the
 * tensor cores inside exp_step_kernel (the same machinery as the commutator-free schemes: 16 systems per tile, basis resident in
 * shared memory). No closure under commutation assumed, no structure tensor, no n x n matrix per system; works with a run-time
 * compiled generator. 1.8x the throughput of the dense commutator on config 5's shape (18.0 against 32.4 ms per step of 10^5 systems). */
int32_t vo_exp_set_applied_commutator(vo_expsolver s, int32_t on);
/* MagnusExpLinearSolver::norm AS WRITTEN (exp/magnus.rs:274-276): it takes the norm of adaptive_dat.dx, a clone of x0 that
 * try_step never writes (the embedded error goes to self.x_err, magnus.rs:249-250), so the controller sees the constant ||x0||:
 * with rtol <= ||x0|| every attempt is rejected, with rtol > ||x0|| every attempt is accepted and h grows by
 * clamp(0.9 (rtol / ||x0||)^(1/3), 0.3, 2) per step. Off by default: the solvers here give the controller the embedded error it
 * was meant to see. On: the reference's literal behaviour, for comparisons. Magnus only. */
int32_t vo_exp_set_literal_norm(vo_expsolver s, int32_t on);
/* NormedExponentialSplit::norm / ExpCFMSolver's NormFn (exp/mod.rs:37-45, exp/cfm.rs:105, 214-216) as a user-defined functor:
 * exp_step_kernel is re-compiled at run time with it (together with the generator of vo_exp_set_generator, if any).
 * Not available with vo_exp_set_dense_commutator. */
int32_t vo_exp_set_norm_custom(vo_expsolver s, vo_normfn f);
int32_t vo_exp_no_adaptive(vo_expsolver s);                              /* exp/cfm.rs:157-161 */
int32_t vo_exp_with_tolerance(vo_expsolver s, double atol, double rtol);
int32_t vo_exp_with_step_range(vo_expsolver s, double dt_min, double dt_max);
int32_t vo_exp_step(vo_expsolver s, vo_step_result* res);
int32_t vo_exp_step_adaptive(vo_expsolver s, vo_step_result* res);
int32_t vo_exp_run(vo_expsolver s, int32_t adaptive, int64_t max_calls, vo_step_result* res);
int32_t vo_exp_current(vo_expsolver s, double* t_min, double* t_max, double* psi_host /* nullable */);
/* The states in the caller's order as a non-owning device view (one row of 2 * n * N doubles, [N][n] complex interleaved;
 * destroy it with vo_ens_destroy; valid until the next step) — what vo_group_gather_placed takes for a sharded ensemble. */
int32_t vo_exp_current_device(vo_expsolver s, vo_ens* out);
int32_t vo_exp_stats(vo_expsolver s, int64_t* accepted, int64_t* rejected, double* t, double* h, double* dx_norm);
/* Back to (t0, psi0, h): psi0_host NULL re-uses the state given at creation, otherwise uploads a new one. */
int32_t vo_exp_reset(vo_expsolver s, const double* psi0_host);
void* vo_exp_state_device_ptr(vo_expsolver s);
/* Output times: the pub field ODEData.t_list (ode.rs:89-90) in place of [t0, tf] (ode.rs:144), as vo_solver_set_t_list. Steps are
 * clipped to land on every entry (step_size_of / check_step, ode.rs:165-176, 389-399); each system raises Chkpt at every entry
 * before the last and End at the last (ode.rs:192-195), in whatever call it gets there under adaptive control. 1 <= n <= 65535
 * entries (VO_ERR_UNSUPPORTED above, VO_ERR_BAD_ARG for n < 1 or NULL). Refused with VO_ERR_STATE once a step / run has begun;
 * vo_exp_reset rewinds every system to entry 0 and accepts a new list. */
int32_t vo_exp_set_t_list(vo_expsolver s, const double* t_list, int32_t n);
/* Checkpoint output: keep, for every entry k of t_list, the state each system shows through vo_exp_current at its Chkpt / End event
 * for t_list[k] (the kernels write it at the event, also in the middle of a fused vo_exp_run launch). Storage [len][N][n] complex,
 * zeroed when enabled and re-allocated by vo_exp_set_t_list; vo_exp_reset keeps the contents until the next run overwrites them.
 * Snapshot k is complete once every system has passed t_list[k] (vo_exp_stats' t tells). Both readers speak the caller's order
 * (vo_exp_set_order: the kernels write each system to its caller's row) and return VO_ERR_BAD_ARG for k outside the list and
 * VO_ERR_STATE when snapshots are off. vo_exp_snapshot copies [N][n] (re, im) to the host; vo_exp_snapshot_device returns a
 * non-owning device view of one row of 2 n N doubles (destroy it with vo_ens_destroy; the storage belongs to the solver), what
 * vo_group_gather_placed takes. */
int32_t vo_exp_enable_snapshots(vo_expsolver s);
int32_t vo_exp_snapshot(vo_expsolver s, int32_t k, double* psi_host /* [N][n] (re,im) */);
int32_t vo_exp_snapshot_device(vo_expsolver s, int32_t k, vo_ens* out);
/* Observables (no reference counterpart: ODEData keeps checkpoints and nothing else). K operators O_k, [K][n][n] complex row-major
 * and shared by the ensemble like the basis, 1 <= K <= VO_EXP_MAX_OBS. At every Chkpt / End event for t_list[j] the kernels compute,
 * from the state a snapshot would keep (whether or not snapshots are on),
 *     e[j][i][k] = sum_r conj(psi_r) sum_c O_k[r][c] psi_c
 * complex and not normalised by <psi|psi>, so non-Hermitian operators (sigma_-, |0><1|) work; for a Hermitian O_k the imaginary part
 * is rounding. vo_exp_set_observables uploads the operators and allocates [len][N][K] complex, zeroed; vo_exp_set_t_list re-allocates
 * it and vo_exp_reset keeps the contents until the next run overwrites them, as for the snapshots. K = 0 with ops NULL turns
 * observables off and frees the storage; K < 0, K > VO_EXP_MAX_OBS or K > 0 with ops NULL return VO_ERR_BAD_ARG. Refused with
 * VO_ERR_STATE once a step / run has begun, accepted again after vo_exp_reset. Both readers speak the caller's order and return
 * VO_ERR_BAD_ARG for j outside the list and VO_ERR_STATE when observables are off. vo_exp_expectation copies [N][K] (re, im) to the
 * host; vo_exp_expectation_device returns a non-owning device view of one row of 2 K N doubles (destroy it with vo_ens_destroy),
 * what vo_group_gather_placed takes. */
#define VO_EXP_MAX_OBS 8
int32_t vo_exp_set_observables(vo_expsolver s, int32_t K, const double* ops /* [K][n][n] (re,im) row-major */);
int32_t vo_exp_expectation(vo_expsolver s, int32_t j, double* host /* [N][K] (re,im) */);
int32_t vo_exp_expectation_device(vo_expsolver s, int32_t j, vo_ens* out);

/* ---- multi-GPU: one ensemble sharded by trajectory over the GPUs of one box ------------------------------------------ */
/* The reference has no parallelism of any kind; what replaces "one solver object per trajectory, run them in any order" is
 * rank r of G integrating the contiguous range vo_group_shard_range(N, r, G) of the ensemble. Trajectories are independent
 * (nothing in rk_step, handle_step_adaptive, cfm_general or magnus_42 couples them), so stepping needs NO collective; NCCL
 * over NVLink / NVSwitch appears only at the ends of a solve: the gather of the final states, the reduction of the counters
 * (and one scalar per attempt for a domain-decomposed adaptive state, vo_group_allreduce).
 * Two ways to form a group:
 *   one process per GPU   rank 0 calls vo_group_unique_id, the host program ships the VO_GROUP_ID_BYTES to the other ranks,
 *                         every rank calls vo_group_create_rank(its ctx, id, rank, world) — the per-member arrays below then
 *                         have ONE entry;
 *   one process, G GPUs   vo_group_create_local(ctxs, G): one ctx per device, ncclCommInitAll; the per-member arrays have G
 *                         entries (entry i belongs to ctxs[i] = rank i) and one host thread drives all GPUs. */
#define VO_GROUP_ID_BYTES 128
int32_t vo_group_unique_id(void* id_out /* VO_GROUP_ID_BYTES */);
int32_t vo_group_create_rank(vo_ctx ctx, const void* id, int32_t rank, int32_t world, vo_group* out);
int32_t vo_group_create_local(const vo_ctx* ctxs, int32_t n, vo_group* out);
int32_t vo_group_destroy(vo_group g);
int32_t vo_group_world(vo_group g);
int32_t vo_group_local_members(vo_group g);
int32_t vo_group_member_rank(vo_group g, int32_t member);
const char* vo_group_last_error(vo_group g);
int32_t vo_group_nccl_version(void);
/* contiguous ceil(N/G) ranges */
int32_t vo_group_shard_range(int64_t n_total, int32_t rank, int32_t world, int64_t* lo, int64_t* hi);
/* Upload the whole initial ensemble ([n_total][d] or [d][n_total] host array on the root) once and hand every member its
 * shard over NVLink: local_out[i] is member i's ensemble of shape (d, shard length). Synchronous on return. */
int32_t vo_group_scatter(vo_group g, const double* host_in, int32_t layout, int64_t d, int64_t n_total, int32_t root, const vo_ens* local_out);
/* `while let Ok(_) = solver.step() {}` on every local shard (vo_run), then vo_group_reduce_stats if out != NULL. */
typedef struct vo_group_stats {
    int64_t accepted, rejected;                 /* sums over the whole ensemble */
    int64_t n_traj, n_done, n_nonfinite, n_stuck; /* trajectories in all, and with each VO_TRAJ_* bit set */
    double t_min, t_max;
} vo_group_stats;
int32_t vo_group_run(vo_group g, const vo_solver* local, int32_t adaptive, int64_t max_calls, vo_group_stats* out);
/* The final gather: local[i] is member i's shard (for a solver: the ensemble vo_current returns). The root receives the whole
 * ensemble — as a device ensemble [d][n_total] (vo_group_gather_device: a view into the group's gather buffer, valid until the
 * next gather, destroy it with vo_ens_destroy; NULL on the other ranks), or in host_out through ONE device-to-host copy
 * (vo_group_gather: synchronous on the root; pinned host memory makes the copy run at PCIe speed). Enqueued on each member's
 * stream, i.e. after the solve. */
int32_t vo_group_gather_device(vo_group g, const vo_ens* local, int64_t n_total, int32_t root, vo_ens* out);
int32_t vo_group_gather(vo_group g, const vo_ens* local, int64_t n_total, int32_t root, double* host_out, int32_t layout);
/* The general, asynchronous form: rank r holds rows[r] trajectories (any sizes; local[i]->n == rows[rank of member i]; the
 * ensembles may live on other contexts of the member's device — order the group's ctx after them with vo_ctx_wait_for) and
 * the root places them at row row_off[r] of a host array of host_n trajectories. One message per shard, one device-to-host
 * copy per shard straight into its place, nothing synchronises: a pipelined solve gathers its chunks one by one while later
 * chunks still integrate. vo_group_sync waits for everything enqueued on the group's streams. */
int32_t vo_group_gather_placed(vo_group g, const vo_ens* local, int32_t root, const int64_t* rows /* [world] */, const int64_t* row_off /* [world] */,
                               double* host_out, int32_t layout, int64_t host_n);
/* Round-robin sharding (rank r holds trajectories r, r + G, r + 2G, ... of a block of `tot` consecutive ones: the static
 * interleave that balances an adaptive ensemble whose cost varies along the trajectory index): the root interleaves the
 * shards on the device into the block's natural order and copies the block to rows [row0, row0 + tot) of the host array.
 * local[i]->n == ceil((tot - rank) / G). Asynchronous like vo_group_gather_placed. */
int32_t vo_group_gather_interleaved(vo_group g, const vo_ens* local, int32_t root, int64_t tot, int64_t row0, double* host_out, int32_t layout, int64_t host_n);
int32_t vo_group_sync(vo_group g);
/* all-reduce of the per-shard counters; every rank receives the totals */
int32_t vo_group_reduce_stats(vo_group g, const vo_solver* local, vo_group_stats* out);
/* in-place all-reduce of n <= 32 doubles per member, host values in and out ([members][n]); op 0 sum, 1 max, 2 min */
int32_t vo_group_allreduce(vo_group g, double* host_inout, int32_t n, int32_t op);

#ifdef __cplusplus
}
#endif
#endif /* VECODE_B200_H */
