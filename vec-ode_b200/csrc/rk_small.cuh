// rk_small.cuh — whole-attempt Runge-Kutta kernel for ensembles of small systems (d <= 8).
//
// One thread owns one trajectory. A launch executes up to `k_events` calls of the reference's
// `step()` / `step_adaptive()` (src/base/ode.rs:249-253, 337-341) for that trajectory with the state, all
// s stage derivatives and the controller scalars in REGISTERS: state is read from HBM once and written
// once per launch (SoA, coalesced: lane i touches component c at x[c*N + i]). The tableau is a by-value
// kernel parameter, so after full unrolling every coefficient is a constant-bank operand.
//
// Everything the reference does between two calls is reproduced per trajectory:
//   step_size_of/check_step (ode.rs:165-176, 389-399)  ->  Step(dt) | Chkpt | End
//   rk_step (rk.rs:90-155)                             ->  X_b, X_berr, x_err in the reference's op order
//   handle_step_adaptive (ode.rs:311-334)              ->  norm, f = rtol/|err|, h update, Reject iff f <= 1
//   apply_step (ode.rs:402-428)                        ->  advance / checkpoint_update
// Rejected or finished lanes are masked: they neither advance nor write state.
#pragma once
#include "common.cuh"
#include "rhs.cuh"
#include "tile_pipe.cuh"

#define VO_WORD_TGT_MASK 0xffffu
#define VO_WORD_STATUS_SHIFT 16
#define VO_EV_SLOTS 32
#define VO_INLINE_TLIST 8

// Per-trajectory controller state (device arrays of length N).
struct CtlArrays {
    double* t;
    double* h;
    double* prev_h;
    double* dx_norm;
    uint32_t* n_accept;
    uint32_t* n_reject;
    uint32_t* word;  // bits 0..15: tgt_t (ode.rs:90); bits 16..: VO_TRAJ_* status
};

// Controller constants shared by the ensemble (ODEAdaptiveData, ode.rs:98-110) + launch options.
struct CtlShared {
    double rtol, alpha, pw, min_dt, max_dt;
    double inv_rtol, inv_rtol2;  // 1/rtol, 1/rtol^2 (host-computed; the FAST controller works on (dx_norm/rtol)^2)
    double t_list_inline[VO_INLINE_TLIST];
    const double* t_list;  // device copy when n_tlist > VO_INLINE_TLIST
    int n_tlist;
    int norm_kind;
    int adaptive;      // step_adaptive() vs step()
    int use_err;       // tableau has b_err AND the solver still holds x_err (rk.rs:136-151)
    int k_events;      // calls fused into this launch
    int count_events;  // accumulate vo_step_result counters
    int pw_is_third;   // pw == 1.0/3.0 exactly (the order RK45Solver hard-wires, rk.rs:258-260)
    int record_dx_norm;  // keep ODEAdaptiveData.dx_norm (ode.rs:104) per trajectory
    int lazy_prev_h;     // two-trajectory control kernels: write prev_h only when its one reader (the Chkpt / End branch) comes next
    double* snap;        // optional [n_tlist][snap_stride]: the state ([d][N]) each trajectory shows at its Chkpt / End events, else NULL
    int64_t snap_stride; // d * N rounded up to even, so that every entry's block starts 16-byte aligned
};

// Event counters, VO_EV_SLOTS copies 128 bytes apart to spread the atomics (host sums the slots).
struct EvSlot {
    unsigned long long n_step, n_chkpt, n_reject, n_end, n_stuck;
    unsigned long long pad[11];
};

// t_list lookups (ode.rs:165-176 reads t_list[tgt_t] at the head of every call). The list is a kernel parameter (or a
// global array when it is long); indexing it with a per-lane tgt would be a generic load with L1/L2 latency at the head
// of every attempt's dependency chain (14 % of the stall samples of the DoPri5 kernel). The kernels copy the inline list
// into shared memory once per CTA and read it with ld.shared.
struct TList {
    const double* glob;  // non-NULL: long list in global memory
    uint32_t smem;       // shared-window address of the CTA's copy of the inline list
    __device__ __forceinline__ double at(int k) const {
        if (glob) return __ldg(glob + k);
        double v;
        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(smem + 8u * (uint32_t)k) : "memory");
        return v;
    }
};
// Every thread calls it before the first __syncthreads() of the kernel.
__device__ __forceinline__ TList tlist_stage(const CtlShared& cs, double* s_tl) {
    if (threadIdx.x < VO_INLINE_TLIST) s_tl[threadIdx.x] = cs.t_list_inline[threadIdx.x];
    return TList{cs.n_tlist > VO_INLINE_TLIST ? cs.t_list : nullptr, (uint32_t)__cvta_generic_to_shared(s_tl)};
}

template <bool STRICT, int D> __device__ __forceinline__ double err_norm(const double (&e)[D], int kind) {
    using A = Ar<STRICT>;
    double acc = 0.0;
    if (kind == VO_NORM_L2) {
#pragma unroll
        for (int c = 0; c < D; ++c) acc = A::add(acc, A::mul(e[c], e[c]));
        return sqrt(acc);
    }
    if (kind == VO_NORM_LINF) {
#pragma unroll
        for (int c = 0; c < D; ++c) acc = fmax(acc, fabs(e[c]));
        return acc;
    }
    if (kind == VO_NORM_L1) {
#pragma unroll
        for (int c = 0; c < D; ++c) acc = A::add(acc, fabs(e[c]));
        return acc;
    }
#ifdef VO_USER_NORM  // the caller's `Normed` impl (ode.rs:9-11, rk.rs:302-304), compiled in with the kernel: finish(JOIN_c map(e_c, c))
    if (kind == VO_NORM_CUSTOM) {
#pragma unroll
        for (int c = 0; c < D; ++c) {
            const double m = VoUserNorm::map(e[c], 0.0, c, D);
            acc = VoUserNorm::JOIN == 1 ? fmax(acc, m) : A::add(acc, m);
        }
        return VoUserNorm::finish(acc, D);
    }
#endif
    // VO_NORM_HYPOT
    if (D == 2) return hypot(e[0], e[D - 1]);
#pragma unroll
    for (int c = 0; c + 1 < D; c += 2) {
        const double m = hypot(e[c], e[c + 1]);
        acc = A::add(acc, A::mul(m, m));
    }
    return sqrt(acc);
}

template <bool STRICT, int D> __device__ __forceinline__ double err_sumsq(const double (&e)[D]) {
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < D; ++c) acc = Ar<STRICT>::add(acc, Ar<STRICT>::mul(e[c], e[c]));
    return acc;
}

// v[c] = (sum_{j<n} k[j]*K[j][c]) * dt + x0[c]  in the reference's order (lc.rs:20-54, rk.rs:123-124).
template <bool STRICT, int D, int SM>
__device__ __forceinline__ void combine(const double* __restrict__ k, int n, const double (&K)[SM][D], double dt, const double (&x0)[D],
                                        double (&v)[D]) {
    using A = Ar<STRICT>;
    if (STRICT) {
#pragma unroll
        for (int c = 0; c < D; ++c) v[c] = A::mul(k[0], K[0][c]);
#pragma unroll
        for (int j = 1; j < SM; ++j)
            if (j < n) {
#pragma unroll
                for (int c = 0; c < D; ++c) v[c] = A::axpy(v[c], k[j], K[j][c]);
            }
    } else {
        // FMA chain. Zero coefficients are NOT tested for here: a data-dependent skip costs a DSETP + selects per term,
        // more than the FMA it would save (the stage-path kernels, which save a whole HBM pass per zero, do skip).
#pragma unroll
        for (int c = 0; c < D; ++c) v[c] = k[0] * K[0][c];
#pragma unroll
        for (int j = 1; j < SM; ++j)
            if (j < n) {
#pragma unroll
                for (int c = 0; c < D; ++c) v[c] = fma(k[j], K[j][c], v[c]);
            }
    }
#pragma unroll
    for (int c = 0; c < D; ++c) v[c] = A::add(A::mul(v[c], dt), x0[c]);
}

// The two halves of `combine`: the weighted sum of the stage derivatives, and `* dt + x0`. Splitting them lets a final
// combination whose first s-1 weights equal the last row of the tableau (TableauDev::reuse) start from the last stage's sum.
template <bool STRICT, int D, int SM>
__device__ __forceinline__ void combine_sum(const double* __restrict__ k, int n, const double (&K)[SM][D], double (&v)[D]) {
    using A = Ar<STRICT>;
#pragma unroll
    for (int c = 0; c < D; ++c) v[c] = A::mul(k[0], K[0][c]);
#pragma unroll
    for (int j = 1; j < SM; ++j)
        if (j < n) {
#pragma unroll
            for (int c = 0; c < D; ++c) v[c] = A::axpy(v[c], k[j], K[j][c]);
        }
}
template <bool STRICT, int D> __device__ __forceinline__ void combine_finish(const double (&v)[D], double dt, const double (&x0)[D], double (&out)[D]) {
    using A = Ar<STRICT>;
#pragma unroll
    for (int c = 0; c < D; ++c) out[c] = A::add(A::mul(v[c], dt), x0[c]);
}
// out = ((vsum + k_last * K_last) * dt) + x0: the tail of a final combination that shares its first s-1 terms with vsum
template <bool STRICT, int D>
__device__ __forceinline__ void combine_tail(const double (&vsum)[D], double k_last, const double (&K_last)[D], double dt, const double (&x0)[D], double (&out)[D]) {
    using A = Ar<STRICT>;
#pragma unroll
    for (int c = 0; c < D; ++c) out[c] = A::add(A::mul(A::axpy(vsum[c], k_last, K_last[c]), dt), x0[c]);
}

// Rust's `v.max(lo)` / `v.min(hi)` for a bound that is not NaN: a NaN v yields the bound (ode.rs:321-324). A compare and two
// selects; CUDA's fmax / fmin cost seven instructions each for the NaN cases of BOTH operands.
__device__ __forceinline__ double at_least(double v, double lo) { return v > lo ? v : lo; }
__device__ __forceinline__ double at_most(double v, double hi) { return v < hi ? v : hi; }

// rk_step (src/base/rk.rs:90-155). On return xf is the state the reference propagates (X_berr when the error
// branch runs, else X_b) and xe = X_b - X_berr.
template <class RHS, int S, bool STRICT>
__device__ __forceinline__ void rk_attempt(const TableauDev& tb, bool use_err, double t, double dt, const double (&x0)[RHS::D],
                                           const double (&p)[RHS::NP], double (&xf)[RHS::D], double (&xe)[RHS::D]) {
    using A = Ar<STRICT>;
    constexpr int D = RHS::D;
    constexpr int SM = S > 0 ? S : VO_MAX_STAGES;
    const int s = S > 0 ? S : tb.s;
    double K[SM][D], vlast[D];
    RHS::template eval<STRICT>(t, x0, K[0], p);  // rk.rs:111
#pragma unroll
    for (int c = 0; c < D; ++c) vlast[c] = 0.0;
#pragma unroll
    for (int i = 1; i < SM; ++i) {
        if (i < s) {
            const double* row = &tb.ac[i * s];
            const double ti = A::add(t, A::mul(row[i], dt));  // rk.rs:119
            double v[D], xs[D];
            combine_sum<STRICT, D, SM>(row, i, K, v);         // rk.rs:121-122
            combine_finish<STRICT, D>(v, dt, x0, xs);         // rk.rs:123-124
            if (S > 0 && i == S - 1) {
#pragma unroll
                for (int c = 0; c < D; ++c) vlast[c] = v[c];
            }
            RHS::template eval<STRICT>(ti, xs, K[i], p);      // rk.rs:127
        }
    }
    // the final combinations (rk.rs:131-133, 143-146); with the first-same-as-last structure their first s-1 terms are vlast
    if (S > 1 && (tb.reuse & 2)) combine_tail<STRICT, D>(vlast, tb.b[S > 1 ? S - 1 : 0], K[S > 1 ? S - 1 : 0], dt, x0, xf);
    else combine<STRICT, D, SM>(tb.b, s, K, dt, x0, xf);      // rk.rs:131-133
    if (use_err) {                                            // rk.rs:136-151
#pragma unroll
        for (int c = 0; c < D; ++c) xe[c] = xf[c];            // swap: xe := X_b
        if (S > 1 && (tb.reuse & 1)) combine_tail<STRICT, D>(vlast, tb.b_err[S > 1 ? S - 1 : 0], K[S > 1 ? S - 1 : 0], dt, x0, xf);
        else combine<STRICT, D, SM>(tb.b_err, s, K, dt, x0, xf);   // xf := X_berr
#pragma unroll
        for (int c = 0; c < D; ++c) xe[c] = A::sub(xe[c], xf[c]);
    }
}

// ---- lock-step fixed-step kernel -----------------------------------------------------------------------------
// Every trajectory takes the same (t, dt) sequence, which the host has already derived with the reference's state
// machine (ode.rs:165-176, 389-399), so the kernel carries no control arithmetic at all: per trajectory it moves
// 2*d*8 bytes and executes the rk_step FLOPs, nothing else. Persistent grid: each thread walks trajectories
// i, i+stride, ... and loads the NEXT trajectory's state before integrating the current one, so the HBM latency of
// iteration n+1 hides behind the FP64 work of iteration n.
#define VO_MAX_FUSED 32
struct StepList {
    int n;        // steps fused into this launch (<= VO_MAX_FUSED)
    int use_err;  // propagate X_berr (rk.rs:142-146) instead of X_b
    double t[VO_MAX_FUSED];
    double dt[VO_MAX_FUSED];
};

template <class RHS> __device__ __forceinline__ void lane_load(const double* __restrict__ x, int64_t N, const RhsParams& rp, int64_t i,
                                                               double (&xc)[RHS::D], double (&p)[RHS::NP]) {
#pragma unroll
    for (int c = 0; c < RHS::D; ++c) xc[c] = x[c * N + i];
    load_params<RHS::NP>(rp, i, p);
}

template <class RHS, int S, bool STRICT>
__global__ void __launch_bounds__(128) rk_fixed_kernel(double* __restrict__ x, int64_t N, const __grid_constant__ TableauDev tb,
                                                       const __grid_constant__ RhsParams rp, const __grid_constant__ StepList sl) {
    constexpr int D = RHS::D;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double xc[D], p[RHS::NP], xn[D], pn[RHS::NP];
    if (i < N) lane_load<RHS>(x, N, rp, i, xc, p);
    while (i < N) {
        const int64_t j = i + stride;
        if (j < N) lane_load<RHS>(x, N, rp, j, xn, pn);  // prefetch the next trajectory of this thread
        for (int e = 0; e < sl.n; ++e) {
            double xf[D], xe[D];
            rk_attempt<RHS, S, STRICT>(tb, sl.use_err != 0, sl.t[e], sl.dt[e], xc, p, xf, xe);
#pragma unroll
            for (int c = 0; c < D; ++c) xc[c] = xf[c];
        }
#pragma unroll
        for (int c = 0; c < D; ++c) x[c * N + i] = xc[c];
#pragma unroll
        for (int c = 0; c < D; ++c) xc[c] = xn[c];
#pragma unroll
        for (int q = 0; q < RHS::NP; ++q) p[q] = pn[q];
        i = j;
    }
}

// ---- per-trajectory control kernel ---------------------------------------------------------------------------
// alpha * f^pw (ode.rs:133-135). STRICT keeps the general pow of the reference's `powf` (accepted / rejected counts
// then match the CPU restatement step for step). FAST takes the cube root directly when pw is exactly 1.0/3.0 — the
// order RK45Solver hard-wires (rk.rs:258-260): cbrt(f) and powf(f, 0.333...) agree to within an ulp
// (f^(1/3 - fl(1/3)) - 1 < 1e-15 for any finite f), about how far two libm implementations of `powf` differ from each
// other, at a quarter of the FP64 instructions.
// powf(f, 1/3) as the reference evaluates it (`f.powf(order.recip())`, ode.rs:120, 133-135): the exponent is the DOUBLE
// nearest to 1/3, p = 1/3 + d with d = -1.85e-17, and Rust's powf is the C library's pow, which rounds correctly except for
// about one argument in a thousand. So STRICT computes the correctly rounded f^p — cheaper than CUDA's general pow (which is
// a 1-2 ulp function and differs from glibc far more often) and the closest one can get to the reference's bits:
//   z ~ f^(-1/3) from the SFU (2^-20) and one third-order step;  y = f z^2 ~ f^(1/3) to 2^-50;
//   one Newton step on y^3 = f with the residual f - y^3 carried in double-double (error 2^-100);
//   f^p = f^(1/3) (1 + d ln f), added to the correction; the final y + c is the only rounding.
// Explicit _rn intrinsics and fma throughout, so nvcc and NVRTC (--fmad=false) builds agree bit for bit.
// Valid for f in [2^-90, 2^90]; the caller falls back to pow() outside.
__device__ __forceinline__ double pow_third_cr(double f) {
    float lg, z0;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(__double2float_rn(f)));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(z0) : "f"(__fmul_rn(lg, -0.33333334f)));
    double z = (double)z0;
    const double r = fma(-f, __dmul_rn(__dmul_rn(z, z), z), 1.0);                  // 1 - f z^3
    z = fma(__dmul_rn(z, r), fma(r, 2.0 / 9.0, 1.0 / 3.0), z);                     // z (1 - r)^(-1/3) to third order
    const double zz = __dmul_rn(z, z);
    const double y = __dmul_rn(f, zz);
    const double y2 = __dmul_rn(y, y), y2l = fma(y, y, -y2);
    const double y3 = __dmul_rn(y2, y), y3l = __dadd_rn(fma(y2, y, -y3), __dmul_rn(y2l, y));
    const double res = __dadd_rn(__dadd_rn(f, -y3), -y3l);                          // f - y^3 (the first difference is exact)
    double c = __dmul_rn(res, __dmul_rn(zz, 1.0 / 3.0));                            // res / (3 y^2)
    c = fma(__dmul_rn(y, -1.850371707708594e-17), __dmul_rn((double)lg, 0.6931471805599453), c);
    return __dadd_rn(y, c);
}

// the general powf, out of line: inlined, its argument classification is hoisted into the hot path of every attempt
static __device__ __noinline__ double pow_cold(double f, double pw) { return pow(f, pw); }

template <bool STRICT> __device__ __forceinline__ double step_size_mul(double alpha, double f, double pw, int pw_is_third) {
    if (pw_is_third) {
        if (!STRICT) return alpha * cbrt(f);
        if (f > 8.0e-28 && f < 1.2e27) return __dmul_rn(alpha, pow_third_cr(f));
    }
    return alpha * pow_cold(f, pw);
}

// handle_step_adaptive (ode.rs:311-334) from the error norm, literally: f = rtol / dx_norm, factor = clamp(alpha f^pw, 0.3, 2),
// new h from the nominal h, reject iff f <= 1.
template <bool STRICT>
__device__ __forceinline__ void controller_ref(double dxn, double h, const CtlShared& cs, double& new_h, bool& reject) {
    const double f = cs.rtol / dxn;
    const double fp_lim = at_most(at_least(step_size_mul<STRICT>(cs.alpha, f, cs.pw, cs.pw_is_third), 0.3), 2.0);
    new_h = at_most(at_least(fp_lim * h, cs.min_dt), cs.max_dt);
    reject = f <= 1.0;
}
// cold path of the FAST kernels (an order other than the 3 that RK45Solver hard-wires): kept out of line
struct CtlRes {
    double new_h;
    int reject;
};
static __device__ __noinline__ CtlRes controller_ref_cold_call(double dxn, double h, double rtol, double alpha, double pw, double min_dt, double max_dt) {
    const double f = rtol / dxn;
    const double fp_lim = at_most(at_least(alpha * pow(f, pw), 0.3), 2.0);
    return CtlRes{at_most(at_least(fp_lim * h, min_dt), max_dt), f <= 1.0 ? 1 : 0};
}
__device__ __forceinline__ void controller_ref_cold(double dxn, double h, const CtlShared& cs, double& new_h, bool& reject) {
    const CtlRes r = controller_ref_cold_call(dxn, h, cs.rtol, cs.alpha, cs.pw, cs.min_dt, cs.max_dt);  // scalars in registers: no stack frame
    new_h = r.new_h, reject = r.reject != 0;
}

// The same controller for the L2 norm in FAST arithmetic, from acc = sum_c e_c^2 without the square root, the division and
// the cube root (which, not the Runge-Kutta stages, were a quarter of the DoPri5 sweep: 150 of 360 instructions per
// attempt). With g = acc / rtol^2 = f^-2:   f^(1/3) = g^(-1/6),   f <= 1  <=>  g >= 1,   dx_norm = acc * f / rtol.
// g^(-1/6) starts from the SFU (lg2/ex2 in f32: within 2^-20 for the g in [0.008, 729] where the factor is not clamped) and
// takes ONE third-order step in f64: with r = 1 - g y^6, g^(-1/6) = y (1 - r)^(-1/6) = y (1 + r/6 + 7 r^2/72 + O(r^3)), and
// the dropped term is 0.07 r^3 < 2^-57 for |r| <= 6 * 2^-20 — below the rounding of the result, so the factor is good to
// ~1 ulp: the accuracy of the reference's own chain sqrt -> div -> powf.
// Out-of-range g (0, inf, NaN, beyond f32) needs no branch: the seed is clamped to [1e-30, 1e30] and the residual to >= -1,
// which leaves the factor far outside [0.3, 2] on the right side; a NaN ends as 0.3 like Rust's NaN.max(0.3).min(2.0); only
// dx_norm takes the slow road.
// U trajectories at once, statement by statement, so that the U dependent chains (seed -> refinement -> clamps) overlap.
template <int U>
__device__ __forceinline__ void controller_l2_fast_n(const double (&acc)[U], const double (&h)[U], const CtlShared& cs, bool want_dxn, double (&dxn)[U],
                                                     double (&new_h)[U], bool (&reject)[U]) {
    double g[U], y[U];
#pragma unroll
    for (int u = 0; u < U; ++u) g[u] = acc[u] * cs.inv_rtol2;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const float gf = fmaxf(fminf(__double2float_rn(g[u]), 1.0e30f), 1.0e-30f);  // a NaN lands on the 1e30 side
        float lg, y0;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(gf));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y0) : "f"(lg * -0.16666667f));
        y[u] = (double)y0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const double y2 = y[u] * y[u];
        const double r = at_least(fma(-g[u], (y2 * y2) * y2, 1.0), -1.0);  // -1 only for g > 1e30, inf or NaN, where the seed is 1e-5
        y[u] = fma(y[u] * r, fma(r, 7.0 / 72.0, 1.0 / 6.0), y[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const double fp_lim = at_most(at_least(cs.alpha * y[u], 0.3), 2.0);
        new_h[u] = at_most(at_least(fp_lim * h[u], cs.min_dt), cs.max_dt);
        reject[u] = g[u] >= 1.0;
    }
    if (want_dxn) {
#pragma unroll
        for (int u = 0; u < U; ++u) dxn[u] = acc[u] * (((y[u] * y[u]) * y[u]) * cs.inv_rtol);
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (!(g[u] > 1.0e-30 && g[u] < 1.0e30)) dxn[u] = sqrt(acc[u]);  // 0, inf, NaN, beyond the seed's range: the slow road
    }
}

// L2-norm controller of the common adaptive configuration, dispatching on the arithmetic mode, for U trajectories of one
// thread. `want_dxn`: the caller keeps ODEAdaptiveData.dx_norm; `nonfinite` reports a NaN norm.
template <bool STRICT, int U>
__device__ __forceinline__ void controller_l2_n(const double (&acc)[U], const double (&h)[U], const CtlShared& cs, bool want_dxn, double (&dxn)[U],
                                                double (&new_h)[U], bool (&reject)[U], bool (&nonfinite)[U]) {
#pragma unroll
    for (int u = 0; u < U; ++u) nonfinite[u] = !(acc[u] == acc[u]);
    if (STRICT) {  // handle_step_adaptive literally (ode.rs:311-334): sqrt and / are IEEE-exact, powf correctly rounded
        double f[U], m[U];
#pragma unroll
        for (int u = 0; u < U; ++u) dxn[u] = sqrt(acc[u]);
#pragma unroll
        for (int u = 0; u < U; ++u) f[u] = cs.rtol / dxn[u];
        bool third = cs.pw_is_third != 0;
#pragma unroll
        for (int u = 0; u < U; ++u) third = third && (f[u] > 8.0e-28 && f[u] < 1.2e27);
        if (third) {
#pragma unroll
            for (int u = 0; u < U; ++u) m[u] = __dmul_rn(cs.alpha, pow_third_cr(f[u]));
        } else {
#pragma unroll
            for (int u = 0; u < U; ++u) m[u] = step_size_mul<true>(cs.alpha, f[u], cs.pw, cs.pw_is_third);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double fp_lim = at_most(at_least(m[u], 0.3), 2.0);
            new_h[u] = at_most(at_least(fp_lim * h[u], cs.min_dt), cs.max_dt);
            reject[u] = f[u] <= 1.0;
        }
    } else if (cs.pw_is_third) {
        controller_l2_fast_n<U>(acc, h, cs, want_dxn, dxn, new_h, reject);
    } else {
#pragma unroll
        for (int u = 0; u < U; ++u) dxn[u] = sqrt(acc[u]), controller_ref_cold(dxn[u], h[u], cs, new_h[u], reject[u]);
    }
}

template <bool STRICT>
__device__ __forceinline__ void controller_l2(double acc, double h, const CtlShared& cs, bool want_dxn, double& dxn, double& new_h, bool& reject,
                                              bool& nonfinite) {
    const double a[1] = {acc}, hh[1] = {h};
    double d[1] = {dxn}, nh[1];
    bool rj[1], nf[1];
    controller_l2_n<STRICT, 1>(a, hh, cs, want_dxn, d, nh, rj, nf);
    dxn = d[0], new_h = nh[0], reject = rj[0], nonfinite = nf[0];
}

// ---- staged (TMA bulk-copy) variants ---------------------------------------------------------------------------
// Same arithmetic as the two kernels above; the difference is how state reaches the registers. One CTA = 128 lanes =
// one tile of 128 consecutive trajectories; thread 0 keeps VO_STAGES tiles (every SoA row the kernel reads: the d state
// components, per-trajectory RHS parameters, and for the control kernel t, h and the status word) in flight through
// cp.async.bulk + mbarrier; lanes read their element from shared memory, integrate, and store straight to global.
// Needs N even (row starts 16-byte aligned); the host falls back to the register-prefetch kernels otherwise.
#define VO_STAGES 4
#define VO_TILE 128

template <class RHS, int S, bool STRICT>
__global__ void __launch_bounds__(VO_TILE) rk_fixed_staged_kernel(double* __restrict__ x, int64_t N, const __grid_constant__ TableauDev tb,
                                                                  const __grid_constant__ RhsParams rp, const __grid_constant__ StepList sl,
                                                                  const pipe::Chain ch) {
    constexpr int D = RHS::D, NP = RHS::NP, T = VO_TILE;
    extern __shared__ __align__(128) double sbuf[];  // [VO_STAGES][nrows][T]
    __shared__ __align__(8) uint64_t full[VO_STAGES];
    int nrows = D;
#pragma unroll
    for (int q = 0; q < NP; ++q) nrows += rp.per_traj[q] ? 1 : 0;
    const int64_t n_full = N / T, G = gridDim.x, first = blockIdx.x;
    const int64_t my_count = first < n_full ? (n_full - first + G - 1) / G : 0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < VO_STAGES; ++s) pipe::mbar_init(&full[s], 1);
        pipe::fence_mbar_init();
    }
    pipe::chain_enter(ch);
    auto issue = [&](int64_t k) {  // thread 0: all rows of this CTA's k-th tile into stage k % VO_STAGES
        const int st = (int)(k % VO_STAGES);
        const int64_t base = (first + k * G) * T;
        double* dst = sbuf + (size_t)st * nrows * T;
        pipe::mbar_expect_tx(&full[st], (uint32_t)(nrows * T * sizeof(double)));
        int r = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) pipe::bulk_g2s(dst + (r++) * T, x + c * N + base, T * sizeof(double), &full[st]);
#pragma unroll
        for (int q = 0; q < NP; ++q)
            if (rp.per_traj[q]) pipe::bulk_g2s(dst + (r++) * T, rp.per_traj[q] + base, T * sizeof(double), &full[st]);
    };
    if (threadIdx.x == 0)
        for (int64_t k = 0; k < my_count && k < VO_STAGES; ++k) issue(k);
    for (int64_t k = 0; k < my_count; ++k) {
        const int st = (int)(k % VO_STAGES);
        const int64_t i = (first + k * G) * T + threadIdx.x;
        pipe::mbar_wait(&full[st], (uint32_t)((k / VO_STAGES) & 1));
        const double* src = sbuf + (size_t)st * nrows * T + threadIdx.x;
        double xc[D], p[NP];
        int r = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) xc[c] = src[(r++) * T];
#pragma unroll
        for (int q = 0; q < NP; ++q) p[q] = rp.per_traj[q] ? src[(r++) * T] : rp.shared[q];
        __syncthreads();  // every lane has taken its element: the stage may be refilled
        if (threadIdx.x == 0 && k + VO_STAGES < my_count) issue(k + VO_STAGES);
        for (int e = 0; e < sl.n; ++e) {
            double xf[D], xe[D];
            rk_attempt<RHS, S, STRICT>(tb, sl.use_err != 0, sl.t[e], sl.dt[e], xc, p, xf, xe);
#pragma unroll
            for (int c = 0; c < D; ++c) xc[c] = xf[c];
        }
#pragma unroll
        for (int c = 0; c < D; ++c) x[c * N + i] = xc[c];
    }
    // ragged tail (N % 128 trajectories): plain loads, last CTA
    const int64_t i = n_full * T + threadIdx.x;
    if (blockIdx.x == G - 1 && i < N) {
        double xc[D], p[NP];
        lane_load<RHS>(x, N, rp, i, xc, p);
        for (int e = 0; e < sl.n; ++e) {
            double xf[D], xe[D];
            rk_attempt<RHS, S, STRICT>(tb, sl.use_err != 0, sl.t[e], sl.dt[e], xc, p, xf, xe);
#pragma unroll
            for (int c = 0; c < D; ++c) xc[c] = xf[c];
        }
#pragma unroll
        for (int c = 0; c < D; ++c) x[c * N + i] = xc[c];
    }
    pipe::chain_exit(ch);
}

// Where one trajectory's state and controller scalars live in global memory: element i of the SoA ensemble and of every CtlArrays array.
struct SoaAcc {
    double* x;
    int64_t N;
    CtlArrays ca;
    int64_t i;
    __device__ __forceinline__ int64_t gidx() const { return i; }  // trajectory number (snapshots are indexed by it)
    __device__ __forceinline__ int64_t count() const { return N; }
    __device__ __forceinline__ void st_x(int c, double v) const { x[c * N + i] = v; }
    __device__ __forceinline__ void st_t(double v) const { ca.t[i] = v; }
    __device__ __forceinline__ void st_h(double v) const { ca.h[i] = v; }
    __device__ __forceinline__ double ld_prev_h() const { return ca.prev_h[i]; }
    __device__ __forceinline__ void st_prev_h(double v) const { ca.prev_h[i] = v; }
    __device__ __forceinline__ void st_dxn(double v) const { ca.dx_norm[i] = v; }
    __device__ __forceinline__ void st_acc(uint32_t v) const { ca.n_accept[i] = v; }
    __device__ __forceinline__ void st_rej(uint32_t v) const { ca.n_reject[i] = v; }
    __device__ __forceinline__ void st_word(uint32_t v) const { ca.word[i] = v; }
};

// One lane of the per-trajectory control kernel: k_events calls of step()/step_adaptive() on registers, then the
// masked write-back. Shared by the staged kernel body and its ragged tail.
// CFG 1 = the common adaptive configuration (step_adaptive with an error estimate and the L2 norm) resolved at compile
// time; CFG 0 = everything decided from CtlShared at run time.
template <class RHS, int S, bool STRICT, int CFG>
__device__ __forceinline__ void ctl_lane(const SoaAcc& a, const TableauDev& tb, const CtlShared& cs,
                                         const TList& tl, uint32_t word, double (&xc)[RHS::D], const double (&p)[RHS::NP], double t, double h,
                                         uint32_t n_acc, uint32_t n_rej, unsigned& c_step, unsigned& c_chkpt, unsigned& c_rej, unsigned& c_end, unsigned& c_stuck) {
    constexpr int D = RHS::D;
    double prev_h = 0.0;
    bool prev_h_loaded = false, ctl_dirty = false, moved = false;
    int tgt = (int)(word & VO_WORD_TGT_MASK);
    uint32_t status = word >> VO_WORD_STATUS_SHIFT;
    double dxn = 0.0;
    bool dxn_set = false;
    unsigned l_step = 0, l_rej = 0;
    for (int e = 0; e < cs.k_events; ++e) {
        int evk;  // step_size_of (ode.rs:165-176) + check_step (ode.rs:389-399)
        double dt = 0.0;
        if (tgt >= cs.n_tlist) {
            evk = VO_EV_END;
        } else {
            const double rem = tl.at(tgt) - t;
            if (fabs(rem) <= 2.220446049250313e-16) evk = (tgt >= cs.n_tlist - 1) ? VO_EV_END : VO_EV_CHKPT;
            else dt = rem < h ? rem : h, evk = VO_EV_STEP;
        }
        if (evk == VO_EV_STEP) {
            double xf[D], xe[D];
            rk_attempt<RHS, S, STRICT>(tb, CFG == 1 ? true : cs.use_err != 0, t, dt, xc, p, xf, xe);
            if (CFG == 1 || cs.adaptive) {  // handle_step_adaptive, ode.rs:311-334
                double new_h;
                bool rejected, nonfinite;
                if (CFG == 1) {
                    controller_l2<STRICT>(err_sumsq<STRICT, D>(xe), h, cs, cs.record_dx_norm != 0, dxn, new_h, rejected, nonfinite);
                } else {
                    dxn = err_norm<STRICT, D>(xe, cs.norm_kind), nonfinite = !(dxn == dxn);
                    if (STRICT) controller_ref<true>(dxn, h, cs, new_h, rejected);
                    else controller_ref_cold(dxn, h, cs, new_h, rejected);
                }
                dxn_set = true;
                if (nonfinite) status |= VO_TRAJ_NONFINITE;
                if (rejected) {
                    evk = VO_EV_REJECT;
                    if (h <= cs.min_dt) status |= VO_TRAJ_STUCK, ++c_stuck;
                }
                prev_h = h, h = new_h, prev_h_loaded = true, ctl_dirty = true;  // update_step_size, ode.rs:202-205
            }
            if (evk == VO_EV_STEP) {  // accept_step -> advance, ode.rs:184-188
#pragma unroll
                for (int c = 0; c < D; ++c) xc[c] = xf[c];
                t += dt;
                moved = true, ++l_step;
            } else {
                ++l_rej;
            }
        } else {  // Chkpt / End -> checkpoint_update, ode.rs:192-195
            if (cs.snap && tgt < cs.n_tlist) {  // what current() shows the caller at this event
#pragma unroll
                for (int c = 0; c < D; ++c) cs.snap[tgt * cs.snap_stride + (int64_t)c * a.count() + a.gidx()] = xc[c];
            }
            if (!prev_h_loaded) prev_h = a.ld_prev_h(), prev_h_loaded = true;
            tgt += 1, h = prev_h, ctl_dirty = true;
            if (evk == VO_EV_END) {
                status |= VO_TRAJ_DONE, ++c_end;
                break;
            }
            ++c_chkpt;
        }
    }
    if (moved) {
#pragma unroll
        for (int c = 0; c < D; ++c) a.st_x(c, xc[c]);
        a.st_t(t);
    }
    if (ctl_dirty) {
        a.st_h(h);
        a.st_prev_h(prev_h);
    }
    if (dxn_set && cs.record_dx_norm) a.st_dxn(dxn);
    if (l_step) a.st_acc(n_acc + l_step);  // counters came in with the tile: no read-modify-write round trip here
    if (l_rej) a.st_rej(n_rej + l_rej);
    const uint32_t nw = ((uint32_t)tgt & VO_WORD_TGT_MASK) | (status << VO_WORD_STATUS_SHIFT);
    if (nw != word) a.st_word(nw);
    c_step += l_step, c_rej += l_rej;
}

__device__ __forceinline__ void ctl_count_events(const CtlShared& cs, EvSlot* __restrict__ ev, unsigned c_step, unsigned c_chkpt, unsigned c_rej,
                                                 unsigned c_end, unsigned c_stuck) {
    if (!cs.count_events) return;
    // block-level reduction, then at most five atomics per block, spread over VO_EV_SLOTS lines
    __shared__ unsigned sm[5];
    if (threadIdx.x < 5) sm[threadIdx.x] = 0;
    __syncthreads();
    c_step = __reduce_add_sync(0xffffffffu, c_step), c_chkpt = __reduce_add_sync(0xffffffffu, c_chkpt);
    c_rej = __reduce_add_sync(0xffffffffu, c_rej), c_end = __reduce_add_sync(0xffffffffu, c_end);
    c_stuck = __reduce_add_sync(0xffffffffu, c_stuck);
    if ((threadIdx.x & 31) == 0) {
        if (c_step) atomicAdd(&sm[0], c_step);
        if (c_chkpt) atomicAdd(&sm[1], c_chkpt);
        if (c_rej) atomicAdd(&sm[2], c_rej);
        if (c_end) atomicAdd(&sm[3], c_end);
        if (c_stuck) atomicAdd(&sm[4], c_stuck);
    }
    __syncthreads();
    if (threadIdx.x < 5 && sm[threadIdx.x]) {
        EvSlot* slot = ev + (blockIdx.x % VO_EV_SLOTS);
        unsigned long long* dst = threadIdx.x == 0   ? &slot->n_step
                                  : threadIdx.x == 1 ? &slot->n_chkpt
                                  : threadIdx.x == 2 ? &slot->n_reject
                                  : threadIdx.x == 3 ? &slot->n_end
                                                     : &slot->n_stuck;
        atomicAdd(dst, (unsigned long long)sm[threadIdx.x]);
    }
}

#ifndef VO_CTL_MIN_BLOCKS
#define VO_CTL_MIN_BLOCKS 6
#endif
template <class RHS, int S, bool STRICT, int CFG>
__global__ void __launch_bounds__(VO_TILE, VO_CTL_MIN_BLOCKS) rk_ctl_staged_kernel(double* __restrict__ x, int64_t N, const __grid_constant__ TableauDev tb,
                                                                const __grid_constant__ RhsParams rp, const CtlArrays ca,
                                                                const __grid_constant__ CtlShared cs, EvSlot* __restrict__ ev, const pipe::Chain ch) {
    constexpr int D = RHS::D, NP = RHS::NP, T = VO_TILE;
    extern __shared__ __align__(128) double sbuf[];  // [VO_STAGES][nrows][T] doubles, then [VO_STAGES][3][T] words
    __shared__ __align__(8) uint64_t full[VO_STAGES];
    int nrows = D + 2;  // state, t, h
#pragma unroll
    for (int q = 0; q < NP; ++q) nrows += rp.per_traj[q] ? 1 : 0;
    uint32_t* wbuf = reinterpret_cast<uint32_t*>(sbuf + (size_t)VO_STAGES * nrows * T);
    const int64_t n_full = N / T, G = gridDim.x, first = blockIdx.x;
    const int64_t my_count = first < n_full ? (n_full - first + G - 1) / G : 0;
    __shared__ double s_tl[VO_INLINE_TLIST];
    const TList tl = tlist_stage(cs, s_tl);
    unsigned c_step = 0, c_chkpt = 0, c_rej = 0, c_end = 0, c_stuck = 0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < VO_STAGES; ++s) pipe::mbar_init(&full[s], 1);
        pipe::fence_mbar_init();
    }
    pipe::chain_enter(ch);
    auto issue = [&](int64_t k) {
        const int st = (int)(k % VO_STAGES);
        const int64_t base = (first + k * G) * T;
        double* dst = sbuf + (size_t)st * nrows * T;
        pipe::mbar_expect_tx(&full[st], (uint32_t)(nrows * T * sizeof(double) + 3 * T * sizeof(uint32_t)));
        int r = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) pipe::bulk_g2s(dst + (r++) * T, x + c * N + base, T * sizeof(double), &full[st]);
        pipe::bulk_g2s(dst + (r++) * T, ca.t + base, T * sizeof(double), &full[st]);
        pipe::bulk_g2s(dst + (r++) * T, ca.h + base, T * sizeof(double), &full[st]);
#pragma unroll
        for (int q = 0; q < NP; ++q)
            if (rp.per_traj[q]) pipe::bulk_g2s(dst + (r++) * T, rp.per_traj[q] + base, T * sizeof(double), &full[st]);
        uint32_t* wdst = wbuf + (size_t)st * 3 * T;  // status word, accepted, rejected
        pipe::bulk_g2s(wdst, ca.word + base, T * sizeof(uint32_t), &full[st]);
        pipe::bulk_g2s(wdst + T, ca.n_accept + base, T * sizeof(uint32_t), &full[st]);
        pipe::bulk_g2s(wdst + 2 * T, ca.n_reject + base, T * sizeof(uint32_t), &full[st]);
    };
    if (threadIdx.x == 0)
        for (int64_t k = 0; k < my_count && k < VO_STAGES; ++k) issue(k);
    for (int64_t k = 0; k < my_count; ++k) {
        const int st = (int)(k % VO_STAGES);
        const int64_t i = (first + k * G) * T + threadIdx.x;
        pipe::mbar_wait(&full[st], (uint32_t)((k / VO_STAGES) & 1));
        const double* src = sbuf + (size_t)st * nrows * T + threadIdx.x;
        double xc[D], p[NP];
        int r = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) xc[c] = src[(r++) * T];
        const double t = src[(r++) * T], h = src[(r++) * T];
#pragma unroll
        for (int q = 0; q < NP; ++q) p[q] = rp.per_traj[q] ? src[(r++) * T] : rp.shared[q];
        const uint32_t* wsrc = wbuf + (size_t)st * 3 * T + threadIdx.x;
        const uint32_t word = wsrc[0], n_acc = wsrc[T], n_rej = wsrc[2 * T];
        __syncthreads();
        if (threadIdx.x == 0 && k + VO_STAGES < my_count) issue(k + VO_STAGES);
        if (!((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE))
            ctl_lane<RHS, S, STRICT, CFG>(SoaAcc{x, N, ca, i}, tb, cs, tl, word, xc, p, t, h, n_acc, n_rej, c_step, c_chkpt, c_rej, c_end, c_stuck);
    }
    const int64_t i = n_full * T + threadIdx.x;  // ragged tail: plain loads, last CTA
    if (blockIdx.x == G - 1 && i < N) {
        const uint32_t word = ca.word[i];
        if (!((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE)) {
            double xc[D], p[NP];
            lane_load<RHS>(x, N, rp, i, xc, p);
            ctl_lane<RHS, S, STRICT, 0>(SoaAcc{x, N, ca, i}, tb, cs, tl, word, xc, p, ca.t[i], ca.h[i], ca.n_accept[i], ca.n_reject[i], c_step, c_chkpt, c_rej,
                                        c_end, c_stuck);
        }
    }
    ctl_count_events(cs, ev, c_step, c_chkpt, c_rej, c_end, c_stuck);
    pipe::chain_exit(ch);
}

// Register-prefetch fallback of the control kernel (odd N: SoA rows are not 16-byte aligned for bulk copies).
template <class RHS, int S, bool STRICT>
__global__ void __launch_bounds__(128) rk_ctl_kernel(double* __restrict__ x, int64_t N, const __grid_constant__ TableauDev tb,
                                                     const __grid_constant__ RhsParams rp, const CtlArrays ca, const __grid_constant__ CtlShared cs,
                                                     EvSlot* __restrict__ ev) {
    constexpr int D = RHS::D;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned c_step = 0, c_chkpt = 0, c_rej = 0, c_end = 0, c_stuck = 0;
    __shared__ double s_tl[VO_INLINE_TLIST];
    const TList tl = tlist_stage(cs, s_tl);
    __syncthreads();
    uint32_t word = 0, word_n = 0, na = 0, nr = 0, na_n = 0, nr_n = 0;
    double xc[D], p[RHS::NP], t = 0.0, h = 0.0, xn[D], pn[RHS::NP], t_n = 0.0, h_n = 0.0;
    bool live = false, live_n = false;
    if (i < N) {
        word = ca.word[i];
        live = !((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE);
        if (live) lane_load<RHS>(x, N, rp, i, xc, p), t = ca.t[i], h = ca.h[i], na = ca.n_accept[i], nr = ca.n_reject[i];
    }
    while (i < N) {
        const int64_t j = i + stride;
        if (j < N) {  // prefetch the next trajectory of this thread
            word_n = ca.word[j];
            live_n = !((word_n >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE);
            if (live_n) lane_load<RHS>(x, N, rp, j, xn, pn), t_n = ca.t[j], h_n = ca.h[j], na_n = ca.n_accept[j], nr_n = ca.n_reject[j];
        }
        if (live) ctl_lane<RHS, S, STRICT, 0>(SoaAcc{x, N, ca, i}, tb, cs, tl, word, xc, p, t, h, na, nr, c_step, c_chkpt, c_rej, c_end, c_stuck);
        word = word_n, live = (j < N) && live_n, t = t_n, h = h_n, na = na_n, nr = nr_n;
#pragma unroll
        for (int c = 0; c < D; ++c) xc[c] = xn[c];
#pragma unroll
        for (int q = 0; q < RHS::NP; ++q) p[q] = pn[q];
        i = j;
    }
    ctl_count_events(cs, ev, c_step, c_chkpt, c_rej, c_end, c_stuck);
}
