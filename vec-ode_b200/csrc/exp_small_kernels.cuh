// exp_small_kernels.cuh — the exponential integrators for systems of 1 <= n <= 8 levels (qubits, qutrits, few-qubit registers).
// Device code only, like exp_kernels.cuh, so that a user generator or norm (nvrtc_rhs.cu) is compiled at run time into it.
//
// At this size an m8n8k4 tile is mostly padding and a whole state is at most 8 complex numbers, so one thread owns one system:
// state, running sum and Taylor term stay in registers, the basis is a __grid_constant__ kernel parameter (uniform operand of
// the FP64 FMAs, read from the constant bank) and every system runs its own Taylor plan, the plan of the CPU restatements.
// The per-system control logic (step_size_of, the exponents of every scheme, the controller) is exp_kernels.cuh's, shared
// with exp_step_kernel. A launch runs up to kp.n_events events per system with the control values held in registers.
#pragma once
#include "exp_kernels.cuh"

#define VO_EXP_SMALL_THREADS 128

template <int N, int M> struct SmallBasis {
    double2 b[M][N][N];  // B_m[row][col], complex interleaved: the layout of vo_split_basis_create's input
};

// Up to n = 4 exp(sum_m c_m B_m) applies the assembled n x n operator per Taylor term (n^2 complex products instead of M n^2);
// above, its 2 n^2 doubles would not fit next to the vectors, and the term applies the M basis matrices from the constant bank.
template <int N, int M> struct SmallOp {
    static constexpr bool ASSEMBLE = N <= 4 && M > 1;
};

// A system's control values in registers for the events of one launch (the CTL of exp_event_finish).
struct CtlRegs {
    double t_, h_, prev_h_, dx_norm_;
    uint32_t n_accept_, n_reject_, word_;
    __device__ __forceinline__ double& t() { return t_; }
    __device__ __forceinline__ double& h() { return h_; }
    __device__ __forceinline__ double& prev_h() { return prev_h_; }
    __device__ __forceinline__ double& dx_norm() { return dx_norm_; }
    __device__ __forceinline__ uint32_t& n_accept() { return n_accept_; }
    __device__ __forceinline__ uint32_t& n_reject() { return n_reject_; }
    __device__ __forceinline__ uint32_t& word() { return word_; }
};

// y = sum_m c_m (B_m x), c complex; with ACC, y += that
template <int N, int M, bool ACC = false>
__device__ __forceinline__ void small_basis_apply(const SmallBasis<N, M>& B, const double (&cr)[M], const double (&ci)[M], const double (&xr)[N],
                                                  const double (&xi)[N], double (&yr)[N], double (&yi)[N]) {
#pragma unroll
    for (int r = 0; r < N; ++r)
        if (!ACC) yr[r] = yi[r] = 0.0;
    // From n = 4 up the basis matrices go one at a time, in a loop the compiler keeps (its trip count and the basis address carry a 0
    // it cannot see through, even for M = 1): unrolled, it hoists the 2 M n^2 basis values of several products into registers.
    int z = 0;
    if (N > 3) asm volatile("mov.b32 %0, 0;" : "=r"(z));
    const double2* bb = &B.b[0][0][0] + z;
#pragma unroll (N <= 3 ? M : 1)
    for (int m = 0; m < M + z; ++m) {
        double c_r = cr[0], c_i = ci[0];
#pragma unroll
        for (int j = 1; j < M; ++j)
            if (j == m) c_r = cr[j], c_i = ci[j];
#pragma unroll
        for (int r = 0; r < N; ++r) {
            double ar = 0.0, ai = 0.0;
#pragma unroll
            for (int k = 0; k < N; ++k) {
                const double2 b = bb[(m * N + r) * N + k];
                ar = fma(b.x, xr[k], fma(-b.y, xi[k], ar));
                ai = fma(b.x, xi[k], fma(b.y, xr[k], ai));
            }
            yr[r] = fma(c_r, ar, fma(-c_i, ai, yr[r]));
            yi[r] = fma(c_r, ai, fma(c_i, ar, yi[r]));
        }
    }
}

// L = sum_m c_m B_m, c complex
template <int N, int M>
__device__ __forceinline__ void small_assemble(const SmallBasis<N, M>& B, const double (&cr)[M], const double (&ci)[M], double (&Lr)[N][N], double (&Li)[N][N]) {
#pragma unroll
    for (int r = 0; r < N; ++r)
#pragma unroll
        for (int k = 0; k < N; ++k) {
            double sr = 0.0, si = 0.0;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const double2 b = B.b[m][r][k];
                sr = fma(cr[m], b.x, fma(-ci[m], b.y, sr));
                si = fma(cr[m], b.y, fma(ci[m], b.x, si));
            }
            Lr[r][k] = sr, Li[r][k] = si;
        }
}

// y = L x
template <int N>
__device__ __forceinline__ void small_matvec(const double (&Lr)[N][N], const double (&Li)[N][N], const double (&xr)[N], const double (&xi)[N], double (&yr)[N], double (&yi)[N]) {
#pragma unroll
    for (int r = 0; r < N; ++r) {
        double ar = 0.0, ai = 0.0;
#pragma unroll
        for (int k = 0; k < N; ++k) {
            ar = fma(Lr[r][k], xr[k], fma(-Li[r][k], xi[k], ar));
            ai = fma(Lr[r][k], xi[k], fma(Li[r][k], xr[k], ai));
        }
        yr[r] = ar, yi[r] = ai;
    }
}

// 1 / k for the Taylor terms k = 1 .. 60 (taylor_plan's cap), each correctly rounded as the division is: a table read in place of
// a division, whose slow path is a call that makes the compiler save live registers to local memory around it
__constant__ double vo_small_recip[60] = {1.0 / 1, 1.0 / 2, 1.0 / 3, 1.0 / 4, 1.0 / 5, 1.0 / 6, 1.0 / 7, 1.0 / 8, 1.0 / 9, 1.0 / 10, 1.0 / 11, 1.0 / 12, 1.0 / 13, 1.0 / 14, 1.0 / 15, 1.0 / 16, 1.0 / 17, 1.0 / 18, 1.0 / 19, 1.0 / 20, 1.0 / 21, 1.0 / 22, 1.0 / 23, 1.0 / 24, 1.0 / 25, 1.0 / 26, 1.0 / 27, 1.0 / 28, 1.0 / 29, 1.0 / 30, 1.0 / 31, 1.0 / 32, 1.0 / 33, 1.0 / 34, 1.0 / 35, 1.0 / 36, 1.0 / 37, 1.0 / 38, 1.0 / 39, 1.0 / 40, 1.0 / 41, 1.0 / 42, 1.0 / 43, 1.0 / 44, 1.0 / 45, 1.0 / 46, 1.0 / 47, 1.0 / 48, 1.0 / 49, 1.0 / 50, 1.0 / 51, 1.0 / 52, 1.0 / 53, 1.0 / 54, 1.0 / 55, 1.0 / 56, 1.0 / 57, 1.0 / 58, 1.0 / 59, 1.0 / 60};

// x <- sum over sq sub-steps of the degree-deg Taylor series, op(T, W): W = (Omega / sq) T
template <int N, class OP>
__device__ __forceinline__ void small_taylor(int sq, int deg, double (&xr)[N], double (&xi)[N], OP op) {
#pragma unroll 1
    for (int rep = 0; rep < sq; ++rep) {
        double ar[N], ai[N], tr[N], ti[N];
#pragma unroll
        for (int r = 0; r < N; ++r) ar[r] = tr[r] = xr[r], ai[r] = ti[r] = xi[r];
#pragma unroll 1  // one term at a time: two in flight would double the live vectors
        for (int k = 1; k <= deg; ++k) {
            double wr[N], wi[N];
            op(tr, ti, wr, wi);
            const double ik = vo_small_recip[k - 1];
#pragma unroll
            for (int r = 0; r < N; ++r) tr[r] = wr[r] * ik, ti[r] = wi[r] * ik, ar[r] += tr[r], ai[r] += ti[r];
        }
#pragma unroll
        for (int r = 0; r < N; ++r) xr[r] = ar[r], xi[r] = ai[r];
    }
}

// x <- exp(sum_m c_m B_m) x with this system's own Taylor plan
template <int N, int M>
__device__ __forceinline__ void small_map_exp(const ExpKP& kp, const SmallBasis<N, M>& B, const double2 (&c)[M], double (&xr)[N], double (&xi)[N]) {
    int sq, deg;
    taylor_plan(exp_theta<M>(kp, [&](int m) { return c[m]; }), kp.taylor_deg, &sq, &deg);
    const double inv_sq = 1.0 / sq;
    double cr[M], ci[M];
#pragma unroll
    for (int m = 0; m < M; ++m) cr[m] = c[m].x * inv_sq, ci[m] = c[m].y * inv_sq;
    if (SmallOp<N, M>::ASSEMBLE) {
        double Lr[N][N], Li[N][N];
        small_assemble<N, M>(B, cr, ci, Lr, Li);
        small_taylor<N>(sq, deg, xr, xi, [&](const double (&tr)[N], const double (&ti)[N], double (&wr)[N], double (&wi)[N]) { small_matvec<N>(Lr, Li, tr, ti, wr, wi); });
    } else {
        small_taylor<N>(sq, deg, xr, xi, [&](const double (&tr)[N], const double (&ti)[N], double (&wr)[N], double (&wi)[N]) { small_basis_apply<N, M>(B, cr, ci, tr, ti, wr, wi); });
    }
}

// out[k] = <x| O_k |x> = sum_r conj(x_r) sum_c O_k[r][c] x_c for the n_obs operators obs [n_obs][N][N], from this thread's copy of the
// state in shared memory (row r at xs[r * VO_EXP_SMALL_THREADS]). Every thread reads the operators at the same address, so each
// load is a broadcast. Called at Chkpt / End events only, and not inlined: its code and registers stay out of the kernel's step
// loop (DESIGN.md §2.3). Plain pointers rather than the launch parameters, which a call could only take by a local copy.
template <int N>
__device__ __noinline__ void small_expect(const double2* __restrict__ obs, int n_obs, const double2* xs, double2* out) {
#pragma unroll 1
    for (int k = 0; k < n_obs; ++k) {
        double er = 0.0, ei = 0.0;
#pragma unroll (N <= 4 ? N : 1)
        for (int r = 0; r < N; ++r) {
            const double2* O = obs + (k * N + r) * N;
            double ar = 0.0, ai = 0.0;
#pragma unroll
            for (int c = 0; c < N; ++c) {
                const double2 o = O[c], x = xs[c * VO_EXP_SMALL_THREADS];
                ar = fma(o.x, x.x, fma(-o.y, x.y, ar));
                ai = fma(o.x, x.y, fma(o.y, x.x, ai));
            }
            const double2 v = xs[r * VO_EXP_SMALL_THREADS];
            er = fma(v.x, ar, fma(v.y, ai, er));
            ei = fma(v.x, ai, fma(-v.y, ar, ei));
        }
        out[k] = make_double2(er, ei);
    }
}

// x <- exp(Omega) x for magnus_42 with the applied commutator, Omega = W1 + b2 [L0, L1] (w1, l0, l1: real coefficients). Up to n = 3
// Omega is assembled once per exponential from the three operators (6 n^2 doubles at once); above, a Taylor term is
// W1 T + b2 (L0 (L1 T) - L1 (L0 T)) by products, as exp_step_kernel's map_exp_tile_comm does.
template <int N, int M>
__device__ __forceinline__ void small_map_exp_comm(const ExpKP& kp, const SmallBasis<N, M>& B, const double (&w1)[M], const double (&l0)[M], const double (&l1)[M],
                                                   double dt, double (&xr)[N], double (&xi)[N]) {
    double th = exp_theta<M>(kp, [&](int m) { return make_double2(w1[m], 0.0); });
    th += exp_comm_theta<M>(kp, dt, [&](int m) { return l0[m]; }, [&](int m) { return l1[m]; });
    int sq, deg;
    taylor_plan(th, kp.taylor_deg, &sq, &deg);
    const double inv_sq = 1.0 / sq;
    const double b2 = dt * dt * -0.144337567297406441127287195125 * inv_sq;  // magnus.rs:41, per sub-step
    double wr_[M], l0r[M], l1r[M], l0b[M], l1b[M], zero[M];
#pragma unroll
    for (int m = 0; m < M; ++m) wr_[m] = w1[m] * inv_sq, l0r[m] = l0[m], l1r[m] = l1[m], l0b[m] = b2 * l0[m], l1b[m] = -b2 * l1[m], zero[m] = 0.0;
    if (N <= 3) {
        double Or[N][N], Oi[N][N], Ar[N][N], Ai[N][N], Cr[N][N], Ci[N][N];
        small_assemble<N, M>(B, l0r, zero, Ar, Ai);
        small_assemble<N, M>(B, l1r, zero, Cr, Ci);
        small_assemble<N, M>(B, wr_, zero, Or, Oi);
#pragma unroll
        for (int r = 0; r < N; ++r)
#pragma unroll
            for (int k = 0; k < N; ++k) {  // + b2 (L0 L1 - L1 L0)[r][k]
                double sr = 0.0, si = 0.0;
#pragma unroll
                for (int j = 0; j < N; ++j) {
                    sr += Ar[r][j] * Cr[j][k] - Ai[r][j] * Ci[j][k] - (Cr[r][j] * Ar[j][k] - Ci[r][j] * Ai[j][k]);
                    si += Ar[r][j] * Ci[j][k] + Ai[r][j] * Cr[j][k] - (Cr[r][j] * Ai[j][k] + Ci[r][j] * Ar[j][k]);
                }
                Or[r][k] += b2 * sr, Oi[r][k] += b2 * si;
            }
        small_taylor<N>(sq, deg, xr, xi, [&](const double (&tr)[N], const double (&ti)[N], double (&yr)[N], double (&yi)[N]) { small_matvec<N>(Or, Oi, tr, ti, yr, yi); });
    } else {
        small_taylor<N>(sq, deg, xr, xi, [&](const double (&tr)[N], const double (&ti)[N], double (&yr)[N], double (&yi)[N]) {
            double ar[N], ai[N];
            small_basis_apply<N, M>(B, wr_, zero, tr, ti, yr, yi);        // W1 T / sq
            small_basis_apply<N, M>(B, l1r, zero, tr, ti, ar, ai);        // L1 T
            small_basis_apply<N, M, true>(B, l0b, zero, ar, ai, yr, yi);  // + b2 L0 L1 T
            small_basis_apply<N, M>(B, l0r, zero, tr, ti, ar, ai);        // L0 T
            small_basis_apply<N, M, true>(B, l1b, zero, ar, ai, yr, yi);  // - b2 L1 L0 T
        });
    }
}

template <int N, int M, class GEN>
__global__ void __launch_bounds__(VO_EXP_SMALL_THREADS, 1)
exp_small_kernel(const __grid_constant__ ExpKP kp, const __grid_constant__ SmallBasis<N, M> B, double2* __restrict__ psi, double2* __restrict__ psi_out,
                 const double* __restrict__ gp, const double2* __restrict__ coef_in, const CtlArrays ca, EvSlot* __restrict__ ev) {
    constexpr int PG = 3 * (VO_EXP_MAX_M - 1);
    // x0, the state a step starts from, waits here while its exponentials run on the registers in place: the embedded solution
    // starts from it and a rejected step returns to it (in registers it would cost 2 n of them through the whole step)
    __shared__ double2 sx0[N * VO_EXP_SMALL_THREADS];
    int nbase, nerr;
    exp_counts_of(kp, &nbase, &nerr);
    ExpCounts cnt;
    for (int64_t sys = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; sys < kp.N; sys += (int64_t)gridDim.x * blockDim.x) {
        double xr[N], xi[N];
#pragma unroll
        for (int r = 0; r < N; ++r) {
            const double2 v = psi[sys * N + r];
            xr[r] = v.x, xi[r] = v.y;
        }
        if (kp.mode == 1) {  // vo_map_exp / vo_map_exp_seq: nseq exponentials, one after the other
            for (int q = 0; q < kp.nseq; ++q) {
                double2 c[M];
#pragma unroll
                for (int m = 0; m < M; ++m) c[m] = coef_in[((int64_t)q * kp.N + sys) * M + m];
                small_map_exp<N, M>(kp, B, c, xr, xi);
            }
#pragma unroll
            for (int r = 0; r < N; ++r) psi_out[sys * N + r] = make_double2(xr[r], xi[r]);
            continue;
        }
        CtlRegs c{ca.t[sys], ca.h[sys], ca.prev_h[sys], ca.dx_norm[sys], ca.n_accept[sys], ca.n_reject[sys], ca.word[sys]};
        if ((c.word_ >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE) continue;
        double g[PG];
#pragma unroll
        for (int q = 0; q < PG; ++q) g[q] = q < 3 * (kp.M_gen - 1) ? gp[sys * (kp.M_gen - 1) * 3 + q] : 0.0;
        bool moved = false;
        for (int evn = 0; evn < kp.n_events; ++evn) {
            const uint32_t word = c.word_;
            const double t = c.t_, h = c.h_;
            double dt = 0.0;
            const int evk = exp_event_kind(kp, word, t, h, dt);
            if (evk == 255) break;
            double err = 0.0;  // ||x_err||: read by the adaptive controller alone, which always has an embedded solution
            if (evk == VO_EV_STEP) {
#pragma unroll
                for (int r = 0; r < N; ++r) sx0[r * VO_EXP_SMALL_THREADS + threadIdx.x] = make_double2(xr[r], xi[r]);
                double v[VO_EXP_MAX_NODES][M];
                exp_samples<M, GEN>(kp, g, t, dt, v);
                if (kp.applied_comm) {
                    double w1[M], l0[M], l1[M];
                    exp_row<M>(kp, 0, nbase, v, dt, w1), exp_row<M>(kp, 2, nbase, v, dt, l0), exp_row<M>(kp, 3, nbase, v, dt, l1);
                    small_map_exp_comm<N, M>(kp, B, w1, l0, l1, dt, xr, xi);
                } else {
                    for (int e = 0; e < nbase; ++e) {
                        double k[M];
                        double2 ck[M];
                        exp_row<M>(kp, e, nbase, v, dt, k);
#pragma unroll
                        for (int m = 0; m < M; ++m) ck[m] = make_double2(k[m], 0.0);
                        small_map_exp<N, M>(kp, B, ck, xr, xi);
                    }
                }
                if (nerr) {  // embedded lower-order solution from x0 (cfm.rs:88-95, magnus.rs:76-78), then x_err = that - xf
                    double er[N], ei[N];
#pragma unroll
                    for (int r = 0; r < N; ++r) {
                        const double2 v0 = sx0[r * VO_EXP_SMALL_THREADS + threadIdx.x];
                        er[r] = v0.x, ei[r] = v0.y;
                    }
                    for (int e = nbase; e < nbase + nerr; ++e) {
                        double k[M];
                        double2 ck[M];
                        exp_row<M>(kp, e, nbase, v, dt, k);
#pragma unroll
                        for (int m = 0; m < M; ++m) ck[m] = make_double2(k[m], 0.0);
                        small_map_exp<N, M>(kp, B, ck, er, ei);
                    }
                    double nn = 0.0;
#ifdef VO_USER_NORM  // the caller's norm (NormFn): finish(JOIN_r map(x_err_r, r))
#pragma unroll
                    for (int r = 0; r < N; ++r) nn = vo_user_join(nn, VoUserNorm::map(er[r] - xr[r], ei[r] - xi[r], r, N));
                    err = VoUserNorm::finish(nn, N);
#else
#pragma unroll
                    for (int r = 0; r < N; ++r) {
                        const double dr = er[r] - xr[r], di = ei[r] - xi[r];
                        nn += dr * dr + di * di;
                    }
                    err = sqrt(nn);
#endif
                }
            } else if (const int64_t row = exp_out_row(kp, (int)(word & VO_WORD_TGT_MASK), sys); row >= 0) {  // Chkpt / End: the state current() shows
                if (kp.snap)
#pragma unroll
                    for (int r = 0; r < N; ++r) kp.snap[row * N + r] = make_double2(xr[r], xi[r]);
                if (kp.n_obs) {  // from x0's slot, free outside a step
#pragma unroll
                    for (int r = 0; r < N; ++r) sx0[r * VO_EXP_SMALL_THREADS + threadIdx.x] = make_double2(xr[r], xi[r]);
                    small_expect<N>(kp.obs, kp.n_obs, sx0 + threadIdx.x, kp.obs_out + row * kp.n_obs);
                }
            }
            const int fin = exp_event_finish(kp, c, evk, word, h, dt, [&]() { return err; }, cnt);
            if (fin == VO_EV_STEP) {
                moved = true;
            } else if (evk == VO_EV_STEP) {  // rejected: back to x0
#pragma unroll
                for (int r = 0; r < N; ++r) {
                    const double2 v0 = sx0[r * VO_EXP_SMALL_THREADS + threadIdx.x];
                    xr[r] = v0.x, xi[r] = v0.y;
                }
            }
        }
        ca.t[sys] = c.t_, ca.h[sys] = c.h_, ca.prev_h[sys] = c.prev_h_, ca.dx_norm[sys] = c.dx_norm_;
        ca.n_accept[sys] = c.n_accept_, ca.n_reject[sys] = c.n_reject_, ca.word[sys] = c.word_;
        if (moved)
#pragma unroll
            for (int r = 0; r < N; ++r) psi[sys * N + r] = make_double2(xr[r], xi[r]);
    }
    if (kp.mode == 0 && kp.count_events) exp_counts_flush(ev + ((blockIdx.x * (VO_EXP_SMALL_THREADS / 32) + (threadIdx.x >> 5)) % VO_EV_SLOTS), cnt);
}
