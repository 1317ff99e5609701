// exp_kernels.cuh — device side of the exponential integrators (see exp.cu for the design). Kept free of host headers so that
// a user-defined generator (vo_exp_set_generator, nvrtc_rhs.cu) can be compiled at run time into the very same kernel.
#pragma once
#include "common.cuh"
#include "rk_small.cuh"  // CtlArrays / EvSlot / status-word layout shared with the RK solver

#define VO_EXP_MAX_M 4
#define VO_EXP_MAX_NODES 4  // quadrature nodes of a commutator-free scheme (cfm_general's `c`, exp/cfm.rs:47)
#define VO_EXP_MAX_ROWS 8   // exponentials of the propagated solution: rows of `alpha` (cfm.rs:48), or the 2 s + 1 factors of split_cfm
#define VO_EXP_MAX_ERR 4    // exponentials of the embedded lower-order solution: rows of `alph_err` (cfm.rs:52)
#define VO_EXP_MAX_E (VO_EXP_MAX_ROWS + VO_EXP_MAX_ERR)

struct ExpKP {
    int n, M, M_gen, scheme, adaptive, want_err, taylor_deg, mode;  // mode 0: solver event, 1: bare map_exp
    int pw_is_third, count_events;
    int applied_comm;     // vo_exp_set_applied_commutator: magnus_42's commutator applied to the state by products, never formed (no structure tensor)
    int literal_norm;     // vo_exp_set_literal_norm: the controller reads ca.dx_norm (= ||x0||, never rewritten) instead of ||x_err||, magnus.rs:274-276
    int nseq;             // mode 1: exponentials applied one after the other, coefficient sets [nseq][N][M]
    int n_events;         // mode 0, exp_small_kernel: events per system and launch (vo_exp_run fuses several; exp_step_kernel runs one)
    unsigned split_mask;  // VO_EXP_SPLIT_MIDPOINT: bit m set <=> basis matrix m belongs to split A
    // ODEData.t_list (ode.rs:89): the first VO_INLINE_TLIST entries inline, a device copy of the whole list when it is longer
    int n_tlist;
    double t_list_inline[VO_INLINE_TLIST];
    const double* t_list;
    // Output at every Chkpt / End event for t_list[k], row k of the CALLER's order: system `sys` of the device writes row
    // out_perm[sys] (vo_exp_set_order; NULL = the identity), so every entry is a plain view (exp_out_row).
    // snap (nullable): [n_tlist][N][n], the state the system shows at the event.
    // obs_out (with n_obs > 0): [n_tlist][N][n_obs], <psi| O_k |psi> of that state for the operators obs [n_obs][n][n] (row-major).
    double2* snap;
    const int64_t* out_perm;
    int n_obs;
    const double2* obs;
    double2* obs_out;
    double rtol, alpha, pw, min_dt, max_dt;
    double norm1[VO_EXP_MAX_M];
    double cs[VO_EXP_MAX_M * VO_EXP_MAX_M * VO_EXP_MAX_M];
    int64_t N;
    // commutator-free schemes as TABLES, the arguments of cfm_general (exp/cfm.rs:43-53) and split_cfm (exp/split_exp.rs:568-575):
    // exponential e of a step is exp(dt * sum_q tab_alpha[e][q] L(t + tab_c[q] dt)), restricted to the basis matrices of split A
    // (row_split 1) or of split B (2) or to none (0). VO_EXP_CFM4 is the tables of dat/mod.rs:4, 67-74 through the same code.
    int n_nodes, n_rows, n_rows_err;
    double tab_c[VO_EXP_MAX_NODES];
    double tab_alpha[VO_EXP_MAX_ROWS * VO_EXP_MAX_NODES];
    double tab_alpha_err[VO_EXP_MAX_ERR * VO_EXP_MAX_NODES];
    unsigned char row_split[VO_EXP_MAX_ROWS];
};

// (the literals of dat/mod.rs:4, 67-80 — C_GAUSS_LEGENDRE_4, CFM_R2_J1_GL, CFM_R4_J2_GL, BLANES17_R4_J4 — live in exp.cu, which
// hands them to the kernel as tables)

#ifdef VO_USER_NORM
__device__ __forceinline__ double vo_user_join(double a, double b) { return VoUserNorm::JOIN == 1 ? fmax(a, b) : a + b; }
#endif

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Taylor plan of map_exp (same rule as the CPU restatement): sub-steps so that theta/sq <= 1, then the smallest degree
// whose term falls below 2^-53.
__device__ __forceinline__ void taylor_plan(double theta, int forced_deg, int* sq, int* deg) {
    int s = theta > 1.0 ? (int)ceil(theta) : 1;
    const double th = theta / s;
    double term = 1.0;
    int k = 0;
    while (k < 60) {
        ++k;
        term = term * th / k;
        if (term <= 1.1102230246251565e-16) break;
    }
    *sq = s, *deg = forced_deg > 0 ? forced_deg : k;
}

template <int NDIM, int M, int TB> struct Geo {
    static constexpr int NW = NDIM / 8;      // row blocks of 8 (one warp each per column group)
    static constexpr int NK = NDIM / 4;      // k-steps of 4
    static constexpr int NCG = TB / 16;      // column groups of 16 systems
    static constexpr int NT = 2;             // n-tiles of 8 columns per warp
    static constexpr int LDT = NDIM + 4;     // padded row of the term buffer: conflict-free B-fragment loads
    static constexpr int THREADS = NW * NCG * 32;
    static constexpr int NBUF = (M * 2 * NDIM * NDIM * 8 + 2 * 2 * TB * LDT * 8 > 200 * 1024) ? 1 : 2;
    static constexpr size_t SMEM_B = (size_t)M * 2 * NDIM * NDIM * sizeof(double);
    static constexpr size_t SMEM_T = (size_t)NBUF * 2 * TB * LDT * sizeof(double);
    static constexpr size_t SMEM_COEF = (size_t)VO_EXP_MAX_E * M * TB * sizeof(double2);
    static constexpr size_t SMEM_MISC = (size_t)(NW * TB + VO_EXP_MAX_E * TB + TB) * sizeof(double) + (size_t)(TB + 2 * VO_EXP_MAX_E + 8) * sizeof(int) +
                                        (size_t)TB * 2 * sizeof(long long);
    static constexpr size_t SMEM = SMEM_B + SMEM_T + SMEM_COEF + SMEM_MISC;
    static_assert(SMEM <= 227 * 1024, "exp_step_kernel: shared memory budget of one SM exceeded");
};

// Barrier among the NW warps of ONE column group (16 systems). A tile of TB = 16 NCG systems is NCG such groups that share the basis
// in shared memory but nothing else inside a Taylor series: each republishes its own columns of the term buffer, so each can run
// behind its own named barrier and the groups drift apart in phase — while one group waits at its barrier the other keeps the tensor
// pipe busy. NCG == 1 is the plain block barrier.
template <int NW, int NCG> __device__ __forceinline__ void group_sync(int cg) {
    if (NCG == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + cg), "r"(NW * 32) : "memory");
}

// x <- exp(sum_m coef[m][s] B_m) x for the tile, state in C-fragment layout:
// lane l of warp (w, cg) owns row 8w + l/4 and columns 16cg + 8j + 2(l%4) + q, j,q in {0,1}.
template <int NDIM, int M, int TB>
__device__ __forceinline__ void map_exp_tile(const double* __restrict__ sB, double* __restrict__ sT, const double2* __restrict__ sCoefE, int sq, int deg,
                                             double (&xr)[2][2], double (&xi)[2][2], int& buf) {
    using G = Geo<NDIM, M, TB>;
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const int w = wi % G::NW, cg = wi / G::NW;
    const int row = 8 * w + (lane >> 2);
    const double inv_sq = 1.0 / sq;
    double cr[M][2][2], ci[M][2][2];  // coefficients / sq of this lane's four systems
#pragma unroll
    for (int m = 0; m < M; ++m)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const double2 c = sCoefE[m * TB + 16 * cg + 8 * j + 2 * (lane & 3) + q];
                cr[m][j][q] = c.x * inv_sq, ci[m][j][q] = c.y * inv_sq;
            }
    for (int rep = 0; rep < sq; ++rep) {
        double ar[2][2], ai[2][2], tr[2][2], ti[2][2];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) ar[j][q] = tr[j][q] = xr[j][q], ai[j][q] = ti[j][q] = xi[j][q];
        for (int k = 1; k <= deg; ++k) {
            // publish the current term: planar [plane][column][LDT], row fastest
            if (G::NBUF == 1) group_sync<G::NW, G::NCG>(cg);
            double* Tr = sT + (size_t)buf * 2 * TB * G::LDT;
            double* Ti = Tr + TB * G::LDT;
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int col = 16 * cg + 8 * j + 2 * (lane & 3) + q;
                    Tr[col * G::LDT + row] = tr[j][q], Ti[col * G::LDT + row] = ti[j][q];
                }
            group_sync<G::NW, G::NCG>(cg);
            double Wr[M][2][2], Wi[M][2][2];
#pragma unroll
            for (int m = 0; m < M; ++m)
#pragma unroll
                for (int j = 0; j < 2; ++j) Wr[m][j][0] = Wr[m][j][1] = Wi[m][j][0] = Wi[m][j][1] = 0.0;
            const double* bA = sB + ((size_t)w * G::NK) * 32 + lane;  // + ((m*2 + plane) * NW) * NK * 32 + kk * 32
            const double* bX = Tr + (16 * cg + (lane >> 2)) * G::LDT + (lane & 3);
#pragma unroll 4
            for (int kk = 0; kk < G::NK; ++kk) {
                double fr[2], fi[2], nfi[2];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    fr[j] = bX[8 * j * G::LDT + 4 * kk];
                    fi[j] = bX[TB * G::LDT + 8 * j * G::LDT + 4 * kk];
                    nfi[j] = -fi[j];
                }
                // the asm statements are volatile, so the DMMAs issue in program order: every accumulator is written twice per k-step, and the
                // two writes are kept 4 M instructions apart (first the products with Xr, then those with Xi) instead of back to back
                double a_re[M], a_im[M];
#pragma unroll
                for (int m = 0; m < M; ++m) {
                    a_re[m] = bA[((size_t)(m * 2 + 0) * G::NW) * G::NK * 32 + kk * 32];
                    a_im[m] = bA[((size_t)(m * 2 + 1) * G::NW) * G::NK * 32 + kk * 32];
                }
#pragma unroll
                for (int m = 0; m < M; ++m)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        dmma(Wr[m][j][0], Wr[m][j][1], a_re[m], fr[j]);   // Re += Br Xr
                        dmma(Wi[m][j][0], Wi[m][j][1], a_im[m], fr[j]);   // Im += Bi Xr
                    }
#pragma unroll
                for (int m = 0; m < M; ++m)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        dmma(Wr[m][j][0], Wr[m][j][1], a_im[m], nfi[j]);  // Re -= Bi Xi
                        dmma(Wi[m][j][0], Wi[m][j][1], a_re[m], fi[j]);   // Im += Br Xi
                    }
            }
            const double ik = 1.0 / k;
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    double sr = 0.0, si = 0.0;
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        sr += cr[m][j][q] * Wr[m][j][q] - ci[m][j][q] * Wi[m][j][q];
                        si += cr[m][j][q] * Wi[m][j][q] + ci[m][j][q] * Wr[m][j][q];
                    }
                    tr[j][q] = sr * ik, ti[j][q] = si * ik;
                    ar[j][q] += tr[j][q], ai[j][q] += ti[j][q];
                }
            if (G::NBUF == 2) buf ^= 1;
        }
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) xr[j][q] = ar[j][q], xi[j][q] = ai[j][q];
    }
}

// W_m = B_m T for every basis matrix, T the tile of column vectors held in C-fragment layout (tr, ti): the body of one Taylor term
// of map_exp_tile as a function. Publishes T to the term buffer, one block barrier, NK k-steps of 8 M DMMAs.
template <int NDIM, int M, int TB>
__device__ __forceinline__ void basis_apply(const double* __restrict__ sB, double* __restrict__ sT, int& buf, const double (&tr)[2][2], const double (&ti)[2][2],
                                            double (&Wr)[M][2][2], double (&Wi)[M][2][2]) {
    using G = Geo<NDIM, M, TB>;
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const int w = wi % G::NW, cg = wi / G::NW;
    const int row = 8 * w + (lane >> 2);
    if (G::NBUF == 1) group_sync<G::NW, G::NCG>(cg);
    double* Tr = sT + (size_t)buf * 2 * TB * G::LDT;
    double* Ti = Tr + TB * G::LDT;
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int col = 16 * cg + 8 * j + 2 * (lane & 3) + q;
            Tr[col * G::LDT + row] = tr[j][q], Ti[col * G::LDT + row] = ti[j][q];
        }
    group_sync<G::NW, G::NCG>(cg);
#pragma unroll
    for (int m = 0; m < M; ++m)
#pragma unroll
        for (int j = 0; j < 2; ++j) Wr[m][j][0] = Wr[m][j][1] = Wi[m][j][0] = Wi[m][j][1] = 0.0;
    const double* bA = sB + ((size_t)w * G::NK) * 32 + lane;
    const double* bX = Tr + (16 * cg + (lane >> 2)) * G::LDT + (lane & 3);
#pragma unroll 4
    for (int kk = 0; kk < G::NK; ++kk) {
        double fr[2], fi[2], nfi[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            fr[j] = bX[8 * j * G::LDT + 4 * kk];
            fi[j] = bX[TB * G::LDT + 8 * j * G::LDT + 4 * kk];
            nfi[j] = -fi[j];
        }
        double a_re[M], a_im[M];  // dependent DMMAs 4 M instructions apart, as in map_exp_tile
#pragma unroll
        for (int m = 0; m < M; ++m) {
            a_re[m] = bA[((size_t)(m * 2 + 0) * G::NW) * G::NK * 32 + kk * 32];
            a_im[m] = bA[((size_t)(m * 2 + 1) * G::NW) * G::NK * 32 + kk * 32];
        }
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                dmma(Wr[m][j][0], Wr[m][j][1], a_re[m], fr[j]);
                dmma(Wi[m][j][0], Wi[m][j][1], a_im[m], fr[j]);
            }
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                dmma(Wr[m][j][0], Wr[m][j][1], a_im[m], nfi[j]);
                dmma(Wi[m][j][0], Wi[m][j][1], a_re[m], fi[j]);
            }
    }
    if (G::NBUF == 2) buf ^= 1;
}

// x <- exp(Omega) x for magnus_42 (exp/magnus.rs:28-83) WITHOUT forming the commutator: with L0, L1 the generator at the two Gauss
// nodes, Omega = W1 + b2 [L0, L1], W1 = b1 (L0 + L1), and a Taylor term needs only Omega T = W1 T + b2 (L0 (L1 T) - L1 (L0 T)): three
// passes over the shared basis per term (T; L1 T; L0 T), each M tile products on the tensor cores, combined with the per-system REAL
// coefficients of L0, L1 and W1. Nothing about closure under commutation is assumed and no n x n matrix is formed per system.
// sW1 / sL0 / sL1: coefficient slots [M][TB] (imaginary parts ignored: the generator coefficients are real), sDt: the step per system.
template <int NDIM, int M, int TB>
__device__ __forceinline__ void map_exp_tile_comm(const double* __restrict__ sB, double* __restrict__ sT, const double2* __restrict__ sW1,
                                                  const double2* __restrict__ sL0, const double2* __restrict__ sL1, const double* __restrict__ sDt, int sq, int deg,
                                                  double (&xr)[2][2], double (&xi)[2][2], int& buf) {
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const int cg = wi / Geo<NDIM, M, TB>::NW;
    const double inv_sq = 1.0 / sq;
    int col[2][2];
    double b2[2][2];
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            col[j][q] = 16 * cg + 8 * j + 2 * (lane & 3) + q;
            const double dt = sDt[col[j][q]];
            b2[j][q] = dt * dt * -0.144337567297406441127287195125 * inv_sq;  // magnus.rs:41 (b2 = -sqrt(3)/12 dt^2), per sub-step
        }
    for (int rep = 0; rep < sq; ++rep) {
        double ar[2][2], ai[2][2], tr[2][2], ti[2][2];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) ar[j][q] = tr[j][q] = xr[j][q], ai[j][q] = ti[j][q] = xi[j][q];
        for (int k = 1; k <= deg; ++k) {
            double Wr[M][2][2], Wi[M][2][2];
            double lr[2][2], li[2][2], u0r[2][2], u0i[2][2], u1r[2][2], u1i[2][2];
            basis_apply<NDIM, M, TB>(sB, sT, buf, tr, ti, Wr, Wi);  // W_m = B_m T
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    double a = 0.0, b = 0.0, c = 0.0, d = 0.0, e = 0.0, f = 0.0;
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        const double w1 = sW1[m * TB + col[j][q]].x, l0 = sL0[m * TB + col[j][q]].x, l1 = sL1[m * TB + col[j][q]].x;
                        a += w1 * Wr[m][j][q], b += w1 * Wi[m][j][q];
                        c += l0 * Wr[m][j][q], d += l0 * Wi[m][j][q];
                        e += l1 * Wr[m][j][q], f += l1 * Wi[m][j][q];
                    }
                    lr[j][q] = a * inv_sq, li[j][q] = b * inv_sq, u0r[j][q] = c, u0i[j][q] = d, u1r[j][q] = e, u1i[j][q] = f;
                }
            basis_apply<NDIM, M, TB>(sB, sT, buf, u1r, u1i, Wr, Wi);  // B_m (L1 T)
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    double c = 0.0, d = 0.0;
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        const double l0 = sL0[m * TB + col[j][q]].x;
                        c += l0 * Wr[m][j][q], d += l0 * Wi[m][j][q];
                    }
                    lr[j][q] += b2[j][q] * c, li[j][q] += b2[j][q] * d;  // + b2 L0 L1 T
                }
            basis_apply<NDIM, M, TB>(sB, sT, buf, u0r, u0i, Wr, Wi);  // B_m (L0 T)
            const double ik = 1.0 / k;
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    double e = 0.0, f = 0.0;
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        const double l1 = sL1[m * TB + col[j][q]].x;
                        e += l1 * Wr[m][j][q], f += l1 * Wi[m][j][q];
                    }
                    tr[j][q] = (lr[j][q] - b2[j][q] * e) * ik, ti[j][q] = (li[j][q] - b2[j][q] * f) * ik;  // - b2 L1 L0 T, then / k
                    ar[j][q] += tr[j][q], ai[j][q] += ti[j][q];
                }
        }
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) xr[j][q] = ar[j][q], xi[j][q] = ai[j][q];
    }
}

// generator family: L(t) = B_0 + sum_{m=1}^{M_gen-1} amp_m cos(omega_m t + phase_m) B_m ; coefficients beyond M_gen are 0.
// The generator closures of the reference (`FnMut(T) -> L`, exp/cfm.rs:54, exp/magnus.rs:12,32) are a functor GEN with this
// shape; GenCos is the compiled-in family, a user-defined one is compiled at run time (vo_exp_set_generator).
struct GenCos {
    template <int M> static __device__ __forceinline__ void coef(const double* __restrict__ gp, int M_gen, double t, double (&c)[M]) {
#pragma unroll
        for (int m = 0; m < M; ++m) c[m] = 0.0;
        c[0] = 1.0;
#pragma unroll
        for (int m = 1; m < M; ++m)
            if (m < M_gen) c[m] = gp[(m - 1) * 3 + 0] * cos(gp[(m - 1) * 3 + 1] * t + gp[(m - 1) * 3 + 2]);
    }
};

// ---- per-system logic of one event, shared by exp_step_kernel (tiles of 16 systems on the tensor cores, n >= 16) and
// exp_small_kernel (exp_small_kernels.cuh: one system per thread, n <= 8). Only the exponentials differ between the two.

// Exponentials of an event: nbase for the propagated solution, then nerr for the embedded lower-order one (from x0).
__device__ __forceinline__ void exp_counts_of(const ExpKP& kp, int* nbase, int* nerr) {
    const bool tables = kp.scheme == VO_EXP_CFM4 || kp.scheme == VO_EXP_CFM_TABLE || kp.scheme == VO_EXP_SPLIT_CFM;
    *nbase = kp.mode == 1 ? 1 : (tables ? kp.n_rows : (kp.scheme == VO_EXP_SPLIT_MIDPOINT ? 3 : 1));
    *nerr = (kp.mode == 0 && kp.want_err) ? (tables ? kp.n_rows_err : (kp.scheme == VO_EXP_MAGNUS42 ? 1 : 0)) : 0;
}

// step_size_of (ode.rs:165-176) + check_step (ode.rs:389-399) against t_list[tgt]: the kind of this system's coming event (255: the
// trajectory is done) and, for a step, its size dt. Chkpt at every entry before the last, End at the last.
__device__ __forceinline__ int exp_event_kind(const ExpKP& kp, uint32_t word, double t, double h, double& dt) {
    int evk = 255;
    if (!((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE)) {
        const int tgt = (int)(word & VO_WORD_TGT_MASK);
        if (tgt >= kp.n_tlist) {
            evk = VO_EV_END;
        } else {
            const double rem = (kp.n_tlist > VO_INLINE_TLIST ? kp.t_list[tgt] : kp.t_list_inline[tgt]) - t;
            if (fabs(rem) <= 2.220446049250313e-16) evk = tgt >= kp.n_tlist - 1 ? VO_EV_END : VO_EV_CHKPT;
            else dt = rem < h ? rem : h, evk = VO_EV_STEP;
        }
    }
    return evk;
}

// The row of the [n_tlist][N] outputs that system `sys` writes at its Chkpt / End event for t_list[tgt] (tgt: the target of the status
// word the event started from), or -1 when neither snapshots nor observables are on or the target lies past the list. The snapshot
// goes to kp.snap + row n, the expectation values to kp.obs_out + row n_obs.
__device__ __forceinline__ int64_t exp_out_row(const ExpKP& kp, int tgt, int64_t sys) {
    if ((!kp.snap && !kp.n_obs) || tgt >= kp.n_tlist) return -1;
    return (int64_t)tgt * kp.N + (kp.out_perm ? kp.out_perm[sys] : sys);
}

// dst[k] = <x| O_k |x> = sum_r conj(x_r) sum_c O_k[r][c] x_c for k = k0, k0 + dk, ... < n_obs (obs [n_obs][n][n]), by one warp (all 32
// lanes call; n a multiple of 8, at most 64). Lane l owns columns c = l and l + 32: it forms (O_k^T conj(x))_c from coalesced reads of the operator
// rows (ROWS of them in flight: the operators come from L2) and broadcast reads of x_r, multiplies by x_c, and a shuffle reduction
// adds the lanes. x: one system's state in global memory, not written during the call.
template <int ROWS>
__device__ __forceinline__ void exp_expect_warp(const double2* __restrict__ obs, int n_obs, int n, const double2* x, int k0, int dk, double2* dst) {
    const int lane = threadIdx.x & 31;
    const double2 zero = make_double2(0.0, 0.0);
    const double2 x0 = lane < n ? x[lane] : zero, x1 = lane + 32 < n ? x[lane + 32] : zero;
    for (int k = k0; k < n_obs; k += dk) {
        const double2* O = obs + (size_t)k * n * n;
        double er = 0.0, ei = 0.0;
#pragma unroll 1
        for (int h = 0; h < 2 && 32 * h < n; ++h) {
            const int c = lane + 32 * h;
            const bool mine = c < n;
            double ar = 0.0, ai = 0.0;
#pragma unroll ROWS
            for (int r = 0; r < n; ++r) {
                const double2 o = mine ? O[r * n + c] : zero;
                const double2 v = x[r];
                ar = fma(v.x, o.x, fma(v.y, o.y, ar));
                ai = fma(v.x, o.y, fma(-v.y, o.x, ai));
            }
            const double2 v = h ? x1 : x0;
            er = fma(ar, v.x, fma(-ai, v.y, er));
            ei = fma(ar, v.y, fma(ai, v.x, ei));
        }
        for (int o = 16; o > 0; o >>= 1) er += __shfl_xor_sync(0xffffffffu, er, o), ei += __shfl_xor_sync(0xffffffffu, ei, o);
        if (lane == 0) dst[k] = make_double2(er, ei);
    }
}

// The generator samples a step's exponents are built from (g: this system's generator parameters): midpoint at t + dt/2
// (exp/magnus.rs:10-26); the tables at every node t + c_q dt (cfm.rs:70-72); split midpoint at t (split_exp.rs:520-562 samples
// there, not at t + dt/2); magnus_42 at the two Gauss nodes (magnus.rs:28-83).
template <int M, class GEN>
__device__ __forceinline__ void exp_samples(const ExpKP& kp, const double* g, double t, double dt, double (&v)[VO_EXP_MAX_NODES][M]) {
    if (kp.scheme == VO_EXP_MIDPOINT) {
        GEN::template coef<M>(g, kp.M_gen, t + dt * 0.5, v[0]);
    } else if (kp.scheme == VO_EXP_CFM4 || kp.scheme == VO_EXP_CFM_TABLE || kp.scheme == VO_EXP_SPLIT_CFM) {
#pragma unroll
        for (int q = 0; q < VO_EXP_MAX_NODES; ++q)
            if (q < kp.n_nodes) GEN::template coef<M>(g, kp.M_gen, t + kp.tab_c[q] * dt, v[q]);
    } else if (kp.scheme == VO_EXP_SPLIT_MIDPOINT) {
        GEN::template coef<M>(g, kp.M_gen, t, v[0]);
    } else {
        const double c_mid = 0.288675134594812882254574390251;
        const double b1 = dt * 0.5;
        const double mid_t = t + b1;
        GEN::template coef<M>(g, kp.M_gen, mid_t - c_mid * dt, v[0]);
        GEN::template coef<M>(g, kp.M_gen, mid_t + c_mid * dt, v[1]);
    }
}

// Exponent e of a step, exp(sum_m k[m] B_m), from the samples v (real generator coefficients, so k is real).
//   midpoint: e = 0 only. Tables (cfm_general / split_cfm): cfm_exp (cfm.rs:31-37), k = a_0 m_0; k += a_q m_q; k *= dt, with row e of
//   alpha (e < nbase) or of alph_err, restricted to split A or B by row_split. Split midpoint: A, B, A, each scaled by dt/2
//   (split_exp.rs:540-559). magnus_42: 0 = w1 + w2 b2 (w1 alone with the applied commutator), 1 = w1 (the embedded solution),
//   2 = L0, 3 = L1 (the applied commutator's two generators).
template <int M>
__device__ __forceinline__ void exp_row(const ExpKP& kp, int e, int nbase, const double (&v)[VO_EXP_MAX_NODES][M], double dt, double (&k)[M]) {
    if (kp.scheme == VO_EXP_MIDPOINT) {
#pragma unroll
        for (int m = 0; m < M; ++m) k[m] = v[0][m] * dt;
    } else if (kp.scheme == VO_EXP_CFM4 || kp.scheme == VO_EXP_CFM_TABLE || kp.scheme == VO_EXP_SPLIT_CFM) {
        const double* a = e < nbase ? &kp.tab_alpha[e * VO_EXP_MAX_NODES] : &kp.tab_alpha_err[(e - nbase) * VO_EXP_MAX_NODES];
        const int side = e < nbase ? kp.row_split[e] : 0;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            double s = a[0] * v[0][m];
#pragma unroll
            for (int q = 1; q < VO_EXP_MAX_NODES; ++q)
                if (q < kp.n_nodes) s = s + (a[q] * v[q][m]);
            const bool in_a = (kp.split_mask >> m) & 1u;
            const bool keep = side == 0 || (side == 1 ? in_a : !in_a);
            k[m] = keep ? s * dt : 0.0;
        }
    } else if (kp.scheme == VO_EXP_SPLIT_MIDPOINT) {
        const double dt0 = dt * 0.5;
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const bool in_a = (kp.split_mask >> m) & 1u;
            k[m] = ((e == 1) != in_a) ? v[0][m] * dt0 : 0.0;
        }
    } else {
        const double b1 = dt * 0.5, b2 = dt * dt * -0.144337567297406441127287195125;
        if (e >= 2) {
#pragma unroll
            for (int m = 0; m < M; ++m) k[m] = e == 2 ? v[0][m] : v[1][m];
            return;
        }
        double w2[M];
#pragma unroll
        for (int c = 0; c < M; ++c) w2[c] = 0.0;
        if (e == 0 && !kp.applied_comm) {
#pragma unroll
            for (int a = 0; a < M; ++a)
#pragma unroll
                for (int b = 0; b < M; ++b) {
                    const double ab = v[0][a] * v[1][b];
#pragma unroll
                    for (int c = 0; c < M; ++c) {
                        const double sc = kp.cs[(a * M + b) * M + c];
                        if (sc != 0.0) w2[c] = w2[c] + ab * sc;
                    }
                }
        }
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const double w1 = (v[0][m] + v[1][m]) * b1;
            k[m] = (e == 0 && !kp.applied_comm) ? w1 + w2[m] * b2 : w1;  // u = exp(w1 + w2); u1 = exp(w1), the 2nd-order embedded solution
        }
    }
}

// theta = sum_m |c_m| ||B_m||_1, the bound of ||sum_m c_m B_m||_1 that the Taylor plan (taylor_plan) is made from
template <int M, class C> __device__ __forceinline__ double exp_theta(const ExpKP& kp, C coef) {
    double th = 0.0;
#pragma unroll
    for (int m = 0; m < M; ++m) {
        const double2 c = coef(m);
        th += hypot(c.x, c.y) * kp.norm1[m];
    }
    return th;
}

// The applied commutator's share of the bound: ||Omega||_1 <= ||W1||_1 + 2 |b2| ||L0||_1 ||L1||_1 (l0, l1: real coefficients)
template <int M, class C0, class C1> __device__ __forceinline__ double exp_comm_theta(const ExpKP& kp, double dt, C0 l0, C1 l1) {
    double n0 = 0.0, n1 = 0.0;
#pragma unroll
    for (int m = 0; m < M; ++m) n0 += fabs(l0(m)) * kp.norm1[m], n1 += fabs(l1(m)) * kp.norm1[m];
    return 2.0 * (dt * dt * 0.144337567297406441127287195125) * n0 * n1;
}

// A system's control values in the solver's arrays, read and written in place.
struct CtlAt {
    CtlArrays ca;
    int64_t i;
    __device__ __forceinline__ double& t() { return ca.t[i]; }
    __device__ __forceinline__ double& h() { return ca.h[i]; }
    __device__ __forceinline__ double& prev_h() { return ca.prev_h[i]; }
    __device__ __forceinline__ double& dx_norm() { return ca.dx_norm[i]; }
    __device__ __forceinline__ uint32_t& n_accept() { return ca.n_accept[i]; }
    __device__ __forceinline__ uint32_t& n_reject() { return ca.n_reject[i]; }
    __device__ __forceinline__ uint32_t& word() { return ca.word[i]; }
};

struct ExpCounts {
    unsigned step = 0, chkpt = 0, rej = 0, end = 0, stuck = 0;
};

// The end of one event of one system (phase D): for a step the controller (handle_step_adaptive, ode.rs:311-334) or the fixed-step
// advance, for Chkpt / End checkpoint_update (ode.rs:192-195); then the status word. word and h are the values the event started
// from, dt its step. err_norm() gives ||x_err|| and is called by the adaptive controller alone. Returns the event's final kind
// (a step may become a rejection); only a VO_EV_STEP commits the new state.
template <class CTL, class NRM>
__device__ __forceinline__ int exp_event_finish(const ExpKP& kp, CTL& c, int evk, uint32_t word, double h, double dt, NRM err_norm, ExpCounts& cnt) {
    int tgt = (int)(word & VO_WORD_TGT_MASK);
    uint32_t status = word >> VO_WORD_STATUS_SHIFT;
    if (evk == VO_EV_STEP) {
        if (kp.adaptive) {
            const double dxn = kp.literal_norm ? c.dx_norm() : err_norm();
            const double f = kp.rtol / dxn;
            const double mul = step_size_mul<true>(kp.alpha, f, kp.pw, kp.pw_is_third);  // ode.rs:133-135, powf correctly rounded (rk_small.cuh)
            const double fp_lim = at_most(at_least(mul, 0.3), 2.0);
            const double new_h = at_most(at_least(fp_lim * h, kp.min_dt), kp.max_dt);
            if (!(dxn == dxn)) status |= VO_TRAJ_NONFINITE;
            if (f <= 1.0) {
                evk = VO_EV_REJECT;
                if (h <= kp.min_dt) status |= VO_TRAJ_STUCK, ++cnt.stuck;
            }
            c.prev_h() = h, c.h() = new_h, c.dx_norm() = dxn;
        }
        if (evk == VO_EV_STEP) c.t() += dt, c.n_accept() += 1, ++cnt.step;
        else c.n_reject() += 1, ++cnt.rej;
    } else {  // Chkpt / End
        tgt += 1, c.h() = c.prev_h();
        if (evk == VO_EV_END) status |= VO_TRAJ_DONE, ++cnt.end;
        else ++cnt.chkpt;
    }
    const uint32_t nw = ((uint32_t)tgt & VO_WORD_TGT_MASK) | (status << VO_WORD_STATUS_SHIFT);
    if (nw != word) c.word() = nw;
    return evk;
}

// The event counters of one warp (all 32 lanes call), added to one of the VO_EV_SLOTS slots by lane 0.
__device__ __forceinline__ void exp_counts_flush(EvSlot* slot, ExpCounts cnt) {
    cnt.step = __reduce_add_sync(0xffffffffu, cnt.step), cnt.chkpt = __reduce_add_sync(0xffffffffu, cnt.chkpt);
    cnt.rej = __reduce_add_sync(0xffffffffu, cnt.rej), cnt.end = __reduce_add_sync(0xffffffffu, cnt.end);
    cnt.stuck = __reduce_add_sync(0xffffffffu, cnt.stuck);
    if ((threadIdx.x & 31) == 0) {
        if (cnt.step) atomicAdd(&slot->n_step, (unsigned long long)cnt.step);
        if (cnt.chkpt) atomicAdd(&slot->n_chkpt, (unsigned long long)cnt.chkpt);
        if (cnt.rej) atomicAdd(&slot->n_reject, (unsigned long long)cnt.rej);
        if (cnt.end) atomicAdd(&slot->n_end, (unsigned long long)cnt.end);
        if (cnt.stuck) atomicAdd(&slot->n_stuck, (unsigned long long)cnt.stuck);
    }
}

template <int NDIM, int M, int TB, class GEN>
__global__ void __launch_bounds__(Geo<NDIM, M, TB>::THREADS, 1)
exp_step_kernel(const __grid_constant__ ExpKP kp, const double* __restrict__ frag, double2* __restrict__ psi, double2* __restrict__ psi_out,
                const double* __restrict__ gp, const double2* __restrict__ coef_in, const CtlArrays ca, EvSlot* __restrict__ ev,
                const int* __restrict__ order /* nullable: slot -> system, tiles of systems with similar ||L h|| (exp.cu: dynamic grouping) */,
                int* __restrict__ tile_ctr /* nullable: with `order`, tiles are handed out by this counter, largest theta first */) {
    using G = Geo<NDIM, M, TB>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* sB = reinterpret_cast<double*>(smem_raw);
    double* sT = reinterpret_cast<double*>(smem_raw + G::SMEM_B);
    double2* sCoef = reinterpret_cast<double2*>(smem_raw + G::SMEM_B + G::SMEM_T);               // [E][M][TB]
    double* sNorm = reinterpret_cast<double*>(smem_raw + G::SMEM_B + G::SMEM_T + G::SMEM_COEF);  // [NW][TB]
    double* sTheta = sNorm + G::NW * TB;                                                         // [E][TB]
    double* sDt = sTheta + VO_EXP_MAX_E * TB;                                                    // [TB]
    int* sEv = reinterpret_cast<int*>(sDt + TB);                                                 // [TB] event, then [2 E] plan, [1] any
    int* sPlan = sEv + TB;
    long long* sSys = reinterpret_cast<long long*>(smem_raw + G::SMEM - TB * sizeof(long long));  // [TB] system of each tile slot (kp.N = none)
    long long* sRow = sSys - TB;  // [TB] output row (exp_out_row) of the slot's Chkpt / End event of this tile, or -1
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const int w = wi % G::NW, cg = wi / G::NW;
    const int row = 8 * w + (lane >> 2);

    // the basis, already in A-fragment order, stays in shared memory for the life of the CTA
    for (size_t i = threadIdx.x; i < G::SMEM_B / sizeof(double2); i += blockDim.x)
        reinterpret_cast<double2*>(sB)[i] = reinterpret_cast<const double2*>(frag)[i];
    __syncthreads();

    const int64_t n_tiles = (kp.N + TB - 1) / TB;
    int buf = 0;
    ExpCounts cnt;
    // Tile -> slots. With the dynamic grouping the slots are sorted by ascending theta, so tiles differ in cost: they are then taken from
    // the expensive end and handed out by an atomic counter as CTAs become free (longest-processing-time-first), which also removes the
    // 42-or-43-tiles-per-CTA quantisation of a static stride. Without it: the static stride.
    const bool dyn_tiles = order != nullptr && tile_ctr != nullptr;
    auto tile_base = [&](int64_t tl) { return (dyn_tiles ? n_tiles - 1 - tl : tl) * TB; };
    // Control data of a tile's systems (solver events): which system sits in the slot, its status word, t, h and generator parameters.
    // The thread that owns slot s fetches them for the NEXT tile of this CTA while the current tile's exponentials run, so that phase A
    // starts from registers instead of a chain of four dependent global loads (order -> word -> t, h -> parameters) per tile.
    constexpr int PG = 3 * (VO_EXP_MAX_M - 1);
    long long p_sys = kp.N;
    uint32_t p_word = 0;
    double p_t = 0.0, p_h = 0.0, p_g[PG];
#pragma unroll
    for (int q = 0; q < PG; ++q) p_g[q] = 0.0;
    auto prefetch_ctl = [&](int64_t tl) {
        p_sys = kp.N;
        if (tl < n_tiles) {
            const int64_t slot = tile_base(tl) + threadIdx.x;
            if (slot < kp.N) p_sys = order ? (long long)order[slot] : slot;
        }
        if (p_sys < kp.N) {
            p_word = ca.word[p_sys], p_t = ca.t[p_sys], p_h = ca.h[p_sys];
            const double* g = gp + p_sys * (kp.M_gen - 1) * 3;
#pragma unroll
            for (int q = 0; q < PG; ++q)
                if (q < 3 * (kp.M_gen - 1)) p_g[q] = g[q];
        }
    };
    int64_t next_tile = 0;
    if (kp.mode == 0 && threadIdx.x < TB) prefetch_ctl(blockIdx.x);
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile = next_tile) {
        const int64_t base = tile_base(tile);
        uint32_t a_word = 0;  // this slot's status word and step size, from phase A to phase D (same thread)
        double a_h = 0.0;
        int nbase, nerr;
        exp_counts_of(kp, &nbase, &nerr);
        const int nexp = nbase + nerr;
        // ---- phase A: per-system control and exponent coefficients (one thread per system), written straight to shared memory
        if (threadIdx.x < TB) {
            const int s = threadIdx.x;
            const int64_t slot = base + s;
            int64_t sys;
            double a_t = 0.0, a_g[PG];
            if (kp.mode == 0) {  // from the prefetch of the previous iteration (the next tile's loads go out after phase B)
                sys = p_sys, a_word = p_word, a_t = p_t, a_h = p_h;
#pragma unroll
                for (int q = 0; q < PG; ++q) a_g[q] = p_g[q];
                prefetch_ctl(tile + gridDim.x);
            } else {
                sys = slot < kp.N ? (order ? (int64_t)order[slot] : slot) : kp.N;
#pragma unroll
                for (int q = 0; q < PG; ++q) a_g[q] = 0.0;
            }
            sSys[s] = sys;
            int evk = 255;  // not live
            double dt = 0.0;
            auto put = [&](int e, int m, double re, double im) { sCoef[(e * M + m) * TB + s] = make_double2(re, im); };
            for (int e = 0; e < (kp.applied_comm ? 4 : nexp); ++e)
#pragma unroll
                for (int m = 0; m < M; ++m) put(e, m, 0.0, 0.0);
            if (sys < kp.N) {
                if (kp.mode == 1) {
                    evk = VO_EV_STEP;
#pragma unroll
                    for (int m = 0; m < M; ++m) sCoef[m * TB + s] = coef_in[sys * M + m];
                } else {
                    evk = exp_event_kind(kp, a_word, a_t, a_h, dt);
                    if (evk == VO_EV_STEP) {
                        double v[VO_EXP_MAX_NODES][M];
                        exp_samples<M, GEN>(kp, a_g, a_t, dt, v);
                        for (int e = 0; e < (kp.applied_comm ? 4 : nexp); ++e) {
                            double k[M];
                            exp_row<M>(kp, e, nbase, v, dt, k);
#pragma unroll
                            for (int m = 0; m < M; ++m) put(e, m, k[m], 0.0);
                        }
                    }
                }
            }
            sEv[s] = evk, sDt[s] = dt;
            for (int e = 0; e < nexp; ++e) {
                const double th = exp_theta<M>(kp, [&](int m) { return sCoef[(e * M + m) * TB + s]; });
                sTheta[e * TB + s] = evk == VO_EV_STEP ? th : 0.0;
            }
            if (kp.applied_comm && kp.scheme == VO_EXP_MAGNUS42 && kp.mode == 0 && evk == VO_EV_STEP)
                sTheta[s] += exp_comm_theta<M>(kp, dt, [&](int m) { return sCoef[(2 * M + m) * TB + s].x; }, [&](int m) { return sCoef[(3 * M + m) * TB + s].x; });
        }
        __syncthreads();
        // ---- phase B: tile-uniform Taylor plan, one thread per exponential
        if (threadIdx.x < nexp) {
            const int e = threadIdx.x;
            double th = 0.0;
            for (int s = 0; s < TB; ++s) th = fmax(th, sTheta[e * TB + s]);
            taylor_plan(th, kp.taylor_deg, &sPlan[2 * e], &sPlan[2 * e + 1]);
        }
        if (threadIdx.x == 32) {
            int any = 0;
            for (int s = 0; s < TB; ++s) any |= sEv[s] == VO_EV_STEP;
            sPlan[2 * VO_EXP_MAX_E] = any;
            sPlan[2 * VO_EXP_MAX_E + 1] = dyn_tiles ? (int)gridDim.x + atomicAdd(tile_ctr, 1) : (int)(tile + gridDim.x);  // this CTA's next tile
        }
        __syncthreads();
        const bool any_step = sPlan[2 * VO_EXP_MAX_E] != 0;
        next_tile = sPlan[2 * VO_EXP_MAX_E + 1];
        if (kp.mode == 0 && threadIdx.x < TB) prefetch_ctl(next_tile);  // in flight during the exponentials below
        // ---- phase C: the exponentials
        double x0r[2][2], x0i[2][2], xfr[2][2], xfi[2][2], xer[2][2], xei[2][2];
        if (any_step) {
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int64_t sys = sSys[16 * cg + 8 * j + 2 * (lane & 3) + q];
                    const double2 v = sys < kp.N ? psi[sys * NDIM + row] : make_double2(0.0, 0.0);
                    x0r[j][q] = xfr[j][q] = v.x, x0i[j][q] = xfi[j][q] = v.y;
                    xer[j][q] = xei[j][q] = 0.0;
                }
            if (kp.applied_comm && kp.scheme == VO_EXP_MAGNUS42 && kp.mode == 0)
                map_exp_tile_comm<NDIM, M, TB>(sB, sT, sCoef, sCoef + 2 * M * TB, sCoef + 3 * M * TB, sDt, sPlan[0], sPlan[1], xfr, xfi, buf);
            else
                for (int e = 0; e < nbase; ++e) map_exp_tile<NDIM, M, TB>(sB, sT, sCoef + e * M * TB, sPlan[2 * e], sPlan[2 * e + 1], xfr, xfi, buf);
            for (int q = 1; kp.mode == 1 && q < kp.nseq; ++q) {  // vo_map_exp_seq: the next exponential of the composition
                __syncthreads();
                if (threadIdx.x < TB) {
                    const int64_t sys = sSys[threadIdx.x];
                    double th = 0.0;
#pragma unroll
                    for (int m = 0; m < M; ++m) {
                        const double2 c = sys < kp.N ? coef_in[((int64_t)q * kp.N + sys) * M + m] : make_double2(0.0, 0.0);
                        sCoef[m * TB + threadIdx.x] = c;
                        th += hypot(c.x, c.y) * kp.norm1[m];
                    }
                    sTheta[threadIdx.x] = th;
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    double th = 0.0;
                    for (int s = 0; s < TB; ++s) th = fmax(th, sTheta[s]);
                    taylor_plan(th, kp.taylor_deg, &sPlan[0], &sPlan[1]);
                }
                __syncthreads();
                map_exp_tile<NDIM, M, TB>(sB, sT, sCoef, sPlan[0], sPlan[1], xfr, xfi, buf);
            }
            if (nerr) {  // embedded lower-order solution from x0 (cfm.rs:88-95, magnus.rs:76-78), then x_err = that - xf
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int q = 0; q < 2; ++q) xer[j][q] = x0r[j][q], xei[j][q] = x0i[j][q];
                for (int e = nbase; e < nexp; ++e) map_exp_tile<NDIM, M, TB>(sB, sT, sCoef + e * M * TB, sPlan[2 * e], sPlan[2 * e + 1], xer, xei, buf);
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int q = 0; q < 2; ++q) xer[j][q] -= xfr[j][q], xei[j][q] -= xfi[j][q];
            }
        }
        // ---- phase D: error norm (2-norm of x_err per system), controller, apply_step
        if (kp.mode == 0) {
            if (any_step && kp.adaptive) {
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
#ifdef VO_USER_NORM  // the caller's norm (NormFn, exp/cfm.rs:105, 214-216): finish(JOIN_r map(x_err_r, r)); this lane holds row 8 w + lane / 4
                        double v = VoUserNorm::map(xer[j][q], xei[j][q], 8 * w + (lane >> 2), NDIM);
                        v = vo_user_join(v, __shfl_xor_sync(0xffffffffu, v, 4)), v = vo_user_join(v, __shfl_xor_sync(0xffffffffu, v, 8));
                        v = vo_user_join(v, __shfl_xor_sync(0xffffffffu, v, 16));
#else
                        double v = xer[j][q] * xer[j][q] + xei[j][q] * xei[j][q];
                        v += __shfl_xor_sync(0xffffffffu, v, 4), v += __shfl_xor_sync(0xffffffffu, v, 8), v += __shfl_xor_sync(0xffffffffu, v, 16);
#endif
                        if ((lane >> 2) == 0) sNorm[w * TB + 16 * cg + 8 * j + 2 * (lane & 3) + q] = v;
                    }
            }
            __syncthreads();
            if (threadIdx.x < TB) {
                const int s = threadIdx.x;
                const int64_t sys = sSys[s];
                int evk = sEv[s];
                sRow[s] = (evk == VO_EV_CHKPT || evk == VO_EV_END) ? exp_out_row(kp, (int)(a_word & VO_WORD_TGT_MASK), sys) : -1;
                if (evk != 255) {  // a_word, a_h: read in phase A by this thread; nothing has written them since
                    CtlAt c{ca, sys};
                    sEv[s] = exp_event_finish(kp, c, evk, a_word, a_h, sDt[s], [&]() {
                        double nn = 0.0;
#ifdef VO_USER_NORM
                        for (int ww = 0; ww < G::NW; ++ww) nn = vo_user_join(nn, sNorm[ww * TB + s]);
                        return VoUserNorm::finish(nn, NDIM);
#else
                        for (int ww = 0; ww < G::NW; ++ww) nn += sNorm[ww * TB + s];
                        return sqrt(nn);
#endif
                    }, cnt);
                }
            }
            __syncthreads();
        }
        // ---- phase E: masked commit (accepted systems only)
        if (any_step) {
            double2* dst = kp.mode == 1 ? psi_out : psi;
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int col = 16 * cg + 8 * j + 2 * (lane & 3) + q;
                    const int64_t sys = sSys[col];
                    if (sys < kp.N && sEv[col] == VO_EV_STEP) dst[sys * NDIM + row] = make_double2(xfr[j][q], xfi[j][q]);
                }
        }
        if (kp.mode == 0 && kp.snap) {  // the unchanged state of the systems at a Chkpt / End event, each lane its own rows
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int col = 16 * cg + 8 * j + 2 * (lane & 3) + q;
                    if (sRow[col] >= 0) kp.snap[sRow[col] * NDIM + row] = psi[sSys[col] * NDIM + row];
                }
        }
        if (kp.mode == 0 && kp.n_obs)  // expectation values of the same unchanged states, one warp per slot
            for (int s = wi; s < TB; s += G::THREADS / 32)
                if (sRow[s] >= 0) exp_expect_warp<8>(kp.obs, kp.n_obs, NDIM, psi + sSys[s] * NDIM, 0, 1, kp.obs_out + sRow[s] * kp.n_obs);
        __syncthreads();  // sEv / sCoef are rewritten by the next tile
    }
    if (kp.mode == 0 && kp.count_events && threadIdx.x < 32) exp_counts_flush(ev + (blockIdx.x % VO_EV_SLOTS), cnt);
}
