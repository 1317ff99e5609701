// exp_dense_kernels.cuh — ExponentialSplit / Commutator (src/exp/mod.rs:11-54) for GENERAL dense operators: every system owns its
// own n x n complex L (and explicit U = exp(L)), nothing is assumed about a shared basis or about closure under commutation.
//
// Storage: an operator ensemble is [N][n][n] complex, row-major, interleaved (re, im) — to the LinearCombination kernels it is
// just a flat vector of 2 n^2 N doubles. One CTA works on one system at a time with the operands in shared memory as two
// planes (re, im) of n rows padded to n + 4 doubles: both DMMA operand fragments (A: lane l holds [row l/4][k l%4]; B: lane l
// holds [k l%4][col l/4]) then read conflict-free from the SAME row-major layout, so a matrix can be the left operand of one
// product and the right operand of the next without re-arranging it (T <- T A in the Taylor series, U <- U U in the squarings,
// L0 L1 - L1 L0 in the commutator). Products run on the FP64 tensor cores (mma.sync m8n8k4; tcgen05 has no f64 kind): warp w
// owns rows 8w .. 8w+7 of the result and all n/8 column blocks, 4 DMMAs per complex 8x8x4 block.
#pragma once
#include "exp_kernels.cuh"

// acc (C-fragment layout: lane l holds [row 8w + l/4][col 8j + 2(l%4) + q]) += sign * A B, planar operands with row stride LD
template <int NB>
__device__ __forceinline__ void zgemm_acc(const double* __restrict__ Ar, const double* __restrict__ Ai, const double* __restrict__ Br, const double* __restrict__ Bi,
                                          int LD, bool negate, double (&cr)[NB][2], double (&ci)[NB][2]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const double* pa_r = Ar + (8 * w + (lane >> 2)) * LD + (lane & 3);
    const double* pa_i = Ai + (8 * w + (lane >> 2)) * LD + (lane & 3);
    const double* pb_r = Br + (lane & 3) * LD + (lane >> 2);
    const double* pb_i = Bi + (lane & 3) * LD + (lane >> 2);
#pragma unroll 2
    for (int kk = 0; kk < 2 * NB; ++kk) {
        double ar = pa_r[4 * kk], ai = pa_i[4 * kk];
        if (negate) ar = -ar, ai = -ai;
        const double nai = -ai;
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            const double br = pb_r[4 * kk * LD + 8 * j], bi = pb_i[4 * kk * LD + 8 * j];
            dmma(cr[j][0], cr[j][1], ar, br);   // Re += Ar Br
            dmma(cr[j][0], cr[j][1], nai, bi);  // Re -= Ai Bi
            dmma(ci[j][0], ci[j][1], ar, bi);   // Im += Ar Bi
            dmma(ci[j][0], ci[j][1], ai, br);   // Im += Ai Br
        }
    }
}

template <int NB> struct DenseGeo {
    static constexpr int N = 8 * NB, LD = N + 4, THREADS = 32 * NB;
    static constexpr size_t PLANE = (size_t)N * LD * sizeof(double);  // one plane of one matrix
    static constexpr size_t MAT = 2 * PLANE;
};

// global [n][n] interleaved -> planar padded shared (re plane, im plane)
template <int NB> __device__ __forceinline__ void dense_load(const double2* __restrict__ g, double* __restrict__ sr, double* __restrict__ si, double scale) {
    constexpr int N = 8 * NB, LD = N + 4;
    for (int e = threadIdx.x; e < N * N; e += 32 * NB) {
        const double2 v = g[e];
        sr[(e / N) * LD + e % N] = v.x * scale, si[(e / N) * LD + e % N] = v.y * scale;
    }
}

// fragment accumulators -> planar shared / interleaved global
template <int NB> __device__ __forceinline__ void frag_to_smem(const double (&cr)[NB][2], const double (&ci)[NB][2], double* __restrict__ sr, double* __restrict__ si) {
    constexpr int LD = 8 * NB + 4;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, row = 8 * w + (lane >> 2);
#pragma unroll
    for (int j = 0; j < NB; ++j)
#pragma unroll
        for (int q = 0; q < 2; ++q) sr[row * LD + 8 * j + 2 * (lane & 3) + q] = cr[j][q], si[row * LD + 8 * j + 2 * (lane & 3) + q] = ci[j][q];
}
template <int NB> __device__ __forceinline__ void frag_to_global(const double (&cr)[NB][2], const double (&ci)[NB][2], double2* __restrict__ g) {
    constexpr int N = 8 * NB;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, row = 8 * w + (lane >> 2);
#pragma unroll
    for (int j = 0; j < NB; ++j)  // two consecutive complex numbers per lane: one 32-byte store
        *reinterpret_cast<double4*>(g + row * N + 8 * j + 2 * (lane & 3)) = make_double4(cr[j][0], ci[j][0], cr[j][1], ci[j][1]);
}

// induced 1-norm of a planar shared matrix (largest column sum of |entries|); every thread returns it. `red` holds N + 1 doubles.
template <int NB> __device__ __forceinline__ double dense_norm1(const double* __restrict__ sr, const double* __restrict__ si, double* __restrict__ red) {
    constexpr int N = 8 * NB, LD = N + 4;
    __syncthreads();
    for (int c = threadIdx.x; c < N; c += 32 * NB) {
        double sum = 0.0;
        for (int r = 0; r < N; ++r) sum += hypot(sr[r * LD + c], si[r * LD + c]);
        red[c] = sum;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double best = 0.0;
        for (int c = 0; c < N; ++c) best = fmax(best, red[c]);
        red[N] = best;
    }
    __syncthreads();
    return red[N];
}

// ---- Commutator::commutator (exp/mod.rs:47-54): out = La Lb - Lb La, 2 x 8 n^3 flops per system --------------------------------
template <int NB>
__global__ void __launch_bounds__(32 * NB) dense_commutator_kernel(const double2* __restrict__ La, const double2* __restrict__ Lb, double2* __restrict__ out, int64_t N) {
    using G = DenseGeo<NB>;
    extern __shared__ __align__(16) unsigned char dsm[];
    double* a_r = reinterpret_cast<double*>(dsm);
    double* a_i = a_r + G::N * G::LD;
    double* b_r = a_i + G::N * G::LD;
    double* b_i = b_r + G::N * G::LD;
    for (int64_t sys = blockIdx.x; sys < N; sys += gridDim.x) {
        __syncthreads();
        dense_load<NB>(La + sys * G::N * G::N, a_r, a_i, 1.0);
        dense_load<NB>(Lb + sys * G::N * G::N, b_r, b_i, 1.0);
        __syncthreads();
        double cr[NB][2], ci[NB][2];
#pragma unroll
        for (int j = 0; j < NB; ++j) cr[j][0] = cr[j][1] = ci[j][0] = ci[j][1] = 0.0;
        zgemm_acc<NB>(a_r, a_i, b_r, b_i, G::LD, false, cr, ci);
        zgemm_acc<NB>(b_r, b_i, a_r, a_i, G::LD, true, cr, ci);
        frag_to_global<NB>(cr, ci, out + sys * G::N * G::N);
    }
}

// ---- ExponentialSplit::exp (exp/mod.rs:23): explicit U = exp(L) by scaling and squaring ---------------------------------------
// A = L / 2^s with ||A||_1 <= 1/2; U = sum_{k<=m} A^k / k! with the first term below 2^-53 (m <= 14); then s squarings.
// (m + s) complex GEMMs of 8 n^3 flops on the tensor cores; T_k = T_{k-1} A / k and U are accumulated in registers.
template <int NB>
__global__ void __launch_bounds__(32 * NB) dense_exp_kernel(const double2* __restrict__ L, double2* __restrict__ U, int64_t N, double k_scale) {
    using G = DenseGeo<NB>;
    extern __shared__ __align__(16) unsigned char dsm[];
    double* a_r = reinterpret_cast<double*>(dsm);
    double* a_i = a_r + G::N * G::LD;
    double* t_r = a_i + G::N * G::LD;
    double* t_i = t_r + G::N * G::LD;
    double* red = t_i + G::N * G::LD;  // N + 1 doubles, then the plan
    int* plan = reinterpret_cast<int*>(red + G::N + 2);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, row = 8 * w + (lane >> 2);
    for (int64_t sys = blockIdx.x; sys < N; sys += gridDim.x) {
        __syncthreads();
        dense_load<NB>(L + sys * G::N * G::N, a_r, a_i, k_scale);
        const double theta = dense_norm1<NB>(a_r, a_i, red);
        if (threadIdx.x == 0) {
            int s = 0;
            double th = theta;
            while (th > 0.5 && s < 60) th *= 0.5, ++s;
            double term = 1.0;
            int k = 0;
            while (k < 40) {
                ++k;
                term = term * th / k;
                if (term <= 1.1102230246251565e-16) break;
            }
            plan[0] = s, plan[1] = k;
        }
        __syncthreads();
        const int sq = plan[0], deg = plan[1];
        const double down = ldexp(1.0, -sq);
        for (int e = threadIdx.x; e < G::N * G::N; e += G::THREADS) {  // A <- A / 2^s (exact), T <- A
            const int o = (e / G::N) * G::LD + e % G::N;
            a_r[o] *= down, a_i[o] *= down;
            t_r[o] = a_r[o], t_i[o] = a_i[o];
        }
        __syncthreads();
        double ur[NB][2], ui[NB][2];  // U = I + A
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int col = 8 * j + 2 * (lane & 3) + q;
                ur[j][q] = a_r[row * G::LD + col] + (row == col ? 1.0 : 0.0), ui[j][q] = a_i[row * G::LD + col];
            }
        for (int k = 2; k <= deg; ++k) {  // T <- T A / k ; U += T
            double cr[NB][2], ci[NB][2];
#pragma unroll
            for (int j = 0; j < NB; ++j) cr[j][0] = cr[j][1] = ci[j][0] = ci[j][1] = 0.0;
            zgemm_acc<NB>(t_r, t_i, a_r, a_i, G::LD, false, cr, ci);
            const double ik = 1.0 / k;
#pragma unroll
            for (int j = 0; j < NB; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) cr[j][q] *= ik, ci[j][q] *= ik, ur[j][q] += cr[j][q], ui[j][q] += ci[j][q];
            __syncthreads();  // every warp has read the old T
            frag_to_smem<NB>(cr, ci, t_r, t_i);
            __syncthreads();
        }
        for (int s = 0; s < sq; ++s) {  // U <- U U
            __syncthreads();
            frag_to_smem<NB>(ur, ui, t_r, t_i);
            __syncthreads();
#pragma unroll
            for (int j = 0; j < NB; ++j) ur[j][0] = ur[j][1] = ui[j][0] = ui[j][1] = 0.0;
            zgemm_acc<NB>(t_r, t_i, t_r, t_i, G::LD, false, ur, ui);
        }
        frag_to_global<NB>(ur, ui, U + sys * G::N * G::N);
    }
}

// ---- ExponentialSplit::map_exp (exp/mod.rs:25) with an explicit U: y_i = U_i x_i, one warp per row group, U streamed once ------
__global__ void dense_matvec_kernel(const double2* __restrict__ U, const double2* __restrict__ x, double2* __restrict__ y, int n, int64_t N) {
    extern __shared__ __align__(16) unsigned char dsm[];
    double2* sx = reinterpret_cast<double2*>(dsm);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int64_t sys = blockIdx.x; sys < N; sys += gridDim.x) {
        __syncthreads();
        for (int c = threadIdx.x; c < n; c += blockDim.x) sx[c] = x[sys * n + c];
        __syncthreads();
        const double2* Us = U + sys * n * n;
        for (int r = w; r < n; r += nw) {
            double ar = 0.0, ai = 0.0;
            for (int c = lane; c < n; c += 32) {
                const double2 u = Us[r * n + c], v = sx[c];
                ar += u.x * v.x - u.y * v.y, ai += u.x * v.y + u.y * v.x;
            }
            for (int o = 16; o > 0; o >>= 1) ar += __shfl_xor_sync(0xffffffffu, ar, o), ai += __shfl_xor_sync(0xffffffffu, ai, o);
            if (lane == 0) y[sys * n + r] = make_double2(ar, ai);
        }
    }
}

// ---- L_i = sum_m coef[i][m] B_m: from the shared-basis representation to a dense operator ensemble -----------------------------
__global__ void dense_assemble_kernel(const double2* __restrict__ basis /* [M][n][n] */, const double2* __restrict__ coef /* [N][M] */, int M, int n, int64_t N,
                                      double2* __restrict__ L) {
    const int64_t nn = (int64_t)n * n;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < N * nn; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t sys = e / nn, k = e % nn;
        double re = 0.0, im = 0.0;
        for (int m = 0; m < M; ++m) {
            const double2 c = coef[sys * M + m], b = basis[m * nn + k];
            re += c.x * b.x - c.y * b.y, im += c.x * b.y + c.y * b.x;
        }
        L[e] = make_double2(re, im);
    }
}

// ---- magnus_42 (exp/magnus.rs:28-83) with the commutator computed densely per system ----------------------------------------------
// For generators that are NOT closed under commutation on the shared basis: L(t) = B_0 + sum_m g_m(t) B_m is assembled per system
// in shared memory at the two Gauss nodes, [L0, L1] is two tensor-core products, Omega = (L0 + L1) dt/2 - sqrt(3)/12 dt^2 [L0, L1]
// overwrites L0 (and the 2nd-order W1 = (L0 + L1) dt/2 overwrites L1 when the embedded error is wanted), and exp(Omega) x is the
// scaled Taylor series applied by matrix-vector products from shared memory. One CTA per system at a time.
template <int NB, class GEN>
__global__ void __launch_bounds__(32 * NB) magnus_dense_kernel(const __grid_constant__ ExpKP kp, const double2* __restrict__ basis /* [M][n][n] */,
                                                               double2* __restrict__ psi, const double* __restrict__ gp, const CtlArrays ca, EvSlot* __restrict__ ev) {
    using G = DenseGeo<NB>;
    constexpr int N = G::N, LD = G::LD, MMAX = VO_EXP_MAX_M;
    extern __shared__ __align__(16) unsigned char dsm[];
    double* l0_r = reinterpret_cast<double*>(dsm);
    double* l0_i = l0_r + N * LD;
    double* l1_r = l0_i + N * LD;
    double* l1_i = l1_r + N * LD;
    double* red = l1_i + N * LD;                         // [N + 2]
    double2* vx = reinterpret_cast<double2*>(red + N + 2);  // x0, acc, term, tmp: 4 vectors of N
    double* sc = reinterpret_cast<double*>(vx + 4 * N);  // scalars: g0[M], g1[M], dt, theta..., event
    int* si = reinterpret_cast<int*>(sc + 2 * MMAX + 8);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, row = 8 * w + (lane >> 2);
    const int M = kp.M;
    unsigned c_step = 0, c_chkpt = 0, c_rej = 0, c_end = 0, c_stuck = 0;
    for (int64_t sys = blockIdx.x; sys < kp.N; sys += gridDim.x) {
        __syncthreads();
        // ---- control: step_size_of (ode.rs:165-176), generator coefficients at the two nodes (magnus.rs:42-52)
        if (threadIdx.x == 0) {
            double dt = 0.0;
            const uint32_t word = ca.word[sys];
            const double t = ca.t[sys], h = ca.h[sys];
            const int evk = exp_event_kind(kp, word, t, h, dt);
            if (evk == VO_EV_STEP) {
                const double c_mid = 0.288675134594812882254574390251;
                const double mid_t = t + dt * 0.5;
                double g0[MMAX], g1[MMAX];
                GEN::template coef<MMAX>(gp + sys * (kp.M_gen - 1) * 3, kp.M_gen, mid_t - c_mid * dt, g0);
                GEN::template coef<MMAX>(gp + sys * (kp.M_gen - 1) * 3, kp.M_gen, mid_t + c_mid * dt, g1);
                for (int m = 0; m < MMAX; ++m) sc[m] = g0[m], sc[MMAX + m] = g1[m];
            }
            si[0] = evk, si[1] = (evk == VO_EV_CHKPT || evk == VO_EV_END) ? (int)(word & VO_WORD_TGT_MASK) : -1, sc[2 * MMAX] = dt;
        }
        __syncthreads();
        int evk = si[0];
        const double dt = sc[2 * MMAX];
        if (evk == VO_EV_STEP) {
            // ---- assemble L0, L1 (planar, padded) from the shared basis
            for (int e = threadIdx.x; e < N * N; e += G::THREADS) {
                double r0 = 0.0, i0 = 0.0, r1 = 0.0, i1 = 0.0;
                for (int m = 0; m < M; ++m) {
                    const double2 b = basis[(size_t)m * N * N + e];
                    r0 += sc[m] * b.x, i0 += sc[m] * b.y, r1 += sc[MMAX + m] * b.x, i1 += sc[MMAX + m] * b.y;
                }
                const int o = (e / N) * LD + e % N;
                l0_r[o] = r0, l0_i[o] = i0, l1_r[o] = r1, l1_i[o] = i1;
            }
            __syncthreads();
            // ---- commutator(l0, l1) (magnus.rs:55) on the tensor cores
            double cr[NB][2], ci[NB][2];
#pragma unroll
            for (int j = 0; j < NB; ++j) cr[j][0] = cr[j][1] = ci[j][0] = ci[j][1] = 0.0;
            zgemm_acc<NB>(l0_r, l0_i, l1_r, l1_i, LD, false, cr, ci);
            zgemm_acc<NB>(l1_r, l1_i, l0_r, l0_i, LD, true, cr, ci);
            // ---- w1 = (l0 + l1) b1, w2 = [l0, l1] b2, Omega = w1 + w2 (magnus.rs:56-66)
            const double b1 = dt * 0.5, b2 = dt * dt * -0.144337567297406441127287195125;
            double wr[NB][2], wi[NB][2];
#pragma unroll
            for (int j = 0; j < NB; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int o = row * LD + 8 * j + 2 * (lane & 3) + q;
                    wr[j][q] = (l0_r[o] + l1_r[o]) * b1, wi[j][q] = (l0_i[o] + l1_i[o]) * b1;
                    cr[j][q] = wr[j][q] + cr[j][q] * b2, ci[j][q] = wi[j][q] + ci[j][q] * b2;
                }
            __syncthreads();  // every warp is done with L0 / L1 as operands
            frag_to_smem<NB>(cr, ci, l0_r, l0_i);
            frag_to_smem<NB>(wr, wi, l1_r, l1_i);
            for (int c = threadIdx.x; c < N; c += G::THREADS) vx[c] = psi[sys * N + c];
            // ---- x <- exp(Omega) x0 (and exp(W1) x0 for the embedded error, magnus.rs:76-79): scaled Taylor series, matrix-vector
            // products from shared memory; thread (r, q4) sums columns q4, q4 + 4, ... of row r
            const int nexp = kp.want_err ? 2 : 1;
            for (int e = 0; e < nexp; ++e) {
                const double* m_r = e == 0 ? l0_r : l1_r;
                const double* m_i = e == 0 ? l0_i : l1_i;
                const double theta = dense_norm1<NB>(m_r, m_i, red);
                if (threadIdx.x == 0) taylor_plan(theta, kp.taylor_deg, &si[2], &si[3]);
                __syncthreads();
                const int sq = si[2], deg = si[3];
                const double inv_sq = 1.0 / sq;
                double2* acc = vx + N * (1 + e);  // acc of exponential e: vx[N..2N) = xf, vx[2N..3N) = the embedded solution
                double2* term = vx + 3 * N;
                for (int c = threadIdx.x; c < N; c += G::THREADS) acc[c] = vx[c];
                for (int rep = 0; rep < sq; ++rep) {
                    __syncthreads();
                    for (int c = threadIdx.x; c < N; c += G::THREADS) term[c] = acc[c];
                    for (int k = 1; k <= deg; ++k) {
                        __syncthreads();
                        const double f = inv_sq / k;
                        double2 out[(N + G::THREADS / 4 - 1) / (G::THREADS / 4)];
                        int no = 0;
                        for (int r = threadIdx.x >> 2; r < N; r += G::THREADS / 4, ++no) {
                            double sr = 0.0, sim = 0.0;
                            for (int c = threadIdx.x & 3; c < N; c += 4) {
                                const double ur = m_r[r * LD + c], ui = m_i[r * LD + c];
                                const double2 v = term[c];
                                sr += ur * v.x - ui * v.y, sim += ur * v.y + ui * v.x;
                            }
                            sr += __shfl_xor_sync(0xffffffffu, sr, 1), sim += __shfl_xor_sync(0xffffffffu, sim, 1);
                            sr += __shfl_xor_sync(0xffffffffu, sr, 2), sim += __shfl_xor_sync(0xffffffffu, sim, 2);
                            out[no] = make_double2(sr * f, sim * f);
                        }
                        __syncthreads();  // every thread has read the old term
                        no = 0;
                        for (int r = threadIdx.x >> 2; r < N; r += G::THREADS / 4, ++no)
                            if ((threadIdx.x & 3) == 0) term[r] = out[no], acc[r] = make_double2(acc[r].x + out[no].x, acc[r].y + out[no].y);
                    }
                }
                __syncthreads();
            }
        } else if (const int64_t orow = si[1] >= 0 ? exp_out_row(kp, si[1], sys) : -1; orow >= 0) {  // Chkpt / End: the state current() shows
            if (kp.snap)
                for (int c = threadIdx.x; c < N; c += G::THREADS) kp.snap[orow * N + c] = psi[sys * N + c];
            if (kp.n_obs)  // one row in flight: more would push the kernel's step path into spills at n = 8 to 24
                exp_expect_warp<1>(kp.obs, kp.n_obs, N, psi + sys * N, w, NB, kp.obs_out + orow * kp.n_obs);
        }
        // ---- error norm, handle_step_adaptive (ode.rs:311-334), apply_step (ode.rs:402-428), masked commit
        if (evk == VO_EV_STEP && kp.adaptive) {
            double v = 0.0;
            for (int c = threadIdx.x; c < N; c += G::THREADS) {
                const double er = vx[2 * N + c].x - vx[N + c].x, ei = vx[2 * N + c].y - vx[N + c].y;
                v += er * er + ei * ei;
            }
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[w] = v;
        }
        __syncthreads();
        if (threadIdx.x == 0 && evk != 255) {
            const uint32_t word = ca.word[sys];
            int tgt = (int)(word & VO_WORD_TGT_MASK);
            uint32_t status = word >> VO_WORD_STATUS_SHIFT;
            if (evk == VO_EV_STEP) {
                const double h = ca.h[sys];
                if (kp.adaptive) {
                    double nn = 0.0;
                    for (int ww = 0; ww < NB; ++ww) nn += red[ww];
                    const double dxn = kp.literal_norm ? ca.dx_norm[sys] : sqrt(nn);
                    const double f = kp.rtol / dxn;
                    const double fp_lim = at_most(at_least(step_size_mul<true>(kp.alpha, f, kp.pw, kp.pw_is_third), 0.3), 2.0);
                    const double new_h = at_most(at_least(fp_lim * h, kp.min_dt), kp.max_dt);
                    if (!(dxn == dxn)) status |= VO_TRAJ_NONFINITE;
                    if (f <= 1.0) {
                        evk = VO_EV_REJECT;
                        if (h <= kp.min_dt) status |= VO_TRAJ_STUCK, ++c_stuck;
                    }
                    ca.prev_h[sys] = h, ca.h[sys] = new_h, ca.dx_norm[sys] = dxn;
                }
                if (evk == VO_EV_STEP) ca.t[sys] += dt, ca.n_accept[sys] += 1, ++c_step;
                else ca.n_reject[sys] += 1, ++c_rej;
            } else {
                tgt += 1, ca.h[sys] = ca.prev_h[sys];
                if (evk == VO_EV_END) status |= VO_TRAJ_DONE, ++c_end;
                else ++c_chkpt;
            }
            const uint32_t nw = ((uint32_t)tgt & VO_WORD_TGT_MASK) | (status << VO_WORD_STATUS_SHIFT);
            if (nw != word) ca.word[sys] = nw;
            si[0] = evk;
        }
        __syncthreads();
        if (si[0] == VO_EV_STEP)
            for (int c = threadIdx.x; c < N; c += G::THREADS) psi[sys * N + c] = vx[N + c];
    }
    if (kp.count_events && threadIdx.x == 0) {
        EvSlot* slot = ev + (blockIdx.x % VO_EV_SLOTS);
        if (c_step) atomicAdd(&slot->n_step, (unsigned long long)c_step);
        if (c_chkpt) atomicAdd(&slot->n_chkpt, (unsigned long long)c_chkpt);
        if (c_rej) atomicAdd(&slot->n_reject, (unsigned long long)c_rej);
        if (c_end) atomicAdd(&slot->n_end, (unsigned long long)c_end);
        if (c_stuck) atomicAdd(&slot->n_stuck, (unsigned long long)c_stuck);
    }
}
