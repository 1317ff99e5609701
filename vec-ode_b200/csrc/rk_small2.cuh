// rk_small2.cuh — the register-resident kernels with TWO trajectories per thread (control kernel; fixed-step kernel below).
// Arithmetic per trajectory is that of the one-trajectory kernels of rk_small.cuh (same operations, same order), so results
// are bit-identical to them.
#pragma once
#include "rk_small.cuh"

#define VO_TILE2 256  // trajectories per CTA tile of both two-trajectory kernels

// rk_step (rk.rs:90-155) for U independent trajectories, interleaved statement by statement.
template <class RHS, int S, bool STRICT, int U>
__device__ __forceinline__ void rk_attempt_n(const TableauDev& tb, const double (&t)[U], const double (&dt)[U], const double (&x0)[U][RHS::D],
                                             const double (&p)[U][RHS::NP], double (&xf)[U][RHS::D], double (&xe)[U][RHS::D]) {
    using A = Ar<STRICT>;
    constexpr int D = RHS::D;
    double K[U][S][D], vlast[U][D];
#pragma unroll
    for (int u = 0; u < U; ++u) RHS::template eval<STRICT>(t[u], x0[u], K[u][0], p[u]);  // rk.rs:111
#pragma unroll
    for (int i = 1; i < S; ++i) {
        const double* row = &tb.ac[i * S];
        double xs[U][D];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            double v[D];
            combine_sum<STRICT, D, S>(row, i, K[u], v);              // rk.rs:121-122
            combine_finish<STRICT, D>(v, dt[u], x0[u], xs[u]);       // rk.rs:123-124
            if (i == S - 1) {
#pragma unroll
                for (int c = 0; c < D; ++c) vlast[u][c] = v[c];
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) RHS::template eval<STRICT>(A::add(t[u], A::mul(row[i], dt[u])), xs[u], K[u][i], p[u]);  // rk.rs:119, 127
    }
    // X_b (rk.rs:131-133, held in xe for the swap of rk.rs:142) and X_berr, the propagated solution. With the first-same-as-last
    // structure (TableauDev::reuse) the first S-1 terms of a combination are the last stage's sum: same operations, same order.
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (tb.reuse & 2) combine_tail<STRICT, D>(vlast[u], tb.b[S - 1], K[u][S - 1], dt[u], x0[u], xe[u]);
        else combine<STRICT, D, S>(tb.b, S, K[u], dt[u], x0[u], xe[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (tb.reuse & 1) combine_tail<STRICT, D>(vlast[u], tb.b_err[S - 1], K[u][S - 1], dt[u], x0[u], xf[u]);
        else combine<STRICT, D, S>(tb.b_err, S, K[u], dt[u], x0[u], xf[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
        for (int c = 0; c < D; ++c) xe[u][c] = A::sub(xe[u][c], xf[u][c]);  // x_err = X_b - X_berr (rk.rs:147)
}

// rk_step without the error branch's difference (lock-step fixed steps) for U independent trajectories sharing t and dt.
template <class RHS, int S, bool STRICT, int U>
__device__ __forceinline__ void rk_attempt_fixed_n(const TableauDev& tb, bool use_err, double t, double dt, const double (&x0)[U][RHS::D],
                                                   const double (&p)[U][RHS::NP], double (&xf)[U][RHS::D]) {
    using A = Ar<STRICT>;
    constexpr int D = RHS::D;
    double K[U][S][D], vlast[U][D];
#pragma unroll
    for (int u = 0; u < U; ++u) RHS::template eval<STRICT>(t, x0[u], K[u][0], p[u]);  // rk.rs:111
#pragma unroll
    for (int i = 1; i < S; ++i) {
        const double* row = &tb.ac[i * S];
        const double ti = A::add(t, A::mul(row[i], dt));  // rk.rs:119
        double xs[U][D];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            double v[D];
            combine_sum<STRICT, D, S>(row, i, K[u], v);          // rk.rs:121-122
            combine_finish<STRICT, D>(v, dt, x0[u], xs[u]);      // rk.rs:123-124
            if (i == S - 1) {
#pragma unroll
                for (int c = 0; c < D; ++c) vlast[u][c] = v[c];
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) RHS::template eval<STRICT>(ti, xs[u], K[u][i], p[u]);  // rk.rs:127
    }
    // the propagated state: X_berr when the error branch runs (rk.rs:136-146), else X_b (rk.rs:131-133)
    const double* w = use_err ? tb.b_err : tb.b;
    const bool reuse = (tb.reuse & (use_err ? 1 : 2)) != 0;  // first S-1 weights == the last row of the tableau: start from the last stage's sum
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (reuse) combine_tail<STRICT, D>(vlast[u], w[S - 1], K[u][S - 1], dt, x0[u], xf[u]);
        else combine<STRICT, D, S>(w, S, K[u], dt, x0[u], xf[u]);
    }
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

// ---- control kernel, two trajectories per thread, warp-autonomous staging -----------------------------------------------
// rk_ctl_staged_kernel (rk_small.cuh) is bound by the FP64 pipe and by instruction issue, not by HBM: an adaptive
// DoPri5 attempt of a 2-component system is one long dependent chain with ILP 2. Giving every thread two independent
// trajectories doubles the ILP, and everything that is per-thread rather than per-trajectory — tableau coefficient
// loads into uniform registers, loop overhead, address arithmetic shared by the pair — is paid once per two attempts.
// Tile = VO_TILE2 trajectories per CTA iteration; every WARP stages its own 64 of them (lane l owns trajectories 2l and
// 2l+1): the rows arrive through a cp.async pipeline per warp (16 bytes per lane per row), so there is no elected thread,
// no mbarrier and no __syncthreads() in the tile loop; a lane reads its two trajectories with ONE 128-bit shared load per
// row and writes them back with 128-bit stores when both of its trajectories commit the same way.
// Compiled for the common adaptive configuration (step_adaptive, error estimate present, L2 norm, one event per launch);
// a thread whose pair does not both take a Step, and the ragged tail of the ensemble, go through ctl_lane of rk_small.cuh.
template <class RHS, int S, bool STRICT>
__global__ void __launch_bounds__(128, 4) rk_ctl2w_staged_kernel(double* __restrict__ x, int64_t N, const __grid_constant__ TableauDev tb,
                                                                 const __grid_constant__ RhsParams rp, const CtlArrays ca,
                                                                 const __grid_constant__ CtlShared cs, EvSlot* __restrict__ ev, const pipe::Chain ch) {
    constexpr int D = RHS::D, NP = RHS::NP, T = VO_TILE2, U = 2, WT = 64, NST = VO_STAGES;
    extern __shared__ __align__(128) double sbuf[];  // [4 warps][NST][nrows x 64 doubles, then 3 x 64 words]
    int nrows = D + 2;  // state, t, h
#pragma unroll
    for (int q = 0; q < NP; ++q) nrows += rp.per_traj[q] ? 1 : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t stage_bytes = (uint32_t)nrows * WT * 8u + 3u * WT * 4u;
    unsigned char* wbase = reinterpret_cast<unsigned char*>(sbuf) + (size_t)warp * NST * stage_bytes;
    const int64_t n_full = N / T, G = gridDim.x, first = blockIdx.x;
    const int64_t my_count = first < n_full ? (n_full - first + G - 1) / G : 0;
    __shared__ double s_tl[VO_INLINE_TLIST];
    const TList tl = tlist_stage(cs, s_tl);
    unsigned c_step = 0, c_chkpt = 0, c_rej = 0, c_end = 0, c_stuck = 0;
    pipe::chain_enter(ch);
    auto issue = [&](int64_t k) {  // every lane; always commits a group so that the group count is uniform
        if (k < my_count) {
            const int64_t base = (first + k * G) * T + warp * WT;
            const uint32_t dst = (uint32_t)__cvta_generic_to_shared(wbase + (size_t)(k % NST) * stage_bytes) + 16u * lane;
            int r = 0;
#pragma unroll
            for (int c = 0; c < D; ++c) cp_async16(dst + 512u * (r++), x + c * N + base + 2 * lane);
            cp_async16(dst + 512u * (r++), ca.t + base + 2 * lane);
            cp_async16(dst + 512u * (r++), ca.h + base + 2 * lane);
#pragma unroll
            for (int q = 0; q < NP; ++q)
                if (rp.per_traj[q]) cp_async16(dst + 512u * (r++), rp.per_traj[q] + base + 2 * lane);
            const uint32_t wdst = dst + 512u * r;  // status word | accepted | rejected: 256 bytes each, 16 lanes per row
            if (lane < 16) {
                cp_async16(wdst, ca.word + base + 4 * lane);
                cp_async16(wdst + 512u, ca.n_reject + base + 4 * lane);
            } else {
                cp_async16(wdst, ca.n_accept + base + 4 * (lane - 16));  // lands at offset 256 + 16 (lane - 16)
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int64_t k = 0; k < NST - 1; ++k) issue(k);
    for (int64_t k = 0; k < my_count; ++k) {
        const int64_t i0 = (first + k * G) * T + warp * WT + 2 * lane;  // this lane's two trajectories: i0, i0 + 1
        __syncwarp();  // every lane is done with the buffer the next copies go to
        issue(k + NST - 1);
        asm volatile("cp.async.wait_group %0;" ::"n"(NST - 1) : "memory");
        __syncwarp();
        const unsigned char* stage = wbase + (size_t)(k % NST) * stage_bytes;
        double xc[U][D], p[U][NP], t[U], h[U];
        uint32_t word[U], n_acc[U], n_rej[U];
        {
            int r = 0;
            auto row2 = [&](double& a, double& b) {
                const double2 v = *reinterpret_cast<const double2*>(stage + 512 * (r++) + 16 * lane);
                a = v.x, b = v.y;
            };
#pragma unroll
            for (int c = 0; c < D; ++c) row2(xc[0][c], xc[1][c]);
            row2(t[0], t[1]);
            row2(h[0], h[1]);
#pragma unroll
            for (int q = 0; q < NP; ++q) {
                if (rp.per_traj[q]) row2(p[0][q], p[1][q]);
                else p[0][q] = p[1][q] = rp.shared[q];
            }
            const unsigned char* w = stage + 512 * r + 8 * lane;
            const uint2 a = *reinterpret_cast<const uint2*>(w), b = *reinterpret_cast<const uint2*>(w + 256), c2 = *reinterpret_cast<const uint2*>(w + 512);
            word[0] = a.x, word[1] = a.y, n_acc[0] = b.x, n_acc[1] = b.y, n_rej[0] = c2.x, n_rej[1] = c2.y;
        }
        bool live[U];
        bool pair = cs.k_events == 1;
#pragma unroll
        for (int u = 0; u < U; ++u) live[u] = !((word[u] >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE), pair = pair && live[u];
        double dt[U] = {0.0, 0.0}, t_tgt[U] = {0.0, 0.0};
        if (pair) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int tgt = (int)(word[u] & VO_WORD_TGT_MASK);
                if (tgt >= cs.n_tlist) {
                    pair = false;
                } else {
                    t_tgt[u] = tl.at(tgt);
                    const double rem = t_tgt[u] - t[u];  // step_size_of (ode.rs:165-176) + check_step (ode.rs:389-399)
                    if (fabs(rem) <= 2.220446049250313e-16) pair = false;
                    dt[u] = rem < h[u] ? rem : h[u];
                }
            }
        }
        if (pair) {
            double xf[U][D], xe[U][D];
            rk_attempt_n<RHS, S, STRICT, U>(tb, t, dt, xc, p, xf, xe);
            double dxn[U] = {0.0, 0.0}, new_h[U], acc[U];
            bool rej[U], nonfin[U];
#pragma unroll
            for (int u = 0; u < U; ++u) acc[u] = err_sumsq<STRICT, D>(xe[u]);
            controller_l2_n<STRICT, U>(acc, h, cs, cs.record_dx_norm != 0, dxn, new_h, rej, nonfin);  // handle_step_adaptive, ode.rs:311-334
            // apply_step (ode.rs:402-428) + masked write-back: 128-bit stores where both trajectories commit the same way
            if (!rej[0] && !rej[1]) {
#pragma unroll
                for (int c = 0; c < D; ++c) *reinterpret_cast<double2*>(x + c * N + i0) = make_double2(xf[0][c], xf[1][c]);
                *reinterpret_cast<double2*>(ca.t + i0) = make_double2(t[0] + dt[0], t[1] + dt[1]);  // advance, ode.rs:184-188
                *reinterpret_cast<uint2*>(ca.n_accept + i0) = make_uint2(n_acc[0] + 1, n_acc[1] + 1);
                c_step += 2;
            } else if (rej[0] && rej[1]) {
                *reinterpret_cast<uint2*>(ca.n_reject + i0) = make_uint2(n_rej[0] + 1, n_rej[1] + 1);
                c_rej += 2;
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (rej[u]) {
                        ca.n_reject[i0 + u] = n_rej[u] + 1, ++c_rej;
                    } else {
#pragma unroll
                        for (int c = 0; c < D; ++c) x[c * N + i0 + u] = xf[u][c];
                        ca.t[i0 + u] = t[u] + dt[u];
                        ca.n_accept[i0 + u] = n_acc[u] + 1, ++c_step;
                    }
                }
            }
            *reinterpret_cast<double2*>(ca.h + i0) = make_double2(new_h[0], new_h[1]);  // update_step_size, ode.rs:202-205
            if (!cs.lazy_prev_h) *reinterpret_cast<double2*>(ca.prev_h + i0) = make_double2(h[0], h[1]);
            if (cs.record_dx_norm) *reinterpret_cast<double2*>(ca.dx_norm + i0) = make_double2(dxn[0], dxn[1]);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                uint32_t status = word[u] >> VO_WORD_STATUS_SHIFT;
                if (nonfin[u]) status |= VO_TRAJ_NONFINITE;
                if (rej[u] && h[u] <= cs.min_dt) status |= VO_TRAJ_STUCK, ++c_stuck;
                // prev_h has one reader, the Chkpt / End branch (ode.rs:192-195): it reaches memory only if that is this trajectory's next event
                if (cs.lazy_prev_h && !rej[u] && fabs(t_tgt[u] - (t[u] + dt[u])) <= 2.220446049250313e-16) ca.prev_h[i0 + u] = h[u];
                const uint32_t nw = (word[u] & VO_WORD_TGT_MASK) | (status << VO_WORD_STATUS_SHIFT);
                if (nw != word[u]) ca.word[i0 + u] = nw;
            }
        } else {
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (live[u])
                    ctl_lane<RHS, S, STRICT, 1>(SoaAcc{x, N, ca, i0 + u}, tb, cs, tl, word[u], xc[u], p[u], t[u], h[u], n_acc[u], n_rej[u], c_step, c_chkpt, c_rej, c_end,
                                                c_stuck);
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    // ragged tail (N % tile trajectories): plain loads, last CTA, one trajectory at a time
    if (blockIdx.x == G - 1) {
        for (int64_t i = n_full * T + threadIdx.x; i < N; i += 128) {
            const uint32_t word = ca.word[i];
            if (!((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE)) {
                double xc[D], p[NP];
                lane_load<RHS>(x, N, rp, i, xc, p);
                ctl_lane<RHS, S, STRICT, 1>(SoaAcc{x, N, ca, i}, tb, cs, tl, word, xc, p, ca.t[i], ca.h[i], ca.n_accept[i], ca.n_reject[i], c_step, c_chkpt, c_rej, c_end,
                                            c_stuck);
            }
        }
    }
    ctl_count_events(cs, ev, c_step, c_chkpt, c_rej, c_end, c_stuck);
    pipe::chain_exit(ch);
}

// ---- lock-step fixed-step kernel, two trajectories per thread, warp-autonomous staging (as rk_ctl2w_staged_kernel) -------
// rk_fixed_staged_kernel spends more issue slots on what is per THREAD (tableau coefficients into uniform registers, tile
// addressing, barrier, loop) than on the ~70-100 FP64 operations of an RK4 step of a 3-component system, and at 10^6
// trajectories per launch that — not HBM — sets its time (an L2-resident ensemble runs no faster). Two trajectories per
// thread halve that overhead per trajectory and double the ILP.
template <class RHS, int S, bool STRICT>
__global__ void __launch_bounds__(128) rk_fixed2w_staged_kernel(double* __restrict__ x, int64_t N, const __grid_constant__ TableauDev tb,
                                                                const __grid_constant__ RhsParams rp, const __grid_constant__ StepList sl,
                                                                const pipe::Chain ch) {
    constexpr int D = RHS::D, NP = RHS::NP, T = VO_TILE2, U = 2, WT = 64, NST = VO_STAGES;
    extern __shared__ __align__(128) double sbuf[];  // [4 warps][NST][nrows x 64 doubles]
    int nrows = D;
#pragma unroll
    for (int q = 0; q < NP; ++q) nrows += rp.per_traj[q] ? 1 : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t stage_bytes = (uint32_t)nrows * WT * 8u;
    unsigned char* wbase = reinterpret_cast<unsigned char*>(sbuf) + (size_t)warp * NST * stage_bytes;
    const int64_t n_full = N / T, G = gridDim.x, first = blockIdx.x;
    const int64_t my_count = first < n_full ? (n_full - first + G - 1) / G : 0;
    pipe::chain_enter(ch);
    auto issue = [&](int64_t k) {
        if (k < my_count) {
            const int64_t base = (first + k * G) * T + warp * WT;
            const uint32_t dst = (uint32_t)__cvta_generic_to_shared(wbase + (size_t)(k % NST) * stage_bytes) + 16u * lane;
            int r = 0;
#pragma unroll
            for (int c = 0; c < D; ++c) cp_async16(dst + 512u * (r++), x + c * N + base + 2 * lane);
#pragma unroll
            for (int q = 0; q < NP; ++q)
                if (rp.per_traj[q]) cp_async16(dst + 512u * (r++), rp.per_traj[q] + base + 2 * lane);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int64_t k = 0; k < NST - 1; ++k) issue(k);
    for (int64_t k = 0; k < my_count; ++k) {
        const int64_t i0 = (first + k * G) * T + warp * WT + 2 * lane;
        __syncwarp();
        issue(k + NST - 1);
        asm volatile("cp.async.wait_group %0;" ::"n"(NST - 1) : "memory");
        __syncwarp();
        const unsigned char* stage = wbase + (size_t)(k % NST) * stage_bytes;
        double xc[U][D], p[U][NP];
        {
            int r = 0;
            auto row2 = [&](double& a, double& b) {
                const double2 v = *reinterpret_cast<const double2*>(stage + 512 * (r++) + 16 * lane);
                a = v.x, b = v.y;
            };
#pragma unroll
            for (int c = 0; c < D; ++c) row2(xc[0][c], xc[1][c]);
#pragma unroll
            for (int q = 0; q < NP; ++q) {
                if (rp.per_traj[q]) row2(p[0][q], p[1][q]);
                else p[0][q] = p[1][q] = rp.shared[q];
            }
        }
        for (int e = 0; e < sl.n; ++e) {
            double xf[U][D];
            rk_attempt_fixed_n<RHS, S, STRICT, U>(tb, sl.use_err != 0, sl.t[e], sl.dt[e], xc, p, xf);
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int c = 0; c < D; ++c) xc[u][c] = xf[u][c];
        }
#pragma unroll
        for (int c = 0; c < D; ++c) *reinterpret_cast<double2*>(x + c * N + i0) = make_double2(xc[0][c], xc[1][c]);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    // ragged tail (N % 256 trajectories): plain loads, last CTA, one trajectory at a time
    if (blockIdx.x == G - 1) {
        for (int64_t i = n_full * T + threadIdx.x; i < N; i += 128) {
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
    }
    pipe::chain_exit(ch);
}
