// exp.cu — exponential integrators (src/exp) for ensembles of dense complex systems on a shared operator basis.
//
// What the reference fixes is the SCHEME: midpoint (exp/magnus.rs:10-26), 4th-order Magnus with one commutator
// (exp/magnus.rs:28-83) and the commutator-free CFM4 of cfm_general (exp/cfm.rs:43-100 with the tables of
// dat/mod.rs:4, 67-74), each wrapped in the ODEData / ODEAdaptiveData state machine (base/ode.rs). What it leaves to the
// user is the operator algebra behind ExponentialSplit / Commutator (exp/mod.rs:11-54): lin_zero, exp, map_exp,
// commutator, norm. This file supplies that algebra for L_i = sum_m coef[i][m] * B_m with M complex n x n matrices B_m
// shared by the ensemble:
//   * an operator `L` is its M complex coefficients, so LinearCombination on L is arithmetic on coefficients;
//   * exp(L) is lazy (U = L) and map_exp(U, x) applies the scaled Taylor series of exp(L) to x without forming U
//     (each U is used exactly once per step in all three schemes);
//   * commutator(La, Lb) is expanded on the basis through a structure tensor supplied by the caller.
// Per Taylor term every system of a tile needs B_m x for all m: that is a GEMM  [n x n] x [n x TB]  with the basis as the
// shared operand. It runs on the FP64 tensor cores (mma.sync m8n8k4 DMMA; tcgen05 has no f64 kind): the basis lives in
// shared memory in A-fragment order for the whole kernel, the Taylor term of the tile is re-published to shared memory
// once per term in B-fragment-friendly layout, accumulators and the running sum stay in registers.
// Systems of 1 <= n <= 8 levels take exp_small_kernel (exp_small_kernels.cuh) instead: one system per thread in FP64 registers,
// the basis a kernel parameter, a Taylor plan per system, and several events per launch inside vo_exp_run.
#include <algorithm>
#include <cmath>
#include <complex>
#include <cstring>
#include <type_traits>
#include <vector>

#include "exp_dense_kernels.cuh"
#include "exp_small_kernels.cuh"

// Events per launch of exp_small_kernel inside vo_exp_run (a run never fuses past its readback batch of at most 16 calls). Measured
// against one event per launch in DESIGN.md §2.3; tools/build_variant.sh rebuilds with another value for such comparisons.
#ifndef VO_EXP_SMALL_FUSE
#define VO_EXP_SMALL_FUSE 16
#endif

// exp_small.cu: exp_small_kernel<n, M, GenCos> for the split's shape, one thread per system
unsigned exp_small_grid(vo_ctx c, int64_t N);
int32_t launch_exp_small(vo_ctx c, int n, int M, const ExpKP& kp, const double* basis, double2* psi, double2* psi_out, const double* gp, const double2* coef_in,
                         const CtlArrays& ca, EvSlot* ev);

// sort_keys.cu
size_t vo_sort_pairs_tmp_bytes(int n);
cudaError_t vo_sort_pairs(void* tmp, size_t tmp_bytes, const float* key_in, float* key_out, const int* idx_in, int* idx_out, int n, cudaStream_t stream);


struct vo_split_s {
    vo_ctx ctx = nullptr;
    int n = 0, M = 0;
    double* frag_dev = nullptr;  // [M][2 planes][n/8 row blocks][n/4 k-steps][32 lanes] (n >= 16)
    std::vector<double> small_basis;  // n <= 8: the basis [M][n][n] complex interleaved, exp_small_kernel's SmallBasis parameter
    double norm1[VO_EXP_MAX_M];  // induced 1-norm of each basis matrix
    double cs[VO_EXP_MAX_M * VO_EXP_MAX_M * VO_EXP_MAX_M];
    bool has_cs = false;
    int taylor_deg = 0;
    double2* basis_dev = nullptr;  // [M][n][n] row-major interleaved: what the dense kernels (exp_dense_kernels.cuh) assemble operators from
    int kind = 0;                  // 0: shared-basis split (operators are coefficient vectors); 1: dense split (every system owns its n x n operators)
    int64_t N = 0;                 // dense split: number of systems
};

struct vo_expsolver_s {
    vo_ctx ctx = nullptr;
    vo_split sp = nullptr;
    int scheme = 0, M_gen = 0;
    int64_t N = 0;
    double t0 = 0, tf = 0, h_init = 0;
    double2* psi = nullptr;   // [N][n]
    double2* psi0 = nullptr;  // copy of the initial state (reset)
    double* gp = nullptr;     // [N][M_gen-1][3]
    CtlArrays ca{};
    EvSlot* ev_dev = nullptr;
    EvSlot* ev_host = nullptr;
    EvSlot ev_seen{};
    int64_t n_done = 0;
    std::vector<double> t_list;   // ODEData.t_list (ode.rs:89): [t0, tf] (ode.rs:144) unless vo_exp_set_t_list
    double* t_list_dev = nullptr;  // device copy of a list longer than VO_INLINE_TLIST
    double2* snap = nullptr;       // [t_list.size()][N][n] in the caller's order (vo_exp_enable_snapshots), else NULL
    int n_obs = 0;                 // vo_exp_set_observables: K operators, 0 = off
    double2* obs = nullptr;        // [n_obs][n][n] row-major
    double2* obs_out = nullptr;    // [t_list.size()][N][n_obs] expectation values in the caller's order
    bool stepped = false;          // an event has run since creation or the last vo_exp_reset: the list is fixed until the next reset
    bool want_err = true;  // alph_err / x_err present (exp/cfm.rs:157-161)
    unsigned split_mask = 1u;  // VO_EXP_SPLIT_MIDPOINT: which basis matrices form split A (default: B_0)
    double atol = 1.0e-6, rtol = 1.0e-4, alpha = 0.9, pw = 1.0 / 3.0, min_dt = 1.0e-6, max_dt = 1.0;
    int64_t* perm = nullptr;     // vo_exp_set_order: device slot j holds the caller's system perm[j] (device copy)
    std::vector<int64_t> perm_host;
    double2* stage = nullptr;    // [N][n] staging for the reordering copies
    // dynamic grouping (vo_exp_set_dynamic_grouping): before every event the systems are sorted by the 1-norm bound of their generator
    // at the coming step, and the kernel takes its tiles in that order (a tile runs the Taylor degree of its largest theta)
    int dynamic_group = 0;
    float *key_in = nullptr, *key_out = nullptr;
    int *idx_in = nullptr, *idx_out = nullptr;
    void* sort_tmp = nullptr;
    int* tile_ctr = nullptr;  // tile counter of the kernel's largest-theta-first schedule, zeroed before every launch
    size_t sort_tmp_bytes = 0;
    int literal_norm = 0;        // vo_exp_set_literal_norm: MagnusExpLinearSolver::norm as written (magnus.rs:274-276)
    int applied_comm = 0;        // vo_exp_set_applied_commutator: magnus_42's commutator applied by products inside the Taylor series, never formed
    int dense_comm = 0;          // vo_exp_set_dense_commutator: magnus_42 forms [L0, L1] densely per system (no structure tensor needed)
    void* gen_module = nullptr;  // vo_exp_set_generator: run-time compiled exp_step_kernel with the user's generator
    void* gen_fn = nullptr;
    std::string gen_body, norm_src;  // sources of the run-time compiled kernel: the user's generator ("" = the cosine family) and norm ("" = 2-norm)
    // commutator-free schemes as tables (cfm_general's c / alpha / alph_err, exp/cfm.rs:43-53; split_cfm's rho / sigma)
    int n_nodes = 0, n_rows = 0, n_rows_err = 0;
    double tab_c[VO_EXP_MAX_NODES] = {};
    double tab_alpha[VO_EXP_MAX_ROWS * VO_EXP_MAX_NODES] = {};
    double tab_alpha_err[VO_EXP_MAX_ERR * VO_EXP_MAX_NODES] = {};
    unsigned char row_split[VO_EXP_MAX_ROWS] = {};
};

// src/dat/mod.rs:4, 67-80 (same literals as the reference)
static const double C_GAUSS_LEGENDRE_4[2] = {0.21132486540518711775, 0.78867513459481288225};
static const double CFM_R2_J1_GL[2] = {0.5, 0.5};
static const double CFM_R4_J2_GL[4] = {0.53867513459481288225, -0.038675134594812882255, -0.038675134594812882255, 0.53867513459481288225};
static const double BLANES17_R4_J4[12] = {0.2463347584748155,  -0.0469610812011527, 0.0119511881315244,  0.0622500005170514, 0.2691833034233750,  -0.0427581693456134,
                                          -0.0427581693456134, 0.2691833034233750,  0.0622500005170514,  0.0119511881315244, -0.0469610812011527, 0.2463347584748155};

static int32_t exp_store_tables(vo_expsolver_s* s, const double* c, int k, const double* alpha, int rows, const double* alpha_err, int rows_err) {
    if (!c || !alpha || k < 1 || k > VO_EXP_MAX_NODES || rows < 1 || rows > VO_EXP_MAX_ROWS || rows_err < 0 || rows_err > VO_EXP_MAX_ERR || (rows_err > 0 && !alpha_err))
        return vo_fail(s->ctx, VO_ERR_SHAPE, "split_cfm: Incompatible array dimensions");  // the reference's panic message (cfm.rs:63, 86)
    if (rows_err > rows) return vo_fail(s->ctx, VO_ERR_SHAPE, "split_cfm: Incompatible array dimensions for alph_err");  // cfm.rs:85-87
    s->n_nodes = k, s->n_rows = rows, s->n_rows_err = rows_err;
    std::memset(s->tab_alpha, 0, sizeof s->tab_alpha), std::memset(s->tab_alpha_err, 0, sizeof s->tab_alpha_err), std::memset(s->row_split, 0, sizeof s->row_split);
    for (int q = 0; q < k; ++q) s->tab_c[q] = c[q];
    for (int e = 0; e < rows; ++e)
        for (int q = 0; q < k; ++q) s->tab_alpha[e * VO_EXP_MAX_NODES + q] = alpha[e * k + q];
    for (int e = 0; e < rows_err; ++e)
        for (int q = 0; q < k; ++q) s->tab_alpha_err[e * VO_EXP_MAX_NODES + q] = alpha_err[e * k + q];
    return VO_OK;
}

namespace {


// NormedExponentialSplit::norm (exp/mod.rs:37-45): 2-norm of every state, one warp per system
__global__ void exp_norm_kernel(const double2* __restrict__ psi, int n, int64_t N, double* __restrict__ out) {
    const int64_t sys = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (sys >= N) return;
    double acc = 0.0;
    for (int r = threadIdx.x & 31; r < n; r += 32) {
        const double2 v = psi[sys * n + r];
        acc += v.x * v.x + v.y * v.y;
    }
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) out[sys] = sqrt(acc);
}

// rows of n complex numbers: dst[j] = src[perm[j]] (gather) or dst[perm[j]] = src[j] (scatter); one warp per row
__global__ void exp_reorder_kernel(const double2* __restrict__ src, double2* __restrict__ dst, const int64_t* __restrict__ perm, int n, int64_t N, int scatter) {
    const int64_t j = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= N) return;
    const int64_t pj = perm[j];
    const double2* s = src + (scatter ? j : pj) * n;
    double2* d = dst + (scatter ? pj : j) * n;
    for (int r = threadIdx.x & 31; r < n; r += 32) d[r] = s[r];
}

__global__ void exp_ctl_fill_kernel(CtlArrays ca, int64_t N, double t, double h) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    ca.t[i] = t, ca.h[i] = h, ca.prev_h[i] = h, ca.dx_norm[i] = 0.0;
    ca.n_accept[i] = 0, ca.n_reject[i] = 0, ca.word[i] = 0;
}

template <int NDIM, int M, int TB>
int32_t launch_exp(vo_ctx c, const ExpKP& kp, const double* frag, double2* psi, double2* psi_out, const double* gp, const double2* coef_in,
                   const CtlArrays& ca, EvSlot* ev, const int* order, int* tile_ctr) {
    using G = Geo<NDIM, M, TB>;
    auto k = exp_step_kernel<NDIM, M, TB, GenCos>;
    if (vo_ensure_smem_attr(c->device, (const void*)k, G::SMEM) != cudaSuccess) return vo_fail(c, VO_ERR_CUDA, "exp: shared-memory carve-out rejected");
    const int64_t tiles = ceil_div(kp.N, TB);
    const unsigned grid = (unsigned)std::min<int64_t>(tiles, c->sm_count);
    k<<<grid, G::THREADS, G::SMEM, c->stream>>>(kp, frag, psi, psi_out, gp, coef_in, ca, ev, order, tile_ctr);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

// launch geometry of exp_step_kernel<n, M, 16, *> for a run-time compiled instance
// Shapes of the lazy shared-basis split that are compiled in: (n, M) with the whole basis (M n^2 complex) resident in one SM's
// shared memory next to the term buffers. A run-time compiled generator or norm (nvrtc_rhs.cu) takes the same list.
#define VO_EXP_SHAPES(X) \
    X(64, 1) X(64, 2) X(64, 3) X(48, 2) X(48, 3) X(40, 2) X(32, 1) X(32, 2) X(32, 3) X(32, 4) X(24, 2) X(24, 3) X(16, 1) X(16, 2) X(16, 3) X(16, 4)

bool exp_geometry(int n, int M, unsigned* threads, size_t* smem) {
    if (n >= 1 && n <= VO_EXP_SMALL_MAX_N && M >= 1 && M <= VO_EXP_MAX_M) {  // exp_small_kernel
        *threads = VO_EXP_SMALL_THREADS, *smem = 0;
        return true;
    }
#define VO_EXP_GEO(NDIM, MM) \
    if (n == NDIM && M == MM) { *threads = Geo<NDIM, MM, 16>::THREADS, *smem = Geo<NDIM, MM, 16>::SMEM; return true; }
    VO_EXP_SHAPES(VO_EXP_GEO)
#undef VO_EXP_GEO
    return false;
}

int32_t dispatch_exp(vo_split sp, const ExpKP& kp, double2* psi, double2* psi_out, const double* gp, const double2* coef_in, const CtlArrays& ca, EvSlot* ev,
                     void* custom_fn = nullptr, const int* order = nullptr, int* tile_ctr = nullptr) {
    vo_ctx c = sp->ctx;
    if (sp->n <= VO_EXP_SMALL_MAX_N) {  // systems of 1 to 8 levels: exp_small_kernel (a per-system plan: `order` has nothing to group)
        if (custom_fn) {
            ExpKP kpc = kp;
            CtlArrays cac = ca;
            void* args[] = {&kpc, const_cast<double*>(sp->small_basis.data()), &psi, &psi_out, &gp, &coef_in, &cac, &ev};
            int32_t r = rtc_exp_launch(c, custom_fn, exp_small_grid(c, kp.N), VO_EXP_SMALL_THREADS, 0, args);
            if (r != VO_OK) return r;
            VO_CHECK_LAUNCH(c);
            return VO_OK;
        }
        return launch_exp_small(c, sp->n, sp->M, kp, sp->small_basis.data(), psi, psi_out, gp, coef_in, ca, ev);
    }
    if (custom_fn) {  // the user's generator: same kernel, compiled at run time
        unsigned threads = 0;
        size_t smem = 0;
        if (!exp_geometry(sp->n, sp->M, &threads, &smem)) return vo_fail(c, VO_ERR_UNSUPPORTED, "exp: unsupported shape");
        ExpKP kpc = kp;
        const double* frag = sp->frag_dev;
        CtlArrays cac = ca;
        void* args[] = {&kpc, &frag, &psi, &psi_out, &gp, &coef_in, &cac, &ev, &order, &tile_ctr};
        const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(kp.N, 16), c->sm_count);
        int32_t r = rtc_exp_launch(c, custom_fn, grid, threads, smem, args);
        if (r != VO_OK) return r;
        VO_CHECK_LAUNCH(c);
        return VO_OK;
    }
#define VO_EXP_CASE(NDIM, MM) \
    if (sp->n == NDIM && sp->M == MM) return launch_exp<NDIM, MM, 16>(c, kp, sp->frag_dev, psi, psi_out, gp, coef_in, ca, ev, order, tile_ctr);
    VO_EXP_SHAPES(VO_EXP_CASE)
#undef VO_EXP_CASE
    return vo_fail(c, VO_ERR_UNSUPPORTED, "exp: the shared-basis split is compiled for 1 <= n <= 8 with M <= 4, n in {16, 32} with M <= 4, n in {24, 48} with M in {2, 3}, (40, 2) and n = 64 with M <= 3 "
                                          "(the whole basis stays in one SM's shared memory); other shapes: the dense split (vo_split_dense_create)");
}

ExpKP make_kp(const vo_split_s* sp, int mode) {
    ExpKP kp;
    std::memset(&kp, 0, sizeof kp);
    kp.n = sp->n, kp.M = sp->M, kp.mode = mode, kp.taylor_deg = sp->taylor_deg, kp.n_events = 1;
    std::memcpy(kp.norm1, sp->norm1, sizeof kp.norm1);
    for (int a = 0; a < sp->M; ++a)
        for (int b = 0; b < sp->M; ++b)
            for (int cc = 0; cc < sp->M; ++cc) kp.cs[(a * sp->M + b) * sp->M + cc] = sp->has_cs ? sp->cs[(a * sp->M + b) * sp->M + cc] : 0.0;
    return kp;
}

// ---- dense operators (exp_dense_kernels.cuh) --------------------------------------------------------------------------------------
template <class K> int32_t dense_grid(vo_ctx c, K kernel, int threads, size_t smem, int64_t N, unsigned* grid) {
    if (vo_ensure_smem_attr(c->device, (const void*)kernel, smem) != cudaSuccess) return vo_fail(c, VO_ERR_CUDA, "dense split: shared-memory carve-out rejected");
    int bps = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kernel, threads, smem) != cudaSuccess || bps < 1) bps = 1;
    *grid = (unsigned)std::min<int64_t>(N, (int64_t)c->sm_count * bps);
    return VO_OK;
}

#define VO_DENSE_DISPATCH(nb, CALL)                                  \
    switch (nb) {                                                    \
        case 1: CALL(1) break;                                       \
        case 2: CALL(2) break;                                       \
        case 3: CALL(3) break;                                       \
        case 4: CALL(4) break;                                       \
        case 5: CALL(5) break;                                       \
        case 6: CALL(6) break;                                       \
        case 7: CALL(7) break;                                       \
        case 8: CALL(8) break;                                       \
        default: return vo_fail(c, VO_ERR_UNSUPPORTED, "dense split: n must be a multiple of 8, 8 <= n <= 64"); \
    }

int32_t launch_magnus_dense(vo_expsolver_s* s, const ExpKP& kp) {
    vo_ctx c = s->ctx;
    if (s->gen_fn) return vo_fail(c, VO_ERR_UNSUPPORTED, "vo_exp_set_dense_commutator: not available together with a run-time compiled generator");
    const int nb = s->sp->n / 8;
#define VO_CALL(NB)                                                                                                                        \
    {                                                                                                                                      \
        using G = DenseGeo<NB>;                                                                                                            \
        auto k = magnus_dense_kernel<NB, GenCos>;                                                                                          \
        const size_t smem = 2 * G::MAT + (G::N + 2) * sizeof(double) + 4 * G::N * sizeof(double2) + (2 * VO_EXP_MAX_M + 8) * sizeof(double) + 16 * sizeof(int); \
        unsigned grid = 0;                                                                                                                 \
        int32_t r = dense_grid(c, k, G::THREADS, smem, kp.N, &grid);                                                                       \
        if (r != VO_OK) return r;                                                                                                          \
        k<<<grid, G::THREADS, smem, c->stream>>>(kp, s->sp->basis_dev, s->psi, s->gp, s->ca, s->ev_dev);                                   \
    }
    VO_DENSE_DISPATCH(nb, VO_CALL)
#undef VO_CALL
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

int32_t exp_ev_read(vo_expsolver_s* s, EvSlot* out) {
    vo_ctx c = s->ctx;
    VO_CUDA(c, vo_small_readback(c, s->ev_host, s->ev_dev, sizeof(EvSlot) * VO_EV_SLOTS));  // not a copy: see ctx.cu
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    EvSlot tot;
    std::memset(&tot, 0, sizeof tot);
    for (int i = 0; i < VO_EV_SLOTS; ++i)
        tot.n_step += s->ev_host[i].n_step, tot.n_chkpt += s->ev_host[i].n_chkpt, tot.n_reject += s->ev_host[i].n_reject, tot.n_end += s->ev_host[i].n_end,
            tot.n_stuck += s->ev_host[i].n_stuck;
    out->n_step = tot.n_step - s->ev_seen.n_step, out->n_chkpt = tot.n_chkpt - s->ev_seen.n_chkpt, out->n_reject = tot.n_reject - s->ev_seen.n_reject;
    out->n_end = tot.n_end - s->ev_seen.n_end, out->n_stuck = tot.n_stuck - s->ev_seen.n_stuck;
    s->ev_seen = tot;
    return VO_OK;
}

// Sort key of the dynamic grouping: the bound sum_m |g_m(t + dt/2)| ||B_m||_1 dt of the 1-norm of this system's exponent at its coming
// step (the mid-point of the step stands in for the scheme's nodes: the key only has to ORDER systems, the kernel plans with the
// exact exponents). Trajectories that are done sort first, together.
__global__ void exp_group_key_kernel(const ExpKP kp, const double* __restrict__ gp, const CtlArrays ca, int64_t N, float* __restrict__ key, int* __restrict__ idx) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    idx[i] = (int)i;
    const uint32_t word = ca.word[i];
    if ((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE) {
        key[i] = 0.0f;
        return;
    }
    const double t = ca.t[i], h = ca.h[i];
    double l[VO_EXP_MAX_M];
    GenCos::coef<VO_EXP_MAX_M>(gp + i * (kp.M_gen - 1) * 3, kp.M_gen, t + 0.5 * h, l);
    double th = 0.0;
    for (int m = 0; m < kp.M; ++m) th += fabs(l[m]) * kp.norm1[m];
    key[i] = (float)(th * h);
}

// Order of the systems for the coming event: ascending key, so that every tile of 16 holds systems of similar theta.
static int32_t exp_dynamic_order(vo_expsolver_s* s, const ExpKP& kp, const int** order) {
    vo_ctx c = s->ctx;
    *order = nullptr;
    // (exp_small_kernel plans every system on its own: there are no tiles to group)
    if (!s->dynamic_group || s->gen_fn || s->sp->n <= VO_EXP_SMALL_MAX_N || s->N < 64 || s->N > 0x7fffffff) return VO_OK;
    const int n = (int)s->N;
    if (!s->key_in) {
        const size_t tmp = vo_sort_pairs_tmp_bytes(n);
        if (vo_dmalloc(&s->key_in, 4 * (size_t)n) != cudaSuccess || vo_dmalloc(&s->key_out, 4 * (size_t)n) != cudaSuccess || vo_dmalloc(&s->idx_in, 4 * (size_t)n) != cudaSuccess ||
            vo_dmalloc(&s->idx_out, 4 * (size_t)n) != cudaSuccess || vo_dmalloc(&s->sort_tmp, tmp) != cudaSuccess)
            return vo_fail(c, VO_ERR_ALLOC, "exp: dynamic grouping buffers");
        s->sort_tmp_bytes = tmp;
    }
    exp_group_key_kernel<<<(unsigned)ceil_div(s->N, 256), 256, 0, c->stream>>>(kp, s->gp, s->ca, s->N, s->key_in, s->idx_in);
    VO_CHECK_LAUNCH(c);
    if (vo_sort_pairs(s->sort_tmp, s->sort_tmp_bytes, s->key_in, s->key_out, s->idx_in, s->idx_out, n, c->stream) != cudaSuccess)
        return vo_fail(c, VO_ERR_CUDA, "exp: dynamic grouping sort");
    if (!s->tile_ctr && vo_dmalloc(&s->tile_ctr, sizeof(int)) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "exp: tile counter");
    VO_CUDA(c, cudaMemsetAsync(s->tile_ctr, 0, sizeof(int), c->stream));
    *order = s->idx_out;
    return VO_OK;
}

// One event of every system, or with events > 1 (exp_small_kernel only) that many in one launch.
int32_t exp_launch_event(vo_expsolver_s* s, bool adaptive, int events = 1) {
    vo_ctx c = s->ctx;
    if (adaptive && !s->want_err) return vo_fail(c, VO_ERR_NOT_ADAPTIVE, "adaptive step validation failed");  // ode.rs:312
    if (adaptive && (s->scheme == VO_EXP_MIDPOINT || s->scheme == VO_EXP_SPLIT_MIDPOINT || s->scheme == VO_EXP_SPLIT_CFM))
        return vo_fail(c, VO_ERR_NOT_ADAPTIVE, "this solver has no error estimate (it only implements ODESolver)");
    const bool tables = s->scheme == VO_EXP_CFM4 || s->scheme == VO_EXP_CFM_TABLE || s->scheme == VO_EXP_SPLIT_CFM;
    if (tables && s->n_rows < 1) return vo_fail(c, VO_ERR_STATE, "exp: the scheme's tables have not been set (vo_exp_set_cfm_tables / vo_exp_set_split_cfm_tables)");
    if (adaptive && tables && s->n_rows_err < 1) return vo_fail(c, VO_ERR_NOT_ADAPTIVE, "adaptive step validation failed");  // alph_err is None (cfm.rs:214-222)
    if (s->scheme == VO_EXP_MAGNUS42 && !s->sp->has_cs && !s->dense_comm && !s->applied_comm)
        return vo_fail(c, VO_ERR_BAD_ARG, "Magnus needs a Commutator (exp/mod.rs:47-54): vo_split_set_commutator for a basis closed under commutation, vo_exp_set_applied_commutator or vo_exp_set_dense_commutator");
    ExpKP kp = make_kp(s->sp, 0);
    kp.M_gen = s->M_gen, kp.scheme = s->scheme, kp.adaptive = adaptive ? 1 : 0;
    kp.want_err = (s->want_err && adaptive) ? 1 : 0;  // the embedded solution only feeds the controller
    kp.N = s->N, kp.count_events = 1, kp.n_events = events;
    kp.n_tlist = (int)s->t_list.size(), kp.t_list = s->t_list_dev;
    for (int i = 0; i < VO_INLINE_TLIST && i < kp.n_tlist; ++i) kp.t_list_inline[i] = s->t_list[i];
    kp.snap = s->snap, kp.out_perm = s->perm;
    kp.n_obs = s->n_obs, kp.obs = s->obs, kp.obs_out = s->obs_out;
    kp.rtol = s->rtol, kp.alpha = s->alpha, kp.pw = s->pw, kp.min_dt = s->min_dt, kp.max_dt = s->max_dt;
    kp.pw_is_third = s->pw == 1.0 / 3.0;
    kp.literal_norm = (s->literal_norm && adaptive) ? 1 : 0;
    kp.applied_comm = (s->scheme == VO_EXP_MAGNUS42 && s->applied_comm) ? 1 : 0;
    kp.split_mask = s->split_mask;
    kp.n_nodes = s->n_nodes, kp.n_rows = s->n_rows, kp.n_rows_err = s->n_rows_err;
    std::memcpy(kp.tab_c, s->tab_c, sizeof kp.tab_c), std::memcpy(kp.tab_alpha, s->tab_alpha, sizeof kp.tab_alpha);
    std::memcpy(kp.tab_alpha_err, s->tab_alpha_err, sizeof kp.tab_alpha_err), std::memcpy(kp.row_split, s->row_split, sizeof kp.row_split);
    s->stepped = true;
    if (s->scheme == VO_EXP_MAGNUS42 && s->dense_comm) return launch_magnus_dense(s, kp);
    const int* order = nullptr;
    int32_t orc = exp_dynamic_order(s, kp, &order);
    if (orc != VO_OK) return orc;
    return dispatch_exp(s->sp, kp, s->psi, nullptr, s->gp, nullptr, s->ca, s->ev_dev, s->gen_fn, order, order ? s->tile_ctr : nullptr);
}

void exp_res_add(vo_step_result* res, const EvSlot& e, int launches) {
    if (!res) return;
    res->n_step += (int64_t)e.n_step, res->n_chkpt += (int64_t)e.n_chkpt, res->n_reject += (int64_t)e.n_reject, res->n_end += (int64_t)e.n_end;
    res->launches += launches;
}

int32_t exp_step_impl(vo_expsolver s, bool adaptive, vo_step_result* res) {
    if (!s) return VO_ERR_BAD_ARG;
    DeviceGuard g(s->ctx->device);
    if (res) std::memset(res, 0, sizeof *res);
    int32_t r = exp_launch_event(s, adaptive);
    if (r != VO_OK) return r;
    EvSlot d;
    r = exp_ev_read(s, &d);
    if (r != VO_OK) return r;
    s->n_done += (int64_t)d.n_end;
    exp_res_add(res, d, 1);
    if (res) res->n_active = s->N - s->n_done, res->state = res->n_active == 0 ? VO_STATE_DONE : VO_STATE_OK;
    return VO_OK;
}

}  // namespace

extern "C" {

int32_t vo_split_basis_create(vo_ctx c, int32_t n, int32_t M, const double* basis, vo_split* out) {
    if (!c || !basis || !out || M < 1 || M > VO_EXP_MAX_M || n < 1 || (n > VO_EXP_SMALL_MAX_N && n % 8))
        return vo_fail(c, VO_ERR_BAD_ARG, "vo_split_basis_create: need 1 <= n <= 8 or n a multiple of 8, and 1 <= M <= 4");
    DeviceGuard g(c->device);
    vo_split sp = new vo_split_s();
    sp->ctx = c, sp->n = n, sp->M = M;
    std::memset(sp->cs, 0, sizeof sp->cs);
    const int NW = n / 8, NK = n / 4;
    const bool small = n <= VO_EXP_SMALL_MAX_N;  // exp_small_kernel takes the basis as it is; the tiles of exp_step_kernel take DMMA fragments
    std::vector<double> frag(small ? 0 : (size_t)M * 2 * n * n);
    if (small) sp->small_basis.assign(basis, basis + (size_t)M * 2 * n * n);
    for (int m = 0; m < M; ++m) {
        double best = 0.0;  // induced 1-norm: max column sum of |B_rc|
        for (int col = 0; col < n; ++col) {
            double sum = 0.0;
            for (int r = 0; r < n; ++r) sum += std::hypot(basis[(((size_t)m * n + r) * n + col) * 2], basis[(((size_t)m * n + r) * n + col) * 2 + 1]);
            best = std::max(best, sum);
        }
        sp->norm1[m] = best;
        for (int p = 0; p < 2 && !small; ++p)
            for (int w = 0; w < NW; ++w)
                for (int kk = 0; kk < NK; ++kk)
                    for (int l = 0; l < 32; ++l)  // A fragment of mma.m8n8k4: lane l holds A[l/4][l%4]
                        frag[((((size_t)(m * 2 + p) * NW + w) * NK + kk) * 32) + l] = basis[(((size_t)m * n + 8 * w + l / 4) * n + 4 * kk + l % 4) * 2 + p];
    }
    if (!small) {
        if (vo_dmalloc(&sp->frag_dev, frag.size() * sizeof(double)) != cudaSuccess) {
            delete sp;
            return vo_fail(c, VO_ERR_ALLOC, "vo_split_basis_create: cudaMalloc failed");
        }
        VO_CUDA(c, cudaMemcpyAsync(sp->frag_dev, frag.data(), frag.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    }
    if (vo_dmalloc(&sp->basis_dev, sizeof(double2) * (size_t)M * n * n) != cudaSuccess) {
        vo_split_destroy(sp);
        return vo_fail(c, VO_ERR_ALLOC, "vo_split_basis_create: cudaMalloc failed");
    }
    VO_CUDA(c, cudaMemcpyAsync(sp->basis_dev, basis, sizeof(double2) * (size_t)M * n * n, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    *out = sp;
    return VO_OK;
}

int32_t vo_split_destroy(vo_split sp) {
    if (!sp) return VO_OK;
    DeviceGuard g(sp->ctx->device);
    cudaStreamSynchronize(sp->ctx->stream);
    vo_dfree(sp->frag_dev), vo_dfree(sp->basis_dev);
    delete sp;
    return VO_OK;
}

int32_t vo_split_set_commutator(vo_split sp, const double* cs) {
    if (!sp || !cs) return VO_ERR_BAD_ARG;
    std::memcpy(sp->cs, cs, sizeof(double) * sp->M * sp->M * sp->M);
    sp->has_cs = true;
    return VO_OK;
}

int32_t vo_split_set_taylor_degree(vo_split sp, int32_t deg) {
    if (!sp || deg < 0 || deg > 60) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_split_set_taylor_degree: 0 <= deg <= 60");
    sp->taylor_deg = deg;
    return VO_OK;
}

int32_t vo_split_norm(vo_split sp, const void* psi_dev, int64_t N, double* out_host) {
    if (!sp || !psi_dev || !out_host || N < 1) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_split_norm: bad argument");
    vo_ctx c = sp->ctx;
    DeviceGuard g(c->device);
    double* out_dev = nullptr;
    VO_CUDA(c, cudaMallocAsync(&out_dev, sizeof(double) * N, c->stream));
    exp_norm_kernel<<<(unsigned)ceil_div(N, 8), 256, 0, c->stream>>>((const double2*)psi_dev, sp->n, N, out_dev);
    VO_CHECK_LAUNCH(c);
    VO_CUDA(c, cudaMemcpyAsync(out_host, out_dev, sizeof(double) * N, cudaMemcpyDeviceToHost, c->stream));
    cudaFreeAsync(out_dev, c->stream);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

// Commutator::commutator (exp/mod.rs:47-54) on coefficient vectors: out_c = sum_ab la_a lb_b cs[a][b][c]. Operators of this
// split ARE their M coefficients, so this is host-side bookkeeping on N*M complex numbers, not a device computation.
int32_t vo_split_commutator(vo_split sp, const double* la, const double* lb, int64_t N, double* out) {
    if (!sp || !la || !lb || !out || N < 1) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_split_commutator: bad argument");
    if (!sp->has_cs) return vo_fail(sp->ctx, VO_ERR_STATE, "vo_split_commutator: no structure tensor (vo_split_set_commutator)");
    const int M = sp->M;
    for (int64_t i = 0; i < N; ++i)
        for (int cc = 0; cc < M; ++cc) {
            std::complex<double> acc(0.0, 0.0);
            for (int a = 0; a < M; ++a)
                for (int b = 0; b < M; ++b) {
                    const double sc = sp->cs[(a * M + b) * M + cc];
                    if (sc != 0.0)
                        acc += std::complex<double>(la[(i * M + a) * 2], la[(i * M + a) * 2 + 1]) * std::complex<double>(lb[(i * M + b) * 2], lb[(i * M + b) * 2 + 1]) * sc;
                }
            out[(i * M + cc) * 2] = acc.real(), out[(i * M + cc) * 2 + 1] = acc.imag();
        }
    return VO_OK;
}

int32_t vo_map_exp_seq(vo_split sp, const double* coef_host, int32_t K, int64_t N, void* psi_in_dev, void* psi_out_dev) {
    if (!sp || !coef_host || N < 1 || K < 1 || !psi_in_dev || !psi_out_dev) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_map_exp_seq: bad argument");
    vo_ctx c = sp->ctx;
    DeviceGuard g(c->device);
    double2* coef_dev = nullptr;
    const size_t bytes = sizeof(double2) * (size_t)K * N * sp->M;
    VO_CUDA(c, cudaMallocAsync(&coef_dev, bytes, c->stream));
    VO_CUDA(c, cudaMemcpyAsync(coef_dev, coef_host, bytes, cudaMemcpyHostToDevice, c->stream));
    ExpKP kp = make_kp(sp, 1);
    kp.N = N, kp.nseq = K;
    CtlArrays none{};
    int32_t r = dispatch_exp(sp, kp, (double2*)psi_in_dev, (double2*)psi_out_dev, nullptr, coef_dev, none, nullptr);
    cudaFreeAsync(coef_dev, c->stream);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return r;
}

int32_t vo_map_exp(vo_split sp, const double* coef_host, int64_t N, void* psi_in_dev, void* psi_out_dev) {
    return vo_map_exp_seq(sp, coef_host, 1, N, psi_in_dev, psi_out_dev);
}

int32_t vo_exp_set_split_mask(vo_expsolver s, uint32_t a_mask) {
    if (!s) return VO_ERR_BAD_ARG;
    s->split_mask = a_mask;
    return VO_OK;
}

int32_t vo_exp_create(vo_ctx c, vo_split sp, int32_t scheme, int32_t M_gen, const double* gp_host, int64_t N, double t0, double tf,
                      const double* psi0_host, double h, vo_expsolver* out) {
    if (!c || !sp || !out || !psi0_host || N < 1 || scheme < 0 || scheme > VO_EXP_SPLIT_CFM || M_gen < 1 || M_gen > sp->M || (M_gen > 1 && !gp_host))
        return vo_fail(c, VO_ERR_BAD_ARG, "vo_exp_create: bad argument");
    if (sp->kind != 0) return vo_fail(c, VO_ERR_BAD_ARG, "vo_exp_create: the solvers take a shared-basis split (vo_split_basis_create)");
    DeviceGuard g(c->device);
    vo_expsolver s = new vo_expsolver_s();
    s->ctx = c, s->sp = sp, s->scheme = scheme, s->M_gen = M_gen, s->N = N, s->t0 = t0, s->tf = tf, s->h_init = h;
    s->t_list = {t0, tf};  // ODEData::new, ode.rs:144
    if (scheme == VO_EXP_CFM4) exp_store_tables(s, C_GAUSS_LEGENDRE_4, 2, CFM_R4_J2_GL, 2, CFM_R2_J1_GL, 1);  // ExpCFMSolver::new, cfm.rs:131-154
    const size_t nb = sizeof(double2) * (size_t)N * sp->n, ngp = sizeof(double) * (size_t)N * std::max(1, M_gen - 1) * 3;
    bool ok = vo_dmalloc(&s->psi, nb) == cudaSuccess && vo_dmalloc(&s->psi0, nb) == cudaSuccess && vo_dmalloc(&s->gp, ngp) == cudaSuccess &&
              vo_dmalloc(&s->ca.t, 8 * N) == cudaSuccess && vo_dmalloc(&s->ca.h, 8 * N) == cudaSuccess && vo_dmalloc(&s->ca.prev_h, 8 * N) == cudaSuccess &&
              vo_dmalloc(&s->ca.dx_norm, 8 * N) == cudaSuccess && vo_dmalloc(&s->ca.n_accept, 4 * N) == cudaSuccess &&
              vo_dmalloc(&s->ca.n_reject, 4 * N) == cudaSuccess && vo_dmalloc(&s->ca.word, 4 * N) == cudaSuccess &&
              vo_dmalloc(&s->ev_dev, sizeof(EvSlot) * VO_EV_SLOTS) == cudaSuccess && cudaMallocHost(&s->ev_host, sizeof(EvSlot) * VO_EV_SLOTS) == cudaSuccess;
    if (!ok) {
        vo_exp_destroy(s);
        return vo_fail(c, VO_ERR_ALLOC, "vo_exp_create: allocation failed");
    }
    VO_CUDA(c, cudaMemcpyAsync(s->psi0, psi0_host, nb, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaMemcpyAsync(s->psi, s->psi0, nb, cudaMemcpyDeviceToDevice, c->stream));
    if (M_gen > 1) VO_CUDA(c, cudaMemcpyAsync(s->gp, gp_host, ngp, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaMemsetAsync(s->ev_dev, 0, sizeof(EvSlot) * VO_EV_SLOTS, c->stream));
    exp_ctl_fill_kernel<<<(unsigned)ceil_div(N, 256), 256, 0, c->stream>>>(s->ca, N, t0, h);
    VO_CHECK_LAUNCH(c);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    *out = s;
    return VO_OK;
}

int32_t vo_exp_destroy(vo_expsolver s) {
    if (!s) return VO_OK;
    DeviceGuard g(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    vo_dfree(s->psi), vo_dfree(s->psi0), vo_dfree(s->gp);
    vo_dfree(s->ca.t), vo_dfree(s->ca.h), vo_dfree(s->ca.prev_h), vo_dfree(s->ca.dx_norm), vo_dfree(s->ca.n_accept), vo_dfree(s->ca.n_reject), vo_dfree(s->ca.word);
    vo_dfree(s->key_in), vo_dfree(s->key_out), vo_dfree(s->idx_in), vo_dfree(s->idx_out), vo_dfree(s->sort_tmp), vo_dfree(s->tile_ctr);
    vo_dfree(s->ev_dev), cudaFreeHost(s->ev_host);
    rtc_exp_unload(s->gen_module);
    vo_dfree(s->perm), vo_dfree(s->stage);
    vo_dfree(s->t_list_dev), vo_dfree(s->snap), vo_dfree(s->obs), vo_dfree(s->obs_out);
    delete s;
    return VO_OK;
}

// Output storage [len(t_list)][N][width] for the current list, zeroed: a system writes its row of entry k at its Chkpt / End event for
// t_list[k] (snapshots: width n; expectation values: width n_obs)
static int32_t exp_alloc_rows(vo_expsolver_s* s, double2** buf, int width) {
    vo_ctx c = s->ctx;
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    vo_dfree(*buf), *buf = nullptr;
    const size_t bytes = sizeof(double2) * s->t_list.size() * (size_t)s->N * width;
    if (vo_dmalloc(buf, bytes) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "exp: output storage: cudaMalloc failed");
    VO_CUDA(c, cudaMemsetAsync(*buf, 0, bytes, c->stream));
    return VO_OK;
}

// (re)build the run-time compiled exp_step_kernel from the solver's generator and norm sources
static int32_t exp_rebuild_rtc(vo_expsolver_s* s) {
    vo_ctx c = s->ctx;
    unsigned threads = 0;
    size_t smem = 0;
    if (!exp_geometry(s->sp->n, s->sp->M, &threads, &smem)) return vo_fail(c, VO_ERR_UNSUPPORTED, "exp: unsupported shape for a run-time compiled kernel");
    void *mod = nullptr, *fn = nullptr;
    int32_t r = rtc_exp_module(c, s->gen_body, s->norm_src, s->sp->n, s->sp->M, smem, &mod, &fn);
    if (r != VO_OK) return r;
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    rtc_exp_unload(s->gen_module);
    s->gen_module = mod, s->gen_fn = fn;
    return VO_OK;
}

int32_t vo_exp_set_generator(vo_expsolver s, const char* body) {
    if (!s || !body) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_set_generator: NULL argument");
    DeviceGuard g(s->ctx->device);
    const std::string old = s->gen_body;
    s->gen_body = body;
    const int32_t r = exp_rebuild_rtc(s);
    if (r != VO_OK) s->gen_body = old;
    return r;
}

int32_t vo_exp_set_norm_custom(vo_expsolver s, vo_normfn f) {
    if (!s || !f) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_set_norm_custom: NULL argument");
    if (s->dense_comm) return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "vo_exp_set_norm_custom: not available together with vo_exp_set_dense_commutator");
    DeviceGuard g(s->ctx->device);
    const std::string old = s->norm_src;
    s->norm_src = norm_source(f);
    const int32_t r = exp_rebuild_rtc(s);
    if (r != VO_OK) s->norm_src = old;
    return r;
}

int32_t vo_exp_set_cfm_tables(vo_expsolver s, const double* c, int32_t k, const double* alpha, int32_t rows, const double* alpha_err, int32_t rows_err) {
    if (!s) return VO_ERR_BAD_ARG;
    if (s->scheme != VO_EXP_CFM_TABLE && s->scheme != VO_EXP_CFM4) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_cfm_tables: the solver was not created with VO_EXP_CFM_TABLE");
    return exp_store_tables(s, c, k, alpha, rows, alpha_err, rows_err);
}

int32_t vo_exp_set_split_cfm_tables(vo_expsolver s, const double* c, int32_t k, const double* rho, const double* sigma, int32_t stages) {
    if (!s) return VO_ERR_BAD_ARG;
    if (s->scheme != VO_EXP_SPLIT_CFM) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_split_cfm_tables: the solver was not created with VO_EXP_SPLIT_CFM");
    if (!c || !rho || !sigma || stages < 1 || 2 * stages + 1 > VO_EXP_MAX_ROWS || k < 1 || k > VO_EXP_MAX_NODES)
        return vo_fail(s->ctx, VO_ERR_SHAPE, "split_cfm: Incompatible array dimensions");  // split_exp.rs:587-592
    // B(sigma_0) A(rho_0) B(sigma_1) ... A(rho_{s-1}) B(sigma_s), split_exp.rs:601-608
    std::vector<double> rows((size_t)(2 * stages + 1) * k);
    for (int i = 0; i <= stages; ++i) std::memcpy(&rows[(size_t)(2 * i) * k], &sigma[(size_t)i * k], sizeof(double) * k);
    for (int i = 0; i < stages; ++i) std::memcpy(&rows[(size_t)(2 * i + 1) * k], &rho[(size_t)i * k], sizeof(double) * k);
    int32_t r = exp_store_tables(s, c, k, rows.data(), 2 * stages + 1, nullptr, 0);
    if (r != VO_OK) return r;
    for (int e = 0; e < 2 * stages + 1; ++e) s->row_split[e] = (e % 2 == 0) ? 2 : 1;
    return VO_OK;
}

int32_t vo_cfm_builtin_table(int32_t which, double* out, int32_t* rows, int32_t* cols) {
    const double* src = nullptr;
    int r = 0, k = 0;
    switch (which) {
        case VO_CFM_C_GAUSS_LEGENDRE_4: src = C_GAUSS_LEGENDRE_4, r = 1, k = 2; break;
        case VO_CFM_R2_J1_GL: src = CFM_R2_J1_GL, r = 1, k = 2; break;
        case VO_CFM_R4_J2_GL: src = CFM_R4_J2_GL, r = 2, k = 2; break;
        case VO_CFM_BLANES17_R4_J4: src = BLANES17_R4_J4, r = 4, k = 3; break;
        default: return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_cfm_builtin_table: unknown table");
    }
    if (out) std::memcpy(out, src, sizeof(double) * r * k);
    if (rows) *rows = r;
    if (cols) *cols = k;
    return VO_OK;
}

int32_t vo_exp_no_adaptive(vo_expsolver s) {
    if (!s) return VO_ERR_BAD_ARG;
    s->want_err = false;  // exp/cfm.rs:157-161: alph_err = None
    return VO_OK;
}

int32_t vo_exp_with_tolerance(vo_expsolver s, double atol, double rtol) {
    if (!s) return VO_ERR_BAD_ARG;
    if (!(atol > 0.0) || !(rtol > 0.0)) return vo_fail(s->ctx, VO_ERR_BAD_ARG, "Invalid tolerances: atol=" + std::to_string(atol) + ", rtol=" + std::to_string(rtol));
    s->atol = atol, s->rtol = rtol;
    return VO_OK;
}

int32_t vo_exp_with_step_range(vo_expsolver s, double dt_min, double dt_max) {
    if (!s) return VO_ERR_BAD_ARG;
    if (!(dt_min > 0.0) || !(dt_max > 0.0) || !(dt_max > dt_min))
        return vo_fail(s->ctx, VO_ERR_BAD_ARG, "Invalid step range: (" + std::to_string(dt_min) + ", " + std::to_string(dt_max) + ")");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    s->min_dt = dt_min, s->max_dt = dt_max;
    s->h_init = std::sqrt(dt_min * dt_max);  // ode.rs:273-280
    exp_ctl_fill_kernel<<<(unsigned)ceil_div(s->N, 256), 256, 0, c->stream>>>(s->ca, s->N, s->t0, s->h_init);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

int32_t vo_exp_step(vo_expsolver s, vo_step_result* res) { return exp_step_impl(s, false, res); }
int32_t vo_exp_step_adaptive(vo_expsolver s, vo_step_result* res) { return exp_step_impl(s, true, res); }

int32_t vo_exp_run(vo_expsolver s, int32_t adaptive, int64_t max_calls, vo_step_result* res) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    vo_step_result acc;
    std::memset(&acc, 0, sizeof acc);
    int64_t calls = 0;
    int batch = 2;
    while (s->n_done < s->N && (max_calls <= 0 || calls < max_calls)) {
        int launched = 0;
        int left = batch;  // calls of this batch
        if (max_calls > 0) left = (int)std::min<int64_t>(left, max_calls - calls);
        const int fuse = s->sp->n <= VO_EXP_SMALL_MAX_N && !(s->scheme == VO_EXP_MAGNUS42 && s->dense_comm) ? VO_EXP_SMALL_FUSE : 1;
        while (left > 0) {
            const int ev = std::min(fuse, left);
            int32_t r = exp_launch_event(s, adaptive != 0, ev);
            if (r != VO_OK) return r;
            left -= ev, calls += ev, ++launched;
        }
        EvSlot d;
        int32_t r = exp_ev_read(s, &d);
        if (r != VO_OK) return r;
        s->n_done += (int64_t)d.n_end;
        exp_res_add(&acc, d, launched);
        if (d.n_stuck && d.n_step == 0 && d.n_chkpt == 0 && d.n_end == 0) {
            acc.n_active = s->N - s->n_done, acc.state = VO_STATE_ERR;
            if (res) *res = acc;
            return vo_fail(c, VO_ERR_STATE, "vo_exp_run: all remaining systems are rejected at h == min_dt");
        }
        batch = std::min(batch * 2, 16);
    }
    acc.n_active = s->N - s->n_done, acc.state = acc.n_active == 0 ? VO_STATE_DONE : VO_STATE_OK;
    if (res) *res = acc;
    return VO_OK;
}

int32_t vo_exp_current(vo_expsolver s, double* t_min, double* t_max, double* psi_host) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    if (t_min || t_max) {
        std::vector<double> t((size_t)s->N);
        VO_CUDA(c, cudaMemcpyAsync(t.data(), s->ca.t, 8 * (size_t)s->N, cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(c, cudaStreamSynchronize(c->stream));
        const auto mm = std::minmax_element(t.begin(), t.end());
        if (t_min) *t_min = *mm.first;
        if (t_max) *t_max = *mm.second;
    }
    if (psi_host) {
        const double2* src = s->psi;
        if (s->perm) {  // back to the caller's order on the device, then one copy
            exp_reorder_kernel<<<(unsigned)ceil_div(s->N, 8), 256, 0, c->stream>>>(s->psi, s->stage, s->perm, s->sp->n, s->N, 1);
            VO_CHECK_LAUNCH(c);
            src = s->stage;
        }
        VO_CUDA(c, cudaMemcpyAsync(psi_host, src, sizeof(double2) * (size_t)s->N * s->sp->n, cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return VO_OK;
}

// The states in the caller's order as a device-side view for device-side consumers (vo_group_gather_*): one row of
// 2 * n * N doubles ([N][n] complex, interleaved), valid until the next step. With vo_exp_set_order in force the view is the
// solver's staging buffer after the device-side reordering, else the state itself.
int32_t vo_exp_current_device(vo_expsolver s, vo_ens* out) {
    if (!s || !out) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    const double2* src = s->psi;
    if (s->perm) {
        exp_reorder_kernel<<<(unsigned)ceil_div(s->N, 8), 256, 0, c->stream>>>(s->psi, s->stage, s->perm, s->sp->n, s->N, 1);
        VO_CHECK_LAUNCH(c);
        src = s->stage;
    }
    return vo_ens_wrap(c, const_cast<double2*>(src), 1, 2 * (int64_t)s->sp->n * s->N, out);
}

int32_t vo_exp_stats(vo_expsolver s, int64_t* accepted, int64_t* rejected, double* t, double* h, double* dx_norm) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    const size_t n = (size_t)s->N;
    std::vector<uint32_t> tmp(n);
    if (accepted) {
        VO_CUDA(c, cudaMemcpyAsync(tmp.data(), s->ca.n_accept, 4 * n, cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(c, cudaStreamSynchronize(c->stream));
        for (size_t i = 0; i < n; ++i) accepted[i] = tmp[i];
    }
    if (rejected) {
        VO_CUDA(c, cudaMemcpyAsync(tmp.data(), s->ca.n_reject, 4 * n, cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(c, cudaStreamSynchronize(c->stream));
        for (size_t i = 0; i < n; ++i) rejected[i] = tmp[i];
    }
    if (t) VO_CUDA(c, cudaMemcpyAsync(t, s->ca.t, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    if (h) VO_CUDA(c, cudaMemcpyAsync(h, s->ca.h, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    if (dx_norm) VO_CUDA(c, cudaMemcpyAsync(dx_norm, s->ca.dx_norm, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    if (!s->perm_host.empty()) {  // device order -> the caller's order (vo_exp_set_order)
        auto unpermute = [&](auto* a) {
            if (!a) return;
            std::vector<typename std::remove_pointer<decltype(a)>::type> v(a, a + n);
            for (size_t j = 0; j < n; ++j) a[(size_t)s->perm_host[j]] = v[j];
        };
        unpermute(accepted), unpermute(rejected), unpermute(t), unpermute(h), unpermute(dx_norm);
    }
    return VO_OK;
}

// adaptive_dat.dx is a clone of x0 that no step ever writes (magnus.rs:182-183, 249-250): its norm, per system, in ca.dx_norm
static int32_t exp_fill_literal_norm(vo_expsolver_s* s) {
    vo_ctx c = s->ctx;
    exp_norm_kernel<<<(unsigned)ceil_div(s->N, 8), 256, 0, c->stream>>>(s->psi0, s->sp->n, s->N, s->ca.dx_norm);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

int32_t vo_exp_reset(vo_expsolver s, const double* psi0_host) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    const size_t nb = sizeof(double2) * (size_t)s->N * s->sp->n;
    if (psi0_host && s->perm) {  // the caller's order on the host, the grouped order on the device
        VO_CUDA(c, cudaMemcpyAsync(s->stage, psi0_host, nb, cudaMemcpyHostToDevice, c->stream));
        exp_reorder_kernel<<<(unsigned)ceil_div(s->N, 8), 256, 0, c->stream>>>(s->stage, s->psi0, s->perm, s->sp->n, s->N, 0);
        VO_CHECK_LAUNCH(c);
    } else if (psi0_host) {
        VO_CUDA(c, cudaMemcpyAsync(s->psi0, psi0_host, nb, cudaMemcpyHostToDevice, c->stream));
    }
    VO_CUDA(c, cudaMemcpyAsync(s->psi, s->psi0, nb, cudaMemcpyDeviceToDevice, c->stream));
    VO_CUDA(c, cudaMemsetAsync(s->ev_dev, 0, sizeof(EvSlot) * VO_EV_SLOTS, c->stream));
    std::memset(&s->ev_seen, 0, sizeof s->ev_seen);
    s->n_done = 0, s->stepped = false;
    exp_ctl_fill_kernel<<<(unsigned)ceil_div(s->N, 256), 256, 0, c->stream>>>(s->ca, s->N, s->t0, s->h_init);
    VO_CHECK_LAUNCH(c);
    if (s->literal_norm) return exp_fill_literal_norm(s);
    return VO_OK;
}

int32_t vo_exp_set_literal_norm(vo_expsolver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    if (on && s->scheme != VO_EXP_MAGNUS42) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_literal_norm: only MagnusExpLinearSolver::norm reads adaptive_dat.dx (magnus.rs:274-276)");
    DeviceGuard g(s->ctx->device);
    s->literal_norm = on ? 1 : 0;
    return on ? exp_fill_literal_norm(s) : VO_OK;
}

int32_t vo_exp_set_order(vo_expsolver s, const int64_t* perm, int64_t n) {
    if (!s || !perm || n != s->N) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_set_order: bad argument");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    std::vector<char> seen((size_t)n, 0);
    for (int64_t j = 0; j < n; ++j) {
        if (perm[j] < 0 || perm[j] >= n || seen[(size_t)perm[j]]) return vo_fail(c, VO_ERR_BAD_ARG, "vo_exp_set_order: not a permutation");
        seen[(size_t)perm[j]] = 1;
    }
    if (!s->perm && (vo_dmalloc(&s->perm, 8 * (size_t)n) != cudaSuccess || vo_dmalloc(&s->stage, sizeof(double2) * (size_t)n * s->sp->n) != cudaSuccess))
        return vo_fail(c, VO_ERR_ALLOC, "vo_exp_set_order: cudaMalloc failed");
    s->perm_host.assign(perm, perm + n);
    VO_CUDA(c, cudaMemcpyAsync(s->perm, perm, 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

void* vo_exp_state_device_ptr(vo_expsolver s) { return s ? (void*)s->psi : nullptr; }

int32_t vo_exp_set_t_list(vo_expsolver s, const double* t_list, int32_t n) {
    if (!s || !t_list || n < 1) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_set_t_list: bad argument");
    if (n > (int32_t)VO_WORD_TGT_MASK) return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "vo_exp_set_t_list: list too long for per-system control");
    if (s->stepped) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_t_list: stepping has begun (vo_exp_reset rewinds it)");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    vo_dfree(s->t_list_dev), s->t_list_dev = nullptr;
    if (n > VO_INLINE_TLIST) {
        if (vo_dmalloc(&s->t_list_dev, sizeof(double) * n) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "vo_exp_set_t_list: cudaMalloc failed");
        VO_CUDA(c, cudaMemcpy(s->t_list_dev, t_list, sizeof(double) * n, cudaMemcpyHostToDevice));
    }
    s->t_list.assign(t_list, t_list + n);
    int32_t r = s->snap ? exp_alloc_rows(s, &s->snap, s->sp->n) : VO_OK;
    return r == VO_OK && s->n_obs ? exp_alloc_rows(s, &s->obs_out, s->n_obs) : r;
}

int32_t vo_exp_enable_snapshots(vo_expsolver s) {
    if (!s) return VO_ERR_BAD_ARG;
    if (s->snap) return VO_OK;
    DeviceGuard g(s->ctx->device);
    return exp_alloc_rows(s, &s->snap, s->sp->n);
}

static int32_t exp_snapshot_check(vo_expsolver s, int32_t k) {
    if (!s->snap) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_snapshot: snapshots are not enabled (vo_exp_enable_snapshots)");
    if (k < 0 || k >= (int32_t)s->t_list.size()) return vo_fail(s->ctx, VO_ERR_BAD_ARG, "vo_exp_snapshot: index outside t_list");
    return VO_OK;
}

int32_t vo_exp_snapshot(vo_expsolver s, int32_t k, double* psi_host) {
    if (!s || !psi_host) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_snapshot: NULL argument");
    int32_t r = exp_snapshot_check(s, k);
    if (r != VO_OK) return r;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    const size_t row = (size_t)s->N * s->sp->n;
    VO_CUDA(c, cudaMemcpyAsync(psi_host, s->snap + (size_t)k * row, sizeof(double2) * row, cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

int32_t vo_exp_snapshot_device(vo_expsolver s, int32_t k, vo_ens* out) {
    if (!s || !out) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_snapshot_device: NULL argument");
    int32_t r = exp_snapshot_check(s, k);
    if (r != VO_OK) return r;
    const int64_t row = (int64_t)s->N * s->sp->n;
    return vo_ens_wrap(s->ctx, s->snap + (size_t)k * row, 1, 2 * row, out);
}

int32_t vo_exp_set_observables(vo_expsolver s, int32_t K, const double* ops) {
    if (!s || K < 0 || K > VO_EXP_MAX_OBS || (K > 0 && !ops)) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_set_observables: bad argument");
    if (s->stepped) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_observables: stepping has begun (vo_exp_reset rewinds it)");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    vo_dfree(s->obs), vo_dfree(s->obs_out), s->obs = nullptr, s->obs_out = nullptr, s->n_obs = 0;
    if (K == 0) return VO_OK;
    const size_t bytes = sizeof(double2) * (size_t)K * s->sp->n * s->sp->n;
    if (vo_dmalloc(&s->obs, bytes) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "vo_exp_set_observables: cudaMalloc failed");
    VO_CUDA(c, cudaMemcpy(s->obs, ops, bytes, cudaMemcpyHostToDevice));
    int32_t r = exp_alloc_rows(s, &s->obs_out, K);
    if (r != VO_OK) {
        vo_dfree(s->obs), s->obs = nullptr;
        return r;
    }
    s->n_obs = K;
    return VO_OK;
}

static int32_t exp_expectation_check(vo_expsolver s, int32_t j) {
    if (!s->n_obs) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_expectation: observables are not set (vo_exp_set_observables)");
    if (j < 0 || j >= (int32_t)s->t_list.size()) return vo_fail(s->ctx, VO_ERR_BAD_ARG, "vo_exp_expectation: index outside t_list");
    return VO_OK;
}

int32_t vo_exp_expectation(vo_expsolver s, int32_t j, double* host) {
    if (!s || !host) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_expectation: NULL argument");
    int32_t r = exp_expectation_check(s, j);
    if (r != VO_OK) return r;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    const size_t row = (size_t)s->N * s->n_obs;
    VO_CUDA(c, cudaMemcpyAsync(host, s->obs_out + (size_t)j * row, sizeof(double2) * row, cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

int32_t vo_exp_expectation_device(vo_expsolver s, int32_t j, vo_ens* out) {
    if (!s || !out) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_exp_expectation_device: NULL argument");
    int32_t r = exp_expectation_check(s, j);
    if (r != VO_OK) return r;
    const int64_t row = (int64_t)s->N * s->n_obs;
    return vo_ens_wrap(s->ctx, s->obs_out + (size_t)j * row, 1, 2 * row, out);
}


// ---- dense split: ExponentialSplit / Commutator / NormedExponentialSplit (exp/mod.rs:11-54) with per-system n x n operators ------
int32_t vo_split_dense_create(vo_ctx c, int32_t n, int64_t N, vo_split* out) {
    if (!c || !out || n < 8 || n > 64 || n % 8 || N < 1) return vo_fail(c, VO_ERR_BAD_ARG, "vo_split_dense_create: need n % 8 == 0, 8 <= n <= 64 and N >= 1");
    vo_split sp = new vo_split_s();
    sp->ctx = c, sp->n = n, sp->M = 0, sp->kind = 1, sp->N = N;
    std::memset(sp->cs, 0, sizeof sp->cs), std::memset(sp->norm1, 0, sizeof sp->norm1);
    *out = sp;
    return VO_OK;
}

static bool dense_op_ok(vo_split sp, vo_ens e) { return sp && sp->kind == 1 && e && e->d == 1 && e->n == 2 * (int64_t)sp->n * sp->n * sp->N && e->ctx->device == sp->ctx->device; }

int32_t vo_dense_lin_zero(vo_split sp, vo_ens* out) {  // exp/mod.rs:20
    if (!sp || sp->kind != 1 || !out) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_dense_lin_zero: needs a dense split");
    return vo_ens_create(sp->ctx, 1, 2 * (int64_t)sp->n * sp->n * sp->N, out);
}

int32_t vo_dense_assemble(vo_split sp, vo_split basis, const double* coef_host, vo_ens L) {
    if (!sp || !basis || basis->kind != 0 || !coef_host || !dense_op_ok(sp, L) || basis->n != sp->n) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_dense_assemble: bad argument");
    vo_ctx c = sp->ctx;
    DeviceGuard g(c->device);
    double2* coef_dev = nullptr;
    const size_t bytes = sizeof(double2) * (size_t)sp->N * basis->M;
    VO_CUDA(c, cudaMallocAsync(&coef_dev, bytes, c->stream));
    VO_CUDA(c, cudaMemcpyAsync(coef_dev, coef_host, bytes, cudaMemcpyHostToDevice, c->stream));
    dense_assemble_kernel<<<(unsigned)std::min<int64_t>(ceil_div((int64_t)sp->n * sp->n * sp->N, 256), (int64_t)c->sm_count * 16), 256, 0, c->stream>>>(
        basis->basis_dev, coef_dev, basis->M, sp->n, sp->N, reinterpret_cast<double2*>(L->p));
    VO_CHECK_LAUNCH(c);
    cudaFreeAsync(coef_dev, c->stream);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

static int32_t dense_exp_scaled(vo_split sp, vo_ens L, double k, vo_ens U) {
    vo_ctx c = sp->ctx;
    const int nb = sp->n / 8;
#define VO_CALL(NB)                                                                                                 \
    {                                                                                                               \
        using G = DenseGeo<NB>;                                                                                     \
        auto kf = dense_exp_kernel<NB>;                                                                             \
        const size_t smem = 2 * G::MAT + (G::N + 2) * sizeof(double) + 8 * sizeof(int);                             \
        unsigned grid = 0;                                                                                          \
        int32_t r = dense_grid(c, kf, G::THREADS, smem, sp->N, &grid);                                              \
        if (r != VO_OK) return r;                                                                                   \
        kf<<<grid, G::THREADS, smem, c->stream>>>(reinterpret_cast<const double2*>(L->p), reinterpret_cast<double2*>(U->p), sp->N, k); \
    }
    VO_DENSE_DISPATCH(nb, VO_CALL)
#undef VO_CALL
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

int32_t vo_dense_exp(vo_split sp, vo_ens L, vo_ens U) {  // exp/mod.rs:23
    if (!dense_op_ok(sp, L) || !dense_op_ok(sp, U)) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_SHAPE, "vo_dense_exp: operators must be [N][n][n] complex ensembles of this dense split");
    DeviceGuard g(sp->ctx->device);
    return dense_exp_scaled(sp, L, 1.0, U);
}

int32_t vo_dense_multi_exp(vo_split sp, vo_ens L, const double* k_arr, int32_t K, const vo_ens* U_out) {  // exp/mod.rs:28-34: exp(k l) for every k
    if (!dense_op_ok(sp, L) || !k_arr || K < 1 || !U_out) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_dense_multi_exp: bad argument");
    DeviceGuard g(sp->ctx->device);
    for (int q = 0; q < K; ++q) {
        if (!dense_op_ok(sp, U_out[q])) return vo_fail(sp->ctx, VO_ERR_SHAPE, "vo_dense_multi_exp: bad output operator");
        int32_t r = dense_exp_scaled(sp, L, k_arr[q], U_out[q]);
        if (r != VO_OK) return r;
    }
    return VO_OK;
}

int32_t vo_dense_map_exp(vo_split sp, vo_ens U, const void* psi_in_dev, void* psi_out_dev) {  // exp/mod.rs:25
    if (!dense_op_ok(sp, U) || !psi_in_dev || !psi_out_dev || psi_in_dev == psi_out_dev) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_BAD_ARG, "vo_dense_map_exp: bad argument (in-place is not supported)");
    vo_ctx c = sp->ctx;
    DeviceGuard g(c->device);
    dense_matvec_kernel<<<(unsigned)std::min<int64_t>(sp->N, (int64_t)c->sm_count * 8), 256, sizeof(double2) * sp->n, c->stream>>>(
        reinterpret_cast<const double2*>(U->p), reinterpret_cast<const double2*>(psi_in_dev), reinterpret_cast<double2*>(psi_out_dev), sp->n, sp->N);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

int32_t vo_dense_commutator(vo_split sp, vo_ens La, vo_ens Lb, vo_ens out) {  // exp/mod.rs:47-54
    if (!dense_op_ok(sp, La) || !dense_op_ok(sp, Lb) || !dense_op_ok(sp, out)) return vo_fail(sp ? sp->ctx : nullptr, VO_ERR_SHAPE, "vo_dense_commutator: operators must be [N][n][n] complex ensembles of this dense split");
    vo_ctx c = sp->ctx;
    DeviceGuard g(c->device);
    const int nb = sp->n / 8;
#define VO_CALL(NB)                                                                                                                          \
    {                                                                                                                                        \
        using G = DenseGeo<NB>;                                                                                                              \
        auto kf = dense_commutator_kernel<NB>;                                                                                               \
        unsigned grid = 0;                                                                                                                   \
        int32_t r = dense_grid(c, kf, G::THREADS, 2 * G::MAT, sp->N, &grid);                                                                 \
        if (r != VO_OK) return r;                                                                                                            \
        kf<<<grid, G::THREADS, 2 * G::MAT, c->stream>>>(reinterpret_cast<const double2*>(La->p), reinterpret_cast<const double2*>(Lb->p), reinterpret_cast<double2*>(out->p), sp->N); \
    }
    VO_DENSE_DISPATCH(nb, VO_CALL)
#undef VO_CALL
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

int32_t vo_exp_set_dynamic_grouping(vo_expsolver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    s->dynamic_group = on ? 1 : 0;
    return VO_OK;
}

int32_t vo_exp_set_applied_commutator(vo_expsolver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    if (on && s->scheme != VO_EXP_MAGNUS42) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_applied_commutator: only the Magnus solver takes a commutator");
    if (on && s->dense_comm) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_applied_commutator: the dense commutator is already selected");
    s->applied_comm = on ? 1 : 0;
    return VO_OK;
}

int32_t vo_exp_set_dense_commutator(vo_expsolver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    if (on && s->scheme != VO_EXP_MAGNUS42) return vo_fail(s->ctx, VO_ERR_STATE, "vo_exp_set_dense_commutator: only the Magnus solver takes a commutator");
    if (on && (s->sp->n > 64 || s->sp->n % 8)) return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "vo_exp_set_dense_commutator: n must be a multiple of 8, n <= 64");
    s->dense_comm = on ? 1 : 0;
    return VO_OK;
}

}  // extern "C"
