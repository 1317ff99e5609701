// rk_small_launch.cuh — host-side dispatch of rk_small_kernel over (stage count, arithmetic mode, control mode).
// Each RHS family is instantiated in its own translation unit (rk_small_<family>.cu) so they compile in parallel.
#pragma once
#include <map>
#include <mutex>
#include <tuple>
#include <utility>

#include "rk_small2.cuh"

constexpr int RK_SMALL_THREADS = 128;

// Host side of pipe::Chain for one solver: which staged kernel wrote the generation flags last, and with which grid. A launch
// may skip the grid-wide wait only if the launch before it (of this solver) was the SAME kernel instantiation on the SAME
// grid — then CTA b of both launches owns the same tiles (the tile -> CTA map is a function of the grid size) — and nothing
// else has touched the solver's state in between (`live`, kept by solver.cu from the ctx's epoch).
struct ChainState {
    uint32_t* flags = nullptr;
    uint32_t gen = 0;
    const void* fn = nullptr;
    unsigned grid = 0;
    bool live = false;
    pipe::Chain next(const void* kernel, unsigned g, bool staged) {
        pipe::Chain ch{flags, ++gen, (staged && live && fn == kernel && grid == g) ? 1 : 0};
        fn = kernel, grid = g, live = staged;
        return ch;
    }
};

struct SmallLaunch {
    vo_ctx ctx;
    double* x;
    int64_t N;
    const TableauDev* tb;
    const RhsParams* rp;
    CtlArrays ca;
    const CtlShared* cs;   // per-trajectory control (sl == nullptr)
    const StepList* sl;    // lock-step fixed steps (cs == nullptr)
    EvSlot* ev;
    ChainState* cst;       // chaining state of the owning solver
};

// The staged kernels need 16-byte aligned SoA rows (N even) and at least one full tile.
static inline bool small_path_is_staged(int64_t N) { return (N % 2 == 0) && N >= RK_SMALL_THREADS; }

// The register-resident kernels. The order is that of a run-time compiled module's function table (nvrtc_rhs.cu).
enum SmallKernel { SK_FIXED2W, SK_FIXED_STAGED, SK_FIXED, SK_CTL2W, SK_CTL_STAGED_L2, SK_CTL_STAGED_GEN, SK_CTL, SK_COUNT };

struct SmallPlan {
    SmallKernel k;
    int tile;     // trajectories per CTA tile, the unit of the persistent grid
    size_t smem;  // dynamic shared memory
    bool staged;  // a staged kernel: chained launches (pipe::Chain)
};

// The one kernel choice of the register-resident path, for the compiled-in families (launch_one) and for run-time compiled
// modules (launch_small_custom). `unrolled`: the stage count has a fully unrolled instantiation (S > 0); `rows`: state
// components + per-trajectory parameter rows; `cs`: per-trajectory control, nullptr for lock-step fixed steps. The
// two-trajectory kernels (rk_small2.cuh) need an unrolled stage count and at least four of their tiles; the control one
// only serves the common adaptive configuration with one event per launch.
static inline SmallPlan small_plan(int64_t N, bool unrolled, int rows, const CtlShared* cs) {
    if (!small_path_is_staged(N)) return {cs ? SK_CTL : SK_FIXED, RK_SMALL_THREADS, 0, false};
    const bool two = unrolled && N >= 4 * VO_TILE2;
    if (!cs) {
        const int tile = two ? VO_TILE2 : VO_TILE;
        return {two ? SK_FIXED2W : SK_FIXED_STAGED, tile, (size_t)VO_STAGES * rows * tile * sizeof(double), true};
    }
    const bool common = cs->adaptive && cs->use_err && cs->norm_kind == VO_NORM_L2;
    const bool ctl2 = two && common && cs->k_events == 1;
    const int tile = ctl2 ? VO_TILE2 : VO_TILE;
    // [stage][rows + t, h][tile] doubles, then [stage][status word, accepted, rejected][tile] words
    const size_t smem = (size_t)VO_STAGES * ((rows + 2) * tile * sizeof(double) + 3 * tile * sizeof(uint32_t));
    return {ctl2 ? SK_CTL2W : common ? SK_CTL_STAGED_L2 : SK_CTL_STAGED_GEN, tile, smem, true};
}

// Persistent grid: every CTA gets the same number of tiles (no partial last wave), all CTAs resident.
static inline unsigned grid_for(int64_t tiles, int sm_count, int blocks_per_sm) {
    const int64_t iters = ceil_div(tiles, (int64_t)sm_count * blocks_per_sm);
    return (unsigned)ceil_div(tiles, iters);
}

// The shared-memory size depends on run-time facts (how many RHS parameters are per-trajectory arrays), and both the large
// shared-memory opt-in and the occupancy are per device, so resident CTAs per SM are cached per (device, kernel, smem).
template <class K> static unsigned persistent_grid(vo_ctx c, K kernel, int64_t N, size_t smem, int tile) {
    static std::map<std::tuple<int, const void*, size_t>, int> cache;
    static std::mutex mu;  // contexts may be driven from different host threads
    int bps;
    {
        std::lock_guard<std::mutex> lock(mu);
        int& slot = cache[std::make_tuple(c->device, (const void*)kernel, smem)];
        if (slot == 0) {
            vo_ensure_smem_attr(c->device, (const void*)kernel, smem);
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&slot, kernel, RK_SMALL_THREADS, smem) != cudaSuccess || slot < 1) slot = 1;
        }
        bps = slot;
    }
    return grid_for(ceil_div(N, tile), c->sm_count, bps);
}

// A CHAINED launch (see pipe::Chain) is submitted with programmatic stream serialisation, so its CTAs are scheduled as
// the previous grid's CTAs retire and each starts as soon as its own predecessor CTA has published its generation flag.
// An unchained launch is an ordinary launch: it starts after everything before it in the stream has completed.
// The kernel's last parameter is the pipe::Chain, which is made here from the solver's ChainState once the grid is known.
template <class... KArgs, class... Args>
static void launch_staged(ChainState* cst, void (*kernel)(KArgs...), unsigned grid, size_t smem, cudaStream_t stream, Args&&... args) {
    const pipe::Chain ch = cst->next((const void*)kernel, grid, true);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid), cfg.blockDim = dim3(RK_SMALL_THREADS), cfg.dynamicSmemBytes = smem, cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = ch.chained ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)..., ch);
}

static inline int per_traj_rows(const RhsParams& rp, int np) {
    int n = 0;
    for (int q = 0; q < np; ++q) n += rp.per_traj[q] ? 1 : 0;
    return n;
}

template <class RHS, int S, bool STRICT> static void launch_one(const SmallLaunch& L) {
    const SmallPlan P = small_plan(L.N, S > 0, RHS::D + per_traj_rows(*L.rp, RHS::NP), L.cs);
    auto staged = [&](auto kernel, auto&&... args) {
        launch_staged(L.cst, kernel, persistent_grid(L.ctx, kernel, L.N, P.smem, P.tile), P.smem, L.ctx->stream, args...);
    };
    auto plain = [&](auto kernel, auto&&... args) {
        L.cst->live = false;
        kernel<<<persistent_grid(L.ctx, kernel, L.N, 0, P.tile), RK_SMALL_THREADS, 0, L.ctx->stream>>>(args...);
    };
    switch (P.k) {
        case SK_FIXED2W:
            if constexpr (S > 0) staged(rk_fixed2w_staged_kernel<RHS, S, STRICT>, L.x, L.N, *L.tb, *L.rp, *L.sl);
            break;
        case SK_FIXED_STAGED: staged(rk_fixed_staged_kernel<RHS, S, STRICT>, L.x, L.N, *L.tb, *L.rp, *L.sl); break;
        case SK_FIXED: plain(rk_fixed_kernel<RHS, S, STRICT>, L.x, L.N, *L.tb, *L.rp, *L.sl); break;
        case SK_CTL2W:
            if constexpr (S > 0) staged(rk_ctl2w_staged_kernel<RHS, S, STRICT>, L.x, L.N, *L.tb, *L.rp, L.ca, *L.cs, L.ev);
            break;
        case SK_CTL_STAGED_L2: staged(rk_ctl_staged_kernel<RHS, S, STRICT, 1>, L.x, L.N, *L.tb, *L.rp, L.ca, *L.cs, L.ev); break;
        case SK_CTL_STAGED_GEN: staged(rk_ctl_staged_kernel<RHS, S, STRICT, 0>, L.x, L.N, *L.tb, *L.rp, L.ca, *L.cs, L.ev); break;
        case SK_CTL: plain(rk_ctl_kernel<RHS, S, STRICT>, L.x, L.N, *L.tb, *L.rp, L.ca, *L.cs, L.ev); break;
        case SK_COUNT: break;
    }
}

template <class RHS, int S> static void launch_s(const SmallLaunch& L) {
    if (L.ctx->arith == VO_ARITH_STRICT) launch_one<RHS, S, true>(L);
    else launch_one<RHS, S, false>(L);
}

// Stage counts with a fully unrolled, register-resident instantiation; anything else (<= VO_MAX_STAGES)
// runs the generic S = 0 instantiation.
template <class RHS> static int32_t launch_family(const SmallLaunch& L) {
    switch (L.tb->s) {
        case 4: launch_s<RHS, 4>(L); break;
        case 6: launch_s<RHS, 6>(L); break;
        case 7: launch_s<RHS, 7>(L); break;
        default: launch_s<RHS, 0>(L); break;
    }
    return VO_OK;
}

// one per family TU
int32_t launch_small_diag(const SmallLaunch& L, int d);
int32_t launch_small_harmonic(const SmallLaunch& L);
int32_t launch_small_lorenz(const SmallLaunch& L);
int32_t launch_small_vdp(const SmallLaunch& L);
// user RHS compiled at run time (nvrtc_rhs.cu)
int32_t launch_small_custom(const SmallLaunch& L, vo_rhs_s* r);
