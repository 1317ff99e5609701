// solver.cu — the ensemble Runge-Kutta solver: RK45Solver + ODESolver + AdaptiveODESolver
// (src/base/rk.rs:158-320, src/base/ode.rs:208-344) for N independent trajectories held SoA on the device.
//
// Where the reference owns one solver object per trajectory, one vo_solver owns the whole ensemble. Control
// state (t, h, prev_h, tgt_t, counters) is either
//   * LOCK-STEP ("uniform"): every trajectory shares the scalars — true for step() on a freshly built solver,
//     because the state machine of ode.rs:165-206 then never looks at the state. The scalars live on the host,
//     are advanced there with the reference's arithmetic, and the kernels read them as launch parameters: the
//     only HBM traffic of a step is the state itself; or
//   * PER-TRAJECTORY: device arrays of length N, entered on the first step_adaptive() (or when per-trajectory
//     initial steps are set). Rejected / finished lanes are masked inside the kernels.
//
// Two kernel paths:
//   * small systems (compiled-in pointwise RHS, d <= 4): rk_small_kernel — a whole attempt (all stages, error
//     estimate, norm, controller, commit) per thread in registers, k events per launch;
//   * stage path (any d; the only path for HEAT1D): one fused kernel per stage over K buffers in HBM, then a
//     norm + controller/commit step.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "rk_small_launch.cuh"
#include "rk_stage.cuh"
#include "rk_heat_fused.cuh"

int32_t vo_norm_device(vo_ens e, int32_t kind, double* out_dev, double* partial_dev, int partial_cap, bool finish);
int32_t launch_stage_stencil_custom(vo_ctx c, vo_rhs_s* r, bool tail, const double* x0, int64_t d, const StageArgs& sa, const RhsParams& rp, double* k_out, double* nx,
                                    double* xe);
int32_t launch_stage_custom(vo_ctx c, vo_rhs_s* r, bool tail, const double* x0, int64_t N, const StageArgs& sa, const RhsParams& rp, double* k_out, double* nx,
                            double* xe);  // nvrtc_rhs.cu

namespace {

constexpr double F64_EPS = 2.220446049250313e-16;
constexpr int PARTIAL_CAP = 1 << 14;
constexpr int CHAIN_FLAGS = 1 << 14;  // >= resident CTAs of any persistent grid (148 SMs x <= 32 CTAs)

}  // namespace

struct vo_solver_s {
    vo_ctx ctx = nullptr;
    vo_tableau_s tab;
    vo_rhs rhs = nullptr;
    int64_t d = 0, n = 0;
    double t0 = 0, tf = 0, h_init = 0;
    vo_ens x = nullptr, next_x = nullptr, x_err = nullptr;
    std::vector<vo_ens> K;  // stage path, allocated on first use
    bool has_x_err = true;  // Option<V> x_err (rk.rs:249 Some; rk.rs:233-237 None)
    // ODEAdaptiveData (ode.rs:98-110)
    double atol = 1.0e-6, rtol = 1.0e-4, alpha = 0.9, pw = 1.0 / 3.0, min_dt = 1.0e-6, max_dt = 1.0;
    std::vector<double> t_list;
    double* t_list_dev = nullptr;
    int norm_kind = VO_NORM_L2;
    vo_normfn norm_fn = nullptr;   // VO_NORM_CUSTOM: the caller's functor (borrowed)
    vo_rhs_s* norm_rhs = nullptr;  // ... and the private RHS handle whose run-time modules carry it (register-resident path)
    double* dxn_pre = nullptr;     // ... stage path, per-trajectory control: norms computed ahead of ctl_commit_kernel
    // lock-step control
    bool uniform = true;
    double u_t = 0, u_h = 0, u_prev_h = 0, u_dx_norm = 0;
    int u_tgt = 0;
    bool u_done = false;
    int64_t u_accept = 0, u_reject = 0;
    bool try_pending = false;  // vo_adaptive_try has run rk_step and waits for vo_adaptive_handle
    double try_dt = 0;
    int try_launches = 0;
    // per-trajectory control
    CtlArrays ca{};
    uint8_t* evv = nullptr;  // stage path: event of the current call per trajectory
    double* dtv = nullptr;   // stage path: dt of the current call per trajectory
    double* norm_partial = nullptr;
    EvSlot* ev_dev = nullptr;
    EvSlot* ev_host = nullptr;  // pinned
    EvSlot ev_seen{};           // counter totals at the last read (device counters are cumulative)
    int64_t n_done = 0;         // per-trajectory mode: trajectories that have emitted End
    int k_events = 0;  // 0 = automatic: 1 per step()/step_many launch, fused inside vo_run (see run_fusion)
    int stage_path = 0;
    int record_dx_norm = 1;
    int mixed_stepping = 0;     // vo_solver_set_mixed_stepping: step() may follow step_adaptive() on per-trajectory control
    bool prev_h_stale = false;  // a lazy-prev_h adaptive launch has run: ca.prev_h is only valid where a checkpoint comes next
    double* snap = nullptr;  // [n_tlist][d][N] checkpoint snapshots (vo_solver_enable_snapshots)
    // CTA-to-CTA chaining of consecutive launches (pipe::Chain): generation flags, one per CTA, and which kernel / grid wrote
    // them last (rk_small_launch.cuh). The chain survives across API calls: it is alive while the ctx's epoch still has the
    // value it had right after this solver's previous register-resident launch, i.e. while nothing but such launches (of this
    // or of other solvers, which touch only their own state) has been enqueued on the ctx since.
    ChainState cst;
    uint64_t chain_epoch = 0;
};

namespace {

// register-resident whole-attempt kernels: compiled-in pointwise families up to 4 components, user right-hand sides up to 8
bool rhs_is_small(const vo_rhs_s* r) {
    if (r->kind == VO_RHS_CUSTOM) return r->d <= 8;
    return r->kind != VO_RHS_HEAT1D && r->kind != VO_RHS_CUSTOM_STENCIL && r->d <= 4;
}
bool use_small(const vo_solver_s* s) { return !s->stage_path && rhs_is_small(s->rhs); }
bool use_err(const vo_solver_s* s) { return s->tab.has_err && s->has_x_err; }
// Events fused per launch. step()/vo_step_many expose every event, so they advance one at a time unless the caller
// asked for more; vo_run only promises the state at the end, so it keeps each trajectory in registers for several
// events per launch (the FP64 pipe, not HBM, then bounds a sweep).
int step_fusion(const vo_solver_s* s) { return s->k_events > 0 ? s->k_events : 1; }
int run_fusion(const vo_solver_s* s) { return s->k_events > 0 ? s->k_events : (s->uniform ? 16 : 8); }
// Snapshot blocks: [d][N] per entry of t_list, each starting 16-byte aligned (vo_ens_wrap) even when d * N is odd.
int64_t snap_stride(const vo_solver_s* s) { return (s->d * s->n + 1) & ~(int64_t)1; }

TableauDev make_tableau_dev(const vo_tableau_s& t) {
    TableauDev d;
    std::memcpy(d.ac, t.ac, sizeof d.ac), std::memcpy(d.b, t.b, sizeof d.b), std::memcpy(d.b_err, t.b_err, sizeof d.b_err);
    d.s = t.s, d.has_err = t.has_err ? 1 : 0;
    d.reuse = 0;
    if (t.s >= 2) {
        const double* last = &t.ac[(t.s - 1) * t.s];
        if (t.has_err && std::memcmp(t.b_err, last, sizeof(double) * (t.s - 1)) == 0) d.reuse |= 1;
        if (std::memcmp(t.b, last, sizeof(double) * (t.s - 1)) == 0) d.reuse |= 2;
    }
    return d;
}

CtlShared make_ctl_shared(const vo_solver_s* s, int adaptive, int k_events) {
    CtlShared cs;
    std::memset(&cs, 0, sizeof cs);
    cs.rtol = s->rtol, cs.alpha = s->alpha, cs.pw = s->pw, cs.min_dt = s->min_dt, cs.max_dt = s->max_dt;
    cs.inv_rtol = 1.0 / s->rtol, cs.inv_rtol2 = 1.0 / (s->rtol * s->rtol);
    cs.n_tlist = (int)s->t_list.size();
    for (int i = 0; i < VO_INLINE_TLIST && i < cs.n_tlist; ++i) cs.t_list_inline[i] = s->t_list[i];
    cs.t_list = s->t_list_dev;
    cs.norm_kind = s->norm_kind;
    cs.adaptive = adaptive;
    cs.use_err = use_err(s) ? 1 : 0;
    cs.k_events = k_events;
    cs.count_events = 1;
    cs.pw_is_third = s->pw == 1.0 / 3.0 ? 1 : 0;
    cs.record_dx_norm = s->record_dx_norm;
    cs.lazy_prev_h = s->mixed_stepping ? 0 : 1;
    cs.snap = s->snap, cs.snap_stride = snap_stride(s);
    return cs;
}

// ---- host copy of the state machine for lock-step control (ode.rs:165-176, 389-399, 184-195) ----------
int uni_step_size(const vo_solver_s* s, double* dt) {
    if (s->u_tgt >= (int)s->t_list.size()) return VO_EV_END;
    const double rem = s->t_list[s->u_tgt] - s->u_t;
    if (std::fabs(rem) <= F64_EPS) return s->u_tgt >= (int)s->t_list.size() - 1 ? VO_EV_END : VO_EV_CHKPT;
    *dt = rem < s->u_h ? rem : s->u_h;
    return VO_EV_STEP;
}
void uni_checkpoint(vo_solver_s* s, bool end) {
    if (s->snap && s->u_tgt < (int)s->t_list.size()) {  // lock-step: the whole ensemble is at the checkpoint, copy it (stream-ordered)
        vo_touch(s->ctx);                                // the copy is not part of the CTA chain
        cudaMemcpyAsync(s->snap + (size_t)s->u_tgt * snap_stride(s), s->x->p, sizeof(double) * s->d * s->n, cudaMemcpyDeviceToDevice, s->ctx->stream);
    }
    s->u_tgt += 1, s->u_h = s->u_prev_h;
    if (end) s->u_done = true;
}

// ---- per-trajectory control helpers ---------------------------------------------------------------------
__global__ void ctl_fill_kernel(CtlArrays ca, int64_t N, double t, double h, double prev_h, double dxn, uint32_t acc, uint32_t rej, uint32_t word) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    ca.t[i] = t, ca.h[i] = h, ca.prev_h[i] = prev_h, ca.dx_norm[i] = dxn;
    ca.n_accept[i] = acc, ca.n_reject[i] = rej, ca.word[i] = word;
}

// stage path, per-trajectory: step_size_of (ode.rs:165-176) for every live trajectory.
__global__ void ctl_prepare_kernel(CtlArrays ca, const __grid_constant__ CtlShared cs, int64_t N, uint8_t* __restrict__ evv, double* __restrict__ dtv) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= N) return;
    const uint32_t word = ca.word[i];
    if ((word >> VO_WORD_STATUS_SHIFT) & VO_TRAJ_DONE) {
        evv[i] = 255;
        return;
    }
    const int tgt = (int)(word & VO_WORD_TGT_MASK);
    const double* tl = cs.n_tlist > VO_INLINE_TLIST ? cs.t_list : cs.t_list_inline;
    int evk;
    double dt = 0.0;
    if (tgt >= cs.n_tlist) {
        evk = VO_EV_END;
    } else {
        const double rem = tl[tgt] - ca.t[i], h = ca.h[i];
        if (fabs(rem) <= 2.220446049250313e-16) evk = (tgt >= cs.n_tlist - 1) ? VO_EV_END : VO_EV_CHKPT;
        else dt = rem < h ? rem : h, evk = VO_EV_STEP;
    }
    evv[i] = (uint8_t)evk, dtv[i] = dt;
}

// stage path, per-trajectory (d <= 64): error norm, handle_step_adaptive (ode.rs:311-334) and apply_step
// (ode.rs:402-428) with a masked commit next_x -> x for accepted lanes.
template <bool STRICT>
__global__ void ctl_commit_kernel(double* __restrict__ x, const double* __restrict__ next_x, const double* __restrict__ x_err, int64_t d, int64_t N,
                                  CtlArrays ca, const __grid_constant__ CtlShared cs, const uint8_t* __restrict__ evv, const double* __restrict__ dtv,
                                  EvSlot* __restrict__ ev, const double* __restrict__ dxn_pre) {
    using A = Ar<STRICT>;
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned c_step = 0, c_chkpt = 0, c_rej = 0, c_end = 0, c_stuck = 0;
    if (i < N && evv[i] != 255) {
        int evk = evv[i];
        const uint32_t word = ca.word[i];
        int tgt = (int)(word & VO_WORD_TGT_MASK);
        uint32_t status = word >> VO_WORD_STATUS_SHIFT;
        if (evk == VO_EV_STEP) {
            if (cs.adaptive) {
                double acc = 0.0;
                if (dxn_pre) {  // a user-defined norm, evaluated by its own run-time compiled kernel just before this one
                    acc = dxn_pre[i];
                } else if (cs.norm_kind == VO_NORM_HYPOT && d == 2) {
                    acc = hypot(x_err[i], x_err[N + i]);
                } else if (cs.norm_kind == VO_NORM_HYPOT) {
                    for (int64_t c = 0; c + 1 < d; c += 2) {
                        const double m = hypot(x_err[c * N + i], x_err[(c + 1) * N + i]);
                        acc = A::add(acc, A::mul(m, m));
                    }
                    acc = sqrt(acc);
                } else {
                    for (int64_t c = 0; c < d; ++c) {
                        const double e = x_err[c * N + i];
                        if (cs.norm_kind == VO_NORM_L2) acc = A::add(acc, A::mul(e, e));
                        else if (cs.norm_kind == VO_NORM_LINF) acc = fmax(acc, fabs(e));
                        else acc = A::add(acc, fabs(e));
                    }
                    if (cs.norm_kind == VO_NORM_L2) acc = sqrt(acc);
                }
                const double h = ca.h[i];
                double new_h;
                bool rejected;
                controller_ref<STRICT>(acc, h, cs, new_h, rejected);
                if (!(acc == acc)) status |= VO_TRAJ_NONFINITE;
                if (rejected) {
                    evk = VO_EV_REJECT;
                    if (h <= cs.min_dt) status |= VO_TRAJ_STUCK, ++c_stuck;
                }
                ca.prev_h[i] = h, ca.h[i] = new_h, ca.dx_norm[i] = acc;
            }
            if (evk == VO_EV_STEP) {
                for (int64_t c = 0; c < d; ++c) x[c * N + i] = next_x[c * N + i];
                ca.t[i] += dtv[i];
                ca.n_accept[i] += 1, ++c_step;
            } else {
                ca.n_reject[i] += 1, ++c_rej;
            }
        } else {
            if (cs.snap && tgt < cs.n_tlist)
                for (int64_t c = 0; c < d; ++c) cs.snap[tgt * cs.snap_stride + c * N + i] = x[c * N + i];
            tgt += 1, ca.h[i] = ca.prev_h[i];
            if (evk == VO_EV_END) status |= VO_TRAJ_DONE, ++c_end;
            else ++c_chkpt;
        }
        const uint32_t nw = ((uint32_t)tgt & VO_WORD_TGT_MASK) | (status << VO_WORD_STATUS_SHIFT);
        if (nw != word) ca.word[i] = nw;
    }
    c_step = __reduce_add_sync(0xffffffffu, c_step), c_chkpt = __reduce_add_sync(0xffffffffu, c_chkpt);
    c_rej = __reduce_add_sync(0xffffffffu, c_rej), c_end = __reduce_add_sync(0xffffffffu, c_end);
    c_stuck = __reduce_add_sync(0xffffffffu, c_stuck);
    if ((threadIdx.x & 31) == 0) {
        EvSlot* slot = ev + (blockIdx.x % VO_EV_SLOTS);
        if (c_step) atomicAdd(&slot->n_step, (unsigned long long)c_step);
        if (c_chkpt) atomicAdd(&slot->n_chkpt, (unsigned long long)c_chkpt);
        if (c_rej) atomicAdd(&slot->n_reject, (unsigned long long)c_rej);
        if (c_end) atomicAdd(&slot->n_end, (unsigned long long)c_end);
        if (c_stuck) atomicAdd(&slot->n_stuck, (unsigned long long)c_stuck);
    }
}

int32_t alloc_ctl(vo_solver_s* s) {
    if (s->ca.t) return VO_OK;
    vo_ctx c = s->ctx;
    const size_t n = (size_t)s->n;
    if (vo_dmalloc(&s->ca.t, 8 * n) != cudaSuccess || vo_dmalloc(&s->ca.h, 8 * n) != cudaSuccess || vo_dmalloc(&s->ca.prev_h, 8 * n) != cudaSuccess ||
        vo_dmalloc(&s->ca.dx_norm, 8 * n) != cudaSuccess || vo_dmalloc(&s->ca.n_accept, 4 * n) != cudaSuccess ||
        vo_dmalloc(&s->ca.n_reject, 4 * n) != cudaSuccess || vo_dmalloc(&s->ca.word, 4 * n) != cudaSuccess)
        return vo_fail(c, VO_ERR_ALLOC, "solver: per-trajectory control allocation failed");
    return VO_OK;
}

void free_ctl(vo_solver_s* s) {
    vo_dfree(s->ca.t), vo_dfree(s->ca.h), vo_dfree(s->ca.prev_h), vo_dfree(s->ca.dx_norm);
    vo_dfree(s->ca.n_accept), vo_dfree(s->ca.n_reject), vo_dfree(s->ca.word);
    s->ca = CtlArrays{};
}

// Per-shard totals for vo_group_reduce_stats: sums[6] = accepted, rejected, trajectories, done, non-finite, stuck;
// mm[2] = max t, max (-t). One block-reduced pass over the controller arrays, a handful of atomics per block.
__global__ void ctl_stats_kernel(CtlArrays ca, int64_t N, unsigned long long* __restrict__ sums, double* __restrict__ mm) {
    unsigned long long acc = 0, rej = 0, done = 0, nonfin = 0, stuck = 0;
    double tmax = -1.0e308, tneg = -1.0e308;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < N; i += (int64_t)gridDim.x * blockDim.x) {
        acc += ca.n_accept[i], rej += ca.n_reject[i];
        const uint32_t st = ca.word[i] >> VO_WORD_STATUS_SHIFT;
        done += (st & VO_TRAJ_DONE) ? 1 : 0, nonfin += (st & VO_TRAJ_NONFINITE) ? 1 : 0, stuck += (st & VO_TRAJ_STUCK) ? 1 : 0;
        const double t = ca.t[i];
        tmax = fmax(tmax, t), tneg = fmax(tneg, -t);
    }
    for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o), rej += __shfl_xor_sync(0xffffffffu, rej, o), done += __shfl_xor_sync(0xffffffffu, done, o);
        nonfin += __shfl_xor_sync(0xffffffffu, nonfin, o), stuck += __shfl_xor_sync(0xffffffffu, stuck, o);
        tmax = fmax(tmax, __shfl_xor_sync(0xffffffffu, tmax, o)), tneg = fmax(tneg, __shfl_xor_sync(0xffffffffu, tneg, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&sums[0], acc), atomicAdd(&sums[1], rej), atomicAdd(&sums[3], done), atomicAdd(&sums[4], nonfin), atomicAdd(&sums[5], stuck);
        // order-preserving integer image of a double, so that atomicMax on the bits is max on the values
        auto key = [](double v) {
            const long long b = __double_as_longlong(v);
            return b >= 0 ? b : (long long)(0x8000000000000000ull - (unsigned long long)b);
        };
        atomicMax(reinterpret_cast<long long*>(&mm[0]), key(tmax)), atomicMax(reinterpret_cast<long long*>(&mm[1]), key(tneg));
    }
}
__global__ void ctl_stats_finish_kernel(unsigned long long* sums, double* mm, unsigned long long n) {
    sums[2] = n;
    for (int q = 0; q < 2; ++q) {
        const long long k = *reinterpret_cast<long long*>(&mm[q]);
        mm[q] = __longlong_as_double(k >= 0 ? k : (long long)(0x8000000000000000ull - (unsigned long long)k));
    }
}

// lock-step -> per-trajectory: every trajectory inherits the shared scalars.
int32_t materialize(vo_solver_s* s) {
    if (!s->uniform) return VO_OK;
    if (s->t_list.size() > VO_WORD_TGT_MASK) return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "solver: t_list too long for per-trajectory control");
    int32_t r = alloc_ctl(s);
    if (r != VO_OK) return r;
    vo_ctx c = s->ctx;
    const uint32_t word = ((uint32_t)s->u_tgt & VO_WORD_TGT_MASK) | ((s->u_done ? (uint32_t)VO_TRAJ_DONE : 0u) << VO_WORD_STATUS_SHIFT);
    ctl_fill_kernel<<<(unsigned)ceil_div(s->n, 256), 256, 0, c->stream>>>(s->ca, s->n, s->u_t, s->u_h, s->u_prev_h, s->u_dx_norm, (uint32_t)s->u_accept,
                                                                         (uint32_t)s->u_reject, word);
    VO_CHECK_LAUNCH(c);
    s->n_done = s->u_done ? s->n : 0;
    s->uniform = false;
    return VO_OK;
}

void ev_sum(const EvSlot* h, EvSlot* out) {
    std::memset(out, 0, sizeof *out);
    for (int i = 0; i < VO_EV_SLOTS; ++i)
        out->n_step += h[i].n_step, out->n_chkpt += h[i].n_chkpt, out->n_reject += h[i].n_reject, out->n_end += h[i].n_end, out->n_stuck += h[i].n_stuck;
}

// The device counters are cumulative since creation / reset; ev_read returns what was added since the previous
// read (synchronises the stream), so launches made without a read-back (vo_step_many) are never lost.
int32_t ev_read(vo_solver_s* s, EvSlot* out) {
    vo_ctx c = s->ctx;
    const uint64_t epoch = c->epoch;
    VO_CUDA(c, vo_small_readback(c, s->ev_host, s->ev_dev, sizeof(EvSlot) * VO_EV_SLOTS));  // not a copy: see ctx.cu
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    c->epoch = epoch;  // reading the counters touches no solver state: the CTA chains stay alive
    EvSlot tot;
    ev_sum(s->ev_host, &tot);
    out->n_step = tot.n_step - s->ev_seen.n_step, out->n_chkpt = tot.n_chkpt - s->ev_seen.n_chkpt;
    out->n_reject = tot.n_reject - s->ev_seen.n_reject, out->n_end = tot.n_end - s->ev_seen.n_end;
    out->n_stuck = tot.n_stuck - s->ev_seen.n_stuck;
    s->ev_seen = tot;
    return VO_OK;
}

void res_add(vo_step_result* res, int64_t st, int64_t ck, int64_t rj, int64_t en, int launches) {
    if (!res) return;
    res->n_step += st, res->n_chkpt += ck, res->n_reject += rj, res->n_end += en, res->launches += launches;
}

// ---- small path ---------------------------------------------------------------------------------------------
int32_t launch_small(vo_solver_s* s, const CtlShared* cs, const StepList* sl) {
    vo_ctx c = s->ctx;
    const TableauDev tb = make_tableau_dev(s->tab);
    const RhsParams rp = make_rhs_params(s->rhs);
    if (s->chain_epoch != c->epoch) s->cst.live = false;  // something else was enqueued on the ctx since our last launch
    SmallLaunch L{c, s->x->p, s->n, &tb, &rp, s->ca, cs, sl, s->ev_dev, &s->cst};
    int32_t r = VO_ERR_UNSUPPORTED;
    if (s->norm_rhs) {  // a user-defined norm: the control kernels come from the run-time module that carries it
        r = launch_small_custom(L, s->norm_rhs);
        if (r != VO_OK) return r;
    } else
    switch (s->rhs->kind) {
        case VO_RHS_DIAG_LINEAR: r = launch_small_diag(L, s->rhs->d); break;
        case VO_RHS_HARMONIC2D: r = launch_small_harmonic(L); break;
        case VO_RHS_LORENZ63: r = launch_small_lorenz(L); break;
        case VO_RHS_VDP: r = launch_small_vdp(L); break;
        case VO_RHS_CUSTOM:
            r = launch_small_custom(L, s->rhs);
            if (r != VO_OK) return r;  // message already set (compile log, driver error)
            break;
    }
    if (r != VO_OK) return vo_fail(c, r, "solver: no register-resident kernel for this RHS");
    VO_CHECK_LAUNCH_CHAINED(c);
    s->chain_epoch = c->epoch;
    return VO_OK;
}

// Lock-step small path: advance the shared scalars through up to k events on the host exactly as the kernel
// does per thread, launching the kernel only when at least one of them is a Step.
int32_t small_uniform_events(vo_solver_s* s, int k, vo_step_result* res, int64_t* calls_done) {
    StepList sl;
    sl.n = 0, sl.use_err = use_err(s) ? 1 : 0;
    int64_t calls = 0;
    auto flush = [&]() -> int32_t {
        if (sl.n == 0) return VO_OK;
        int32_t r = launch_small(s, nullptr, &sl);
        sl.n = 0;
        res_add(res, 0, 0, 0, 0, 1);
        return r;
    };
    for (int e = 0; e < k && !s->u_done; ++e) {
        double dt = 0.0;
        const int ev = uni_step_size(s, &dt);
        ++calls;
        if (ev == VO_EV_STEP) {
            sl.t[sl.n] = s->u_t, sl.dt[sl.n] = dt, ++sl.n;
            s->u_t += dt, s->u_accept += 1;  // advance, ode.rs:184-188
            res_add(res, s->n, 0, 0, 0, 0);
            if (sl.n == VO_MAX_FUSED) {
                int32_t r = flush();
                if (r != VO_OK) return r;
            }
        } else {
            if (s->snap) {  // the steps queued so far must have run before the checkpoint copy
                int32_t r = flush();
                if (r != VO_OK) return r;
            }
            uni_checkpoint(s, ev == VO_EV_END);
            res_add(res, 0, ev == VO_EV_CHKPT ? s->n : 0, 0, ev == VO_EV_END ? s->n : 0, 0);
        }
    }
    if (calls_done) *calls_done = calls;
    return flush();
}

// ---- stage path ---------------------------------------------------------------------------------------------
int32_t ensure_K(vo_solver_s* s, int count) {
    while ((int)s->K.size() < count) {
        vo_ens k = nullptr;
        int32_t r = vo_ens_create(s->ctx, s->d, s->n, &k);
        if (r != VO_OK) return r;
        s->K.push_back(k);
    }
    return VO_OK;
}

template <class RHS, bool TAIL> void launch_pointwise(vo_ctx c, const double* x0, int64_t N, const StageArgs& sa, const RhsParams& rp, double* k_out, double* nx,
                                                       double* xe) {
    const unsigned grid = (unsigned)ceil_div(N, 128);
    if (c->arith == VO_ARITH_STRICT) stage_pointwise_kernel<RHS, true, TAIL><<<grid, 128, 0, c->stream>>>(x0, N, sa, rp, k_out, nx, xe);
    else stage_pointwise_kernel<RHS, false, TAIL><<<grid, 128, 0, c->stream>>>(x0, N, sa, rp, k_out, nx, xe);
}

// TMA-staged heat stage: compact the K's this launch reads (FAST non-tail stages drop zero coefficients; STRICT keeps
// them, like the reference), pick the pipeline depth so that ~200 KB of tiles are in flight per SM, dispatch on NK.
template <bool STRICT, bool TAIL, int NK>
int32_t launch_heat_tma_nk(vo_solver_s* s, const HeatArgs& ha_in, double* k_out, double* nx, double* xe) {
    vo_ctx c = s->ctx;
    auto k = stage_heat_tma_kernel<STRICT, TAIL, NK>;
    constexpr int bps = NK <= 3 ? 2 : 1;
    const size_t row_bytes = (size_t)(NK + 1) * HT_ROW * sizeof(double);
    HeatArgs ha = ha_in;
    ha.nst = (int)std::max<size_t>(2, std::min<size_t>(HT_STAGES_MAX, (size_t)(208 * 1024 / bps) / row_bytes));
    const size_t smem = (size_t)ha.nst * row_bytes;
    VO_CUDA(c, vo_ensure_smem_attr(c->device, (const void*)k, 216 * 1024));
    const int64_t tiles = ceil_div(s->d, HT_TILE);
    const int64_t iters = ceil_div(tiles, (int64_t)c->sm_count * bps);
    k<<<(unsigned)ceil_div(tiles, iters), HT_THREADS, smem, c->stream>>>(s->x->p, s->d, ha, k_out, nx, xe);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

template <bool TAIL> int32_t launch_heat_tma(vo_solver_s* s, const StageArgs& sa, double kappa, double* k_out, double* nx, double* xe) {
    const bool strict = s->ctx->arith == VO_ARITH_STRICT;
    HeatArgs ha;
    std::memset(&ha, 0, sizeof ha);
    ha.dt = sa.dt, ha.kappa = kappa, ha.use_err = sa.use_err;
    const int S = sa.s, nload = TAIL ? S - 1 : sa.i;
    int nk = 0;
    for (int j = 0; j < nload; ++j) {
        const bool in_stage = j < sa.i;
        if (!(strict || TAIL || sa.a[j] != 0.0)) continue;
        // STRICT / TAIL keep every term in order, so the first sa.i compacted rows are exactly the stage's terms
        ha.K[nk] = sa.K[j], ha.a[nk] = in_stage ? sa.a[j] : 0.0, ha.b[nk] = sa.b[j], ha.b_err[nk] = sa.b_err[j];
        ++nk;
    }
    ha.nterm = (strict || TAIL) ? sa.i : nk;
    ha.b_last = sa.b[S - 1], ha.b_err_last = sa.b_err[S - 1];
#define VO_HEAT_CASE(NK) \
    case NK: return strict ? launch_heat_tma_nk<true, TAIL, NK>(s, ha, k_out, nx, xe) : launch_heat_tma_nk<false, TAIL, NK>(s, ha, k_out, nx, xe);
    switch (nk) {
        VO_HEAT_CASE(0) VO_HEAT_CASE(1) VO_HEAT_CASE(2) VO_HEAT_CASE(3) VO_HEAT_CASE(4) VO_HEAT_CASE(5) VO_HEAT_CASE(6) VO_HEAT_CASE(7)
    }
#undef VO_HEAT_CASE
    return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "stage path: HEAT1D needs s <= 8");
}

template <bool TAIL> int32_t launch_stage_kernel(vo_solver_s* s, const StageArgs& sa, double* k_out, double* nx, double* xe) {
    vo_ctx c = s->ctx;
    const vo_rhs_s* r = s->rhs;
    const double* x0 = s->x->p;
    const RhsParams rp = make_rhs_params(r);
    switch (r->kind) {
        case VO_RHS_DIAG_LINEAR:
            switch (r->d) {
                case 1: launch_pointwise<RhsF<VO_RHS_DIAG_LINEAR, 1>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
                case 2: launch_pointwise<RhsF<VO_RHS_DIAG_LINEAR, 2>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
                case 3: launch_pointwise<RhsF<VO_RHS_DIAG_LINEAR, 3>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
                case 4: launch_pointwise<RhsF<VO_RHS_DIAG_LINEAR, 4>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
                default: return vo_fail(c, VO_ERR_UNSUPPORTED, "stage path: DIAG_LINEAR needs d <= 4");
            }
            break;
        case VO_RHS_HARMONIC2D: launch_pointwise<RhsF<VO_RHS_HARMONIC2D, 2>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
        case VO_RHS_LORENZ63: launch_pointwise<RhsF<VO_RHS_LORENZ63, 3>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
        case VO_RHS_VDP: launch_pointwise<RhsF<VO_RHS_VDP, 2>, TAIL>(c, x0, s->n, sa, rp, k_out, nx, xe); break;
        case VO_RHS_CUSTOM: {
            int32_t cr = launch_stage_custom(c, s->rhs, TAIL, x0, s->n, sa, rp, k_out, nx, xe);
            if (cr != VO_OK) return cr;
        } break;
        case VO_RHS_CUSTOM_STENCIL: {
            if (s->n != 1) return vo_fail(c, VO_ERR_UNSUPPORTED, "stage path: a user stencil runs on ONE grid state (N == 1)");
            int32_t cr = launch_stage_stencil_custom(c, s->rhs, TAIL, x0, s->d, sa, rp, k_out, nx, xe);
            if (cr != VO_OK) return cr;
        } break;
        case VO_RHS_HEAT1D: {
            const double kappa = r->shared[0];
            const bool strict = c->arith == VO_ARITH_STRICT;
            if (s->n == 1) {
                if (s->tab.s > 8) return vo_fail(c, VO_ERR_UNSUPPORTED, "stage path: HEAT1D needs s <= 8");
                if (s->d % 2 == 0 && s->d >= 4 * HT_TILE) {
                    return launch_heat_tma<TAIL>(s, sa, kappa, k_out, nx, xe);  // checks its own launch
                } else {
                    const int64_t tiles = ceil_div(s->d, HEAT_TILE);
                    const unsigned grid = (unsigned)std::min<int64_t>(tiles, (int64_t)c->sm_count * 8);
                    if (strict) stage_heat_kernel<true, TAIL><<<grid, HEAT_THREADS, 0, c->stream>>>(x0, s->d, sa, kappa, k_out, nx, xe);
                    else stage_heat_kernel<false, TAIL><<<grid, HEAT_THREADS, 0, c->stream>>>(x0, s->d, sa, kappa, k_out, nx, xe);
                }
            } else {
                const unsigned grid = (unsigned)ceil_div(s->d * s->n, 256);
                if (strict) stage_heat_ens_kernel<true, TAIL><<<grid, 256, 0, c->stream>>>(x0, s->d, s->n, sa, kappa, k_out, nx, xe);
                else stage_heat_ens_kernel<false, TAIL><<<grid, 256, 0, c->stream>>>(x0, s->d, s->n, sa, kappa, k_out, nx, xe);
            }
        } break;
        default: return vo_fail(c, VO_ERR_UNSUPPORTED, "stage path: unknown RHS");
    }
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

// One rk_step (rk.rs:90-155) through the stage kernels: s launches. K_out (nullable) receives all s stage
// derivatives; otherwise K_{s-1} never leaves registers.
int32_t stage_rk_step(vo_solver_s* s, double t, double dt, bool per_traj, double* nx, double* xe, vo_ens* K_out, int* launches) {
    const vo_tableau_s& tb = s->tab;
    const int S = tb.s;
    const bool want_err = tb.has_err && xe != nullptr;
    if (!K_out) {
        int32_t r = ensure_K(s, std::max(1, S - 1));
        if (r != VO_OK) return r;
    }
    StageArgs sa;
    std::memset(&sa, 0, sizeof sa);
    for (int j = 0; j < S; ++j) sa.K[j] = K_out ? K_out[j]->p : (j < (int)s->K.size() ? s->K[j]->p : nullptr);
    sa.s = S, sa.dt = dt;
    if (per_traj) sa.tv = s->ca.t, sa.dtv = s->dtv, sa.evv = s->evv;
    for (int i = 0; i < S; ++i) {
        const double* row = &tb.ac[i * S];
        sa.i = i, sa.c_i = row[i];
        sa.t_i = i == 0 ? t : t + row[i] * dt;  // rk.rs:119
        for (int j = 0; j < i; ++j) sa.a[j] = row[j];
        int32_t r;
        if (i < S - 1) {
            r = launch_stage_kernel<false>(s, sa, const_cast<double*>(sa.K[i]), nullptr, nullptr);
        } else {
            for (int j = 0; j < S; ++j) sa.b[j] = tb.b[j], sa.b_err[j] = tb.b_err[j];
            sa.use_err = want_err ? 1 : 0;
            r = launch_stage_kernel<true>(s, sa, K_out ? K_out[S - 1]->p : nullptr, nx, want_err ? xe : nullptr);
        }
        if (r != VO_OK) return r;
        if (launches) ++*launches;
    }
    return VO_OK;
}

// ---- whole-step path for the heat equation (rk_heat_fused.cuh) ------------------------------------------------
template <int S, bool STRICT> int32_t launch_heat_fused_a(vo_solver_s* s, const TableauDev& tb, const StageArgs& sa, double kappa, double* nx, double* xe) {
    vo_ctx c = s->ctx;
    constexpr int HS = (S + 1) & ~1, T = HF_WL - 2 * HS, WPB = HF_THREADS / 32, BPS = S <= 4 ? 2 : 1;
    if (s->d < 4 * HF_WL) return vo_fail(c, VO_ERR_UNSUPPORTED, "whole-step heat kernel: the state is shorter than four warp tiles");
    auto k = heat_fused_step_kernel<S, STRICT>;
    const size_t smem = (size_t)WPB * HF_NST * HF_WL * sizeof(double);
    VO_CUDA(c, vo_ensure_smem_attr(c->device, (const void*)k, smem));
    const int64_t tiles = ceil_div(s->d, T);                                    // warp tiles
    const int64_t iters = ceil_div(tiles, (int64_t)c->sm_count * BPS * WPB);    // per warp, all CTAs resident
    const int64_t warps = ceil_div(tiles, iters);
    k<<<(unsigned)ceil_div(warps, WPB), HF_THREADS, smem, c->stream>>>(s->x->p, s->d, tb, sa, kappa, nx, xe);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}
template <int S> int32_t launch_heat_fused(vo_solver_s* s, const TableauDev& tb, const StageArgs& sa, double kappa, double* nx, double* xe) {
    return s->ctx->arith == VO_ARITH_STRICT ? launch_heat_fused_a<S, true>(s, tb, sa, kappa, nx, xe) : launch_heat_fused_a<S, false>(s, tb, sa, kappa, nx, xe);
}

bool heat_fused_ok(const vo_solver_s* s) {
    return s->stage_path == 2 && s->rhs->kind == VO_RHS_HEAT1D && s->n == 1 && (s->tab.s == 4 || s->tab.s == 6 || s->tab.s == 7);
}

// One rk_step (rk.rs:90-155) of the single heat state in ONE launch.
int32_t heat_fused_rk_step(vo_solver_s* s, double dt, double* nx, double* xe, int* launches) {
    const vo_tableau_s& t = s->tab;
    const TableauDev tb = make_tableau_dev(t);
    StageArgs sa;
    std::memset(&sa, 0, sizeof sa);
    sa.s = t.s, sa.dt = dt, sa.use_err = (t.has_err && xe) ? 1 : 0;
    for (int j = 0; j < t.s; ++j) sa.b[j] = t.b[j], sa.b_err[j] = t.b_err[j];
    const double kappa = s->rhs->shared[0];
    int32_t r = VO_ERR_UNSUPPORTED;
    switch (t.s) {
        case 4: r = launch_heat_fused<4>(s, tb, sa, kappa, nx, xe); break;
        case 6: r = launch_heat_fused<6>(s, tb, sa, kappa, nx, xe); break;
        case 7: r = launch_heat_fused<7>(s, tb, sa, kappa, nx, xe); break;
    }
    if (r == VO_OK && launches) ++*launches;
    return r;
}

// handle_step_adaptive (ode.rs:311-334) for the shared scalars of a lock-step solver; true = rejected.
bool uni_controller(vo_solver_s* s, double dxn) {
    const double h = s->u_h;  // ode.rs:314
    s->u_dx_norm = dxn;
    const double f = s->rtol / dxn;                                                        // ode.rs:320
    const double fp_lim = std::fmin(std::fmax(s->alpha * std::pow(f, s->pw), 0.3), 2.0);   // ode.rs:321-323
    const double new_h = std::fmin(std::fmax(fp_lim * h, s->min_dt), s->max_dt);          // ode.rs:324
    s->u_prev_h = s->u_h, s->u_h = new_h;                                                  // ode.rs:326
    return f <= 1.0;                                                                       // ode.rs:328-330
}
// apply_step (ode.rs:402-428) of a Step / Reject event on the lock-step stage path
void uni_apply(vo_solver_s* s, int ev, double dt, vo_step_result* res, int launches) {
    if (ev == VO_EV_STEP) {
        std::swap(s->x, s->next_x);  // advance, ode.rs:184-188
        s->u_t += dt, s->u_accept += 1;
        res_add(res, s->n, 0, 0, 0, launches);
    } else {
        s->u_reject += 1;
        res_add(res, 0, 0, s->n, 0, launches);
    }
}

// Lock-step stage path: one event, controller on the host (the norm is read back for adaptive steps).
int32_t stage_uniform_event(vo_solver_s* s, bool adaptive, vo_step_result* res) {
    vo_ctx c = s->ctx;
    double dt = 0.0;
    int ev = uni_step_size(s, &dt);
    int launches = 0;
    if (s->try_pending) return vo_fail(c, VO_ERR_STATE, "a vo_adaptive_try is waiting for its vo_adaptive_handle");
    if (ev == VO_EV_STEP) {
        double* xe_p = use_err(s) ? s->x_err->p : nullptr;
        int32_t r = heat_fused_ok(s) ? heat_fused_rk_step(s, dt, s->next_x->p, xe_p, &launches)
                                     : stage_rk_step(s, s->u_t, dt, false, s->next_x->p, xe_p, nullptr, &launches);
        if (r != VO_OK) return r;
        if (adaptive) {
            double* out = (double*)c->dscratch;
            if (s->n != 1) return vo_fail(c, VO_ERR_UNSUPPORTED, "stage path: lock-step adaptive control needs N == 1");
            const int64_t launches_before = c->launches;
            r = s->norm_kind == VO_NORM_CUSTOM ? norm_custom_device(s->norm_fn, s->x_err->p, s->d, 1, 0, s->d, out, s->norm_partial, PARTIAL_CAP, true)
                                               : vo_norm_device(s->x_err, s->norm_kind, out, s->norm_partial, PARTIAL_CAP, true);
            if (r != VO_OK) return r;
            launches += (int)(c->launches - launches_before);
            VO_CUDA(c, cudaMemcpyAsync(c->pinned, out, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
            VO_CUDA(c, cudaStreamSynchronize(c->stream));
            if (uni_controller(s, *(double*)c->pinned)) ev = VO_EV_REJECT;
        }
        uni_apply(s, ev, dt, res, launches);
    } else {
        uni_checkpoint(s, ev == VO_EV_END);
        res_add(res, 0, ev == VO_EV_CHKPT ? s->n : 0, 0, ev == VO_EV_END ? s->n : 0, 0);
    }
    return VO_OK;
}

// Per-trajectory stage path: prepare -> s stage kernels (masked) -> norm/controller/commit. One event per call.
int32_t stage_pertraj_event(vo_solver_s* s, bool adaptive, int* launches) {
    vo_ctx c = s->ctx;
    if (s->d > 64 || s->rhs->kind == VO_RHS_HEAT1D || s->rhs->kind == VO_RHS_CUSTOM_STENCIL)
        return vo_fail(c, VO_ERR_UNSUPPORTED, "stage path: per-trajectory control needs a pointwise RHS with d <= 64");
    if (!s->evv) {
        if (vo_dmalloc(&s->evv, (size_t)s->n) != cudaSuccess || vo_dmalloc(&s->dtv, 8 * (size_t)s->n) != cudaSuccess)
            return vo_fail(c, VO_ERR_ALLOC, "stage path: event buffers");
    }
    const CtlShared cs = make_ctl_shared(s, adaptive ? 1 : 0, 1);
    const unsigned grid = (unsigned)ceil_div(s->n, 256);
    ctl_prepare_kernel<<<grid, 256, 0, c->stream>>>(s->ca, cs, s->n, s->evv, s->dtv);
    VO_CHECK_LAUNCH(c);
    ++*launches;
    int32_t r = stage_rk_step(s, 0.0, 0.0, true, s->next_x->p, use_err(s) ? s->x_err->p : nullptr, nullptr, launches);
    if (r != VO_OK) return r;
    const double* xe = use_err(s) ? s->x_err->p : nullptr;
    const double* dxn_pre = nullptr;
    if (adaptive && xe && s->norm_kind == VO_NORM_CUSTOM) {
        if (!s->dxn_pre && vo_dmalloc(&s->dxn_pre, 8 * (size_t)s->n) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "stage path: norm buffer");
        const int64_t before = c->launches;
        r = norm_custom_device(s->norm_fn, xe, s->d, s->n, 0, s->d, s->dxn_pre, s->norm_partial, PARTIAL_CAP, true);
        if (r != VO_OK) return r;
        *launches += (int)(c->launches - before);
        dxn_pre = s->dxn_pre;
    }
    if (c->arith == VO_ARITH_STRICT) ctl_commit_kernel<true><<<grid, 256, 0, c->stream>>>(s->x->p, s->next_x->p, xe, s->d, s->n, s->ca, cs, s->evv, s->dtv, s->ev_dev, dxn_pre);
    else ctl_commit_kernel<false><<<grid, 256, 0, c->stream>>>(s->x->p, s->next_x->p, xe, s->d, s->n, s->ca, cs, s->evv, s->dtv, s->ev_dev, dxn_pre);
    VO_CHECK_LAUNCH(c);
    ++*launches;
    return VO_OK;
}

// validate_adaptive (ode.rs:312, rk.rs:317-319) and the switch from lock-step to per-trajectory control.
int32_t prepare_mode(vo_solver_s* s, bool adaptive) {
    vo_ctx c = s->ctx;
    if (adaptive && !s->has_x_err) return vo_fail(c, VO_ERR_NOT_ADAPTIVE, "adaptive step validation failed");  // ode.rs:312
    if (adaptive && !s->tab.has_err)
        return vo_fail(c, VO_ERR_NOT_ADAPTIVE, "step_adaptive: the tableau has no b_err, so no error estimate is ever formed");
    if (s->uniform && adaptive && (use_small(s) || s->n > 1)) return materialize(s);
    return VO_OK;
}

// One call of step()/step_adaptive() for every trajectory (or k fused calls on the small path).
int32_t do_events(vo_solver_s* s, bool adaptive, int k, vo_step_result* res, int64_t* calls_done, bool read_back) {
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    int32_t pr = prepare_mode(s, adaptive);
    if (pr != VO_OK) return pr;
    const bool small = use_small(s);
    if (s->uniform) {
        if (small) return small_uniform_events(s, k, res, calls_done);
        if (calls_done) *calls_done = 1;
        if (s->u_done) return VO_OK;
        return stage_uniform_event(s, adaptive, res);
    }
    // per-trajectory control
    if (!adaptive && s->prev_h_stale)
        return vo_fail(c, VO_ERR_STATE,
                       "step() after step_adaptive() on per-trajectory control: call vo_solver_set_mixed_stepping(s, 1) before the first step_adaptive() "
                       "(by default the adaptive kernels keep prev_h, which only a checkpoint reads (ode.rs:192-195), up to date only where a checkpoint comes next)");
    int launches = 0;
    if (small) {
        const CtlShared cs = make_ctl_shared(s, adaptive ? 1 : 0, k);
        int32_t r = launch_small(s, &cs, nullptr);
        if (r != VO_OK) return r;
        // the two-trajectory control kernel is the only one with a lazy prev_h (the plan's shared-memory size is not needed here)
        const bool unrolled = s->tab.s == 4 || s->tab.s == 6 || s->tab.s == 7;
        if (cs.lazy_prev_h && small_plan(s->n, unrolled, (int)s->d, &cs).k == SK_CTL2W) s->prev_h_stale = true;
        launches = 1;
        if (calls_done) *calls_done = k;
    } else {
        int32_t r = stage_pertraj_event(s, adaptive, &launches);
        if (r != VO_OK) return r;
        if (calls_done) *calls_done = 1;
    }
    if (res) res->launches += launches;
    if (read_back) {
        EvSlot sum;
        int32_t r = ev_read(s, &sum);
        if (r != VO_OK) return r;
        s->n_done += (int64_t)sum.n_end;
        res_add(res, (int64_t)sum.n_step, (int64_t)sum.n_chkpt, (int64_t)sum.n_reject, (int64_t)sum.n_end, 0);
    }
    return VO_OK;
}

void finish_result(vo_solver_s* s, vo_step_result* res) {
    if (!res) return;
    res->n_active = s->uniform ? (s->u_done ? 0 : s->n) : s->n - s->n_done;
    res->state = res->n_active == 0 ? VO_STATE_DONE : VO_STATE_OK;
}

}  // namespace

static int32_t alloc_snapshots(vo_solver s) {
    vo_ctx c = s->ctx;
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    vo_dfree(s->snap), s->snap = nullptr;
    const size_t bytes = sizeof(double) * s->t_list.size() * (size_t)snap_stride(s);
    if (vo_dmalloc(&s->snap, bytes) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "vo_solver_enable_snapshots: cudaMalloc failed");
    VO_CUDA(c, cudaMemsetAsync(s->snap, 0, bytes, c->stream));
    return VO_OK;
}


extern "C" {

int32_t vo_rk_create(vo_ctx c, vo_tableau tableau, vo_rhs rhs, double t0, double tf, vo_ens x0, double h, vo_solver* out) {
    if (!c || !tableau || !rhs || !x0 || !out) return vo_fail(c, VO_ERR_BAD_ARG, "vo_rk_create: NULL argument");
    if (rhs->d != x0->d) return vo_fail(c, VO_ERR_SHAPE, "vo_rk_create: RHS dimension does not match the ensemble");
    for (int q = 0; q < rhs->np; ++q)
        if (rhs->per_traj[q] && rhs->per_traj_n[q] != x0->n) return vo_fail(c, VO_ERR_SHAPE, "vo_rk_create: per-trajectory parameter array length != N");
    DeviceGuard g(c->device);
    vo_solver s = new vo_solver_s();
    s->ctx = c, s->tab = *tableau, s->rhs = rhs, s->d = x0->d, s->n = x0->n;
    s->t0 = t0, s->tf = tf, s->h_init = h;
    s->t_list = {t0, tf};  // ode.rs:144
    s->u_t = t0, s->u_h = h, s->u_prev_h = h, s->u_tgt = 0;
    int32_t r = vo_ens_clone(x0, &s->x);                      // ODEData::new clones x0 into x and next_x (ode.rs:141-150)
    if (r == VO_OK) r = vo_ens_clone(x0, &s->next_x);
    if (r == VO_OK && tableau->has_err) r = vo_ens_clone(x0, &s->x_err);  // Some(x0.clone()), rk.rs:249
    if (r == VO_OK && vo_dmalloc(&s->ev_dev, sizeof(EvSlot) * VO_EV_SLOTS) != cudaSuccess) r = vo_fail(c, VO_ERR_ALLOC, "vo_rk_create: counters");
    if (r == VO_OK && cudaMallocHost(&s->ev_host, sizeof(EvSlot) * VO_EV_SLOTS) != cudaSuccess) r = vo_fail(c, VO_ERR_ALLOC, "vo_rk_create: pinned counters");
    if (r == VO_OK && vo_dmalloc(&s->norm_partial, sizeof(double) * PARTIAL_CAP) != cudaSuccess) r = vo_fail(c, VO_ERR_ALLOC, "vo_rk_create: norm scratch");
    if (r == VO_OK && (vo_dmalloc(&s->cst.flags, sizeof(uint32_t) * CHAIN_FLAGS) != cudaSuccess ||
                       cudaMemsetAsync(s->cst.flags, 0, sizeof(uint32_t) * CHAIN_FLAGS, c->stream) != cudaSuccess))
        r = vo_fail(c, VO_ERR_ALLOC, "vo_rk_create: chain flags");
    if (r == VO_OK) {
        cudaError_t e = cudaMemsetAsync(s->ev_dev, 0, sizeof(EvSlot) * VO_EV_SLOTS, c->stream);
        if (e != cudaSuccess) r = vo_fail(c, VO_ERR_CUDA, cudaGetErrorString(e));
    }
    if (r != VO_OK) {
        vo_solver_destroy(s);
        return r;
    }
    *out = s;
    return VO_OK;
}

int32_t vo_rk45_create(vo_ctx c, vo_rhs rhs, double t0, double tf, vo_ens x0, double h, vo_solver* out) {
    vo_tableau t = nullptr;
    int32_t r = vo_tableau_builtin(VO_TABLEAU_RKF45_REF, &t);  // rk.rs:250-254
    if (r != VO_OK) return r;
    r = vo_rk_create(c, t, rhs, t0, tf, x0, h, out);
    vo_tableau_destroy(t);  // the solver keeps its own copy
    return r;
}

int32_t vo_solver_destroy(vo_solver s) {
    if (!s) return VO_OK;
    DeviceGuard g(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    vo_ens_destroy(s->x), vo_ens_destroy(s->next_x), vo_ens_destroy(s->x_err);
    for (vo_ens k : s->K) vo_ens_destroy(k);
    free_ctl(s);
    vo_dfree(s->evv), vo_dfree(s->dtv), vo_dfree(s->norm_partial), vo_dfree(s->ev_dev), vo_dfree(s->t_list_dev), vo_dfree(s->cst.flags), vo_dfree(s->snap);
    cudaFreeHost(s->ev_host);
    vo_dfree(s->dxn_pre);
    if (s->norm_rhs) custom_rhs_release(s->norm_rhs), delete s->norm_rhs;
    delete s;
    return VO_OK;
}

int32_t vo_solver_no_adaptive(vo_solver s) {
    if (!s) return VO_ERR_BAD_ARG;
    s->has_x_err = false;  // rk.rs:233-237
    return VO_OK;
}

int32_t vo_solver_with_tolerance(vo_solver s, double atol, double rtol) {
    if (!s) return VO_ERR_BAD_ARG;
    if (!(atol > 0.0) || !(rtol > 0.0)) return vo_fail(s->ctx, VO_ERR_BAD_ARG, "Invalid tolerances: atol=" + std::to_string(atol) + ", rtol=" + std::to_string(rtol));
    s->atol = atol, s->rtol = rtol;  // ode.rs:298-306 (atol is stored and never read, as in the reference)
    return VO_OK;
}

int32_t vo_solver_with_step_range(vo_solver s, double dt_min, double dt_max) {
    if (!s) return VO_ERR_BAD_ARG;
    if (!(dt_min > 0.0) || !(dt_max > 0.0) || !(dt_max > dt_min))
        return vo_fail(s->ctx, VO_ERR_BAD_ARG, "Invalid step range: (" + std::to_string(dt_min) + ", " + std::to_string(dt_max) + ")");
    if (!s->uniform) return vo_fail(s->ctx, VO_ERR_STATE, "with_step_range: builder called after per-trajectory stepping began");
    s->min_dt = dt_min, s->max_dt = dt_max;
    const double h = std::sqrt(dt_min * dt_max);  // ode.rs:273-280: reset_step_size(sqrt(min*max))
    s->u_h = h, s->u_prev_h = h;
    return VO_OK;
}

int32_t vo_solver_with_init_step(vo_solver s, double h) {
    if (!s) return VO_ERR_BAD_ARG;
    if (h < s->min_dt || h > s->max_dt)  // ode.rs:287-296
        return vo_fail(s->ctx, VO_ERR_BAD_ARG, "Step " + std::to_string(h) + " is not inside the range (" + std::to_string(s->min_dt) + ", " + std::to_string(s->max_dt) + ")");
    if (!s->uniform) return vo_fail(s->ctx, VO_ERR_STATE, "with_init_step: builder called after per-trajectory stepping began");
    s->u_h = h, s->u_prev_h = h;
    return VO_OK;
}

int32_t vo_solver_set_t_list(vo_solver s, const double* t_list, int32_t n) {
    if (!s || !t_list || n < 1) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_t_list: bad argument");
    if (n > (int32_t)VO_WORD_TGT_MASK) return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "vo_solver_set_t_list: list too long");
    if (!s->uniform) return vo_fail(s->ctx, VO_ERR_STATE, "set_t_list: builder called after per-trajectory stepping began");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    s->t_list.assign(t_list, t_list + n);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    vo_dfree(s->t_list_dev), s->t_list_dev = nullptr;
    if (n > VO_INLINE_TLIST) {
        if (vo_dmalloc(&s->t_list_dev, sizeof(double) * n) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "vo_solver_set_t_list: cudaMalloc");
        VO_CUDA(c, cudaMemcpy(s->t_list_dev, t_list, sizeof(double) * n, cudaMemcpyHostToDevice));
    }
    if (s->snap) return alloc_snapshots(s);
    return VO_OK;
}

int32_t vo_solver_set_order_alpha(vo_solver s, double order, double alpha) {
    if (!s || !(order > 0.0)) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_order_alpha: bad argument");
    s->pw = 1.0 / order, s->alpha = alpha;  // `order.recip()`, ode.rs:120; with_alpha, ode.rs:128-131
    return VO_OK;
}

int32_t vo_solver_set_norm(vo_solver s, int32_t kind) {
    if (!s || kind < 0 || kind > VO_NORM_HYPOT) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_norm: bad norm kind");
    s->norm_kind = kind;
    if (s->norm_rhs) {  // back to a compiled-in norm: drop the run-time modules that carried the user's
        DeviceGuard g(s->ctx->device);
        cudaStreamSynchronize(s->ctx->stream);
        custom_rhs_release(s->norm_rhs), delete s->norm_rhs;
        s->norm_rhs = nullptr, s->cst.live = false;
    }
    s->norm_fn = nullptr;
    return VO_OK;
}

int32_t vo_solver_set_norm_custom(vo_solver s, vo_normfn f) {
    if (!s || !f) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_norm_custom: NULL argument");
    vo_ctx c = s->ctx;
    if (f->ctx != c) return vo_fail(c, VO_ERR_BAD_ARG, "vo_solver_set_norm_custom: the norm belongs to another ctx");
    DeviceGuard g(c->device);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    if (s->norm_rhs) custom_rhs_release(s->norm_rhs), delete s->norm_rhs, s->norm_rhs = nullptr;
    s->norm_kind = VO_NORM_CUSTOM, s->norm_fn = f, s->cst.live = false;
    // register-resident path: the control kernels are re-compiled with the functor in them (a compiled-in family through an alias)
    if (rhs_is_small(s->rhs)) s->norm_rhs = custom_rhs_with_norm(s->rhs, f);
    return VO_OK;
}

int32_t vo_solver_set_h_array(vo_solver s, const double* h_host, int64_t n) {
    if (!s || !h_host || n != s->n) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_h_array: bad argument");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    int32_t r = materialize(s);
    if (r != VO_OK) return r;
    VO_CUDA(c, cudaMemcpyAsync(s->ca.h, h_host, 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaMemcpyAsync(s->ca.prev_h, h_host, 8 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

int32_t vo_solver_set_events_per_launch(vo_solver s, int32_t k) {
    if (!s || k < 0 || k > (1 << 20)) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_events_per_launch: bad k");
    s->k_events = k;
    return VO_OK;
}

int32_t vo_solver_set_record_dx_norm(vo_solver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    s->record_dx_norm = on ? 1 : 0;
    return VO_OK;
}

int32_t vo_solver_set_blocked(vo_solver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    if (on) return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "vo_solver_set_blocked: the tile-blocked state layout was removed (measured no faster than the public layout)");
    return VO_OK;
}

int32_t vo_solver_set_mixed_stepping(vo_solver s, int32_t on) {
    if (!s) return VO_ERR_BAD_ARG;
    if (on && s->prev_h_stale) return vo_fail(s->ctx, VO_ERR_STATE, "vo_solver_set_mixed_stepping: adaptive steps have already run with the lazy prev_h");
    s->mixed_stepping = on ? 1 : 0;
    return VO_OK;
}

int32_t vo_solver_set_path(vo_solver s, int32_t path) {
    if (!s || path < 0 || path > 2) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_solver_set_path: path must be 0, 1 or 2");
    if (path == 2 && !(s->rhs->kind == VO_RHS_HEAT1D && s->n == 1 && (s->tab.s == 4 || s->tab.s == 6 || s->tab.s == 7)))
        return vo_fail(s->ctx, VO_ERR_UNSUPPORTED, "vo_solver_set_path: the whole-step path needs HEAT1D, one state (N = 1) and 4, 6 or 7 stages");
    s->stage_path = path;
    return VO_OK;
}

static int32_t step_impl(vo_solver s, bool adaptive, vo_step_result* res) {
    if (!s) return VO_ERR_BAD_ARG;
    if (res) std::memset(res, 0, sizeof *res);
    int32_t r = do_events(s, adaptive, 1, res, nullptr, true);
    if (r != VO_OK) return r;
    finish_result(s, res);
    return VO_OK;
}

int32_t vo_step(vo_solver s, vo_step_result* res) { return step_impl(s, false, res); }
int32_t vo_step_adaptive(vo_solver s, vo_step_result* res) { return step_impl(s, true, res); }

// AdaptiveODESolver::step_adaptive (ode.rs:336-344) in its two halves — try_step + the error norm, then handle_step_adaptive +
// apply_step — for a state that is ONE vector held in pieces by several solvers (slabs of a grid on several GPUs,
// vec-ode_b200/domain.py): every piece reports the accumulator of its own components [lo, hi), the caller combines them
// (sum or max over the pieces, any communicator) and hands the same global norm to every piece.
int32_t vo_adaptive_try(vo_solver s, int64_t lo, int64_t hi, double* acc, int32_t* event, vo_step_result* res) {
    if (!s || !acc || !event) return vo_fail(s ? s->ctx : nullptr, VO_ERR_BAD_ARG, "vo_adaptive_try: NULL argument");
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    if (!s->uniform || use_small(s) || s->n != 1) return vo_fail(c, VO_ERR_UNSUPPORTED, "vo_adaptive_try: a single state (N == 1) on the stage path");
    if (s->try_pending) return vo_fail(c, VO_ERR_STATE, "vo_adaptive_try: the previous attempt has not been handled");
    if (lo < 0 || hi > s->d || lo >= hi) return vo_fail(c, VO_ERR_SHAPE, "vo_adaptive_try: bad component range");
    if (s->norm_kind == VO_NORM_HYPOT) return vo_fail(c, VO_ERR_UNSUPPORTED, "vo_adaptive_try: L2, L1, Linf or a user-defined norm");
    int32_t r = prepare_mode(s, true);
    if (r != VO_OK) return r;
    *acc = 0.0;
    if (res) std::memset(res, 0, sizeof *res);
    if (s->u_done) {
        *event = VO_EV_END;
        finish_result(s, res);
        return VO_OK;
    }
    double dt = 0.0;
    const int ev = uni_step_size(s, &dt);
    *event = ev;
    if (ev != VO_EV_STEP) {  // Chkpt / End need no norm: done here, nothing to handle
        uni_checkpoint(s, ev == VO_EV_END);
        res_add(res, 0, ev == VO_EV_CHKPT ? s->n : 0, 0, ev == VO_EV_END ? s->n : 0, 0);
        finish_result(s, res);
        return VO_OK;
    }
    int launches = 0;
    r = heat_fused_ok(s) ? heat_fused_rk_step(s, dt, s->next_x->p, s->x_err->p, &launches)
                         : stage_rk_step(s, s->u_t, dt, false, s->next_x->p, s->x_err->p, nullptr, &launches);
    if (r != VO_OK) return r;
    vo_ens_s view;
    view.ctx = c, view.p = s->x_err->p + lo, view.d = hi - lo, view.n = 1, view.owns = false;
    double* out = (double*)c->dscratch;
    const int64_t before = c->launches;
    r = s->norm_kind == VO_NORM_CUSTOM ? norm_custom_device(s->norm_fn, view.p, view.d, 1, lo, s->d, out, s->norm_partial, PARTIAL_CAP, false)
                                       : vo_norm_device(&view, s->norm_kind, out, s->norm_partial, PARTIAL_CAP, false);
    if (r != VO_OK) return r;
    launches += (int)(c->launches - before);
    VO_CUDA(c, cudaMemcpyAsync(c->pinned, out, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    *acc = *(double*)c->pinned;
    s->try_pending = true, s->try_dt = dt, s->try_launches = launches;
    return VO_OK;
}

int32_t vo_adaptive_handle(vo_solver s, double dx_norm, vo_step_result* res) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    if (res) std::memset(res, 0, sizeof *res);
    if (!s->try_pending) return vo_fail(c, VO_ERR_STATE, "vo_adaptive_handle: no attempt is pending (vo_adaptive_try returned Chkpt / End, or was not called)");
    s->try_pending = false;
    const int ev = uni_controller(s, dx_norm) ? VO_EV_REJECT : VO_EV_STEP;
    uni_apply(s, ev, s->try_dt, res, s->try_launches);
    finish_result(s, res);
    return VO_OK;
}

int32_t vo_run(vo_solver s, int32_t adaptive, int64_t max_calls, vo_step_result* res) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_step_result acc;
    std::memset(&acc, 0, sizeof acc);
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    int64_t calls = 0;
    const bool adp = adaptive != 0;
    int32_t r = prepare_mode(s, adp);
    if (r != VO_OK) return r;
    // lock-step phase: no read-back is needed, the host knows every event
    while (s->uniform && !s->u_done && (max_calls <= 0 || calls < max_calls)) {
        int k = use_small(s) ? run_fusion(s) : 1;
        if (max_calls > 0) k = (int)std::min<int64_t>(k, max_calls - calls);
        int64_t done = 0;
        r = do_events(s, adp, k, &acc, &done, false);
        if (r != VO_OK) return r;
        calls += done;
    }
    if (!s->uniform) {
        // per-trajectory phase: launch a batch of sweeps, then read the counters once. Finished lanes exit on
        // their status word, so sweeps past the end of the slowest trajectory only cost 4 bytes per lane.
        int batch = 4;
        while (s->n_done < s->n && (max_calls <= 0 || calls < max_calls)) {
            for (int b = 0; b < batch && (max_calls <= 0 || calls < max_calls); ++b) {
                int k = use_small(s) ? run_fusion(s) : 1;
                if (max_calls > 0) k = (int)std::min<int64_t>(k, max_calls - calls);
                int64_t done = 0;
                r = do_events(s, adp, k, &acc, &done, false);
                if (r != VO_OK) return r;
                calls += done;
            }
            EvSlot sum;
            r = ev_read(s, &sum);
            if (r != VO_OK) return r;
            s->n_done += (int64_t)sum.n_end;
            res_add(&acc, (int64_t)sum.n_step, (int64_t)sum.n_chkpt, (int64_t)sum.n_reject, (int64_t)sum.n_end, 0);
            if (sum.n_stuck && sum.n_step == 0 && sum.n_chkpt == 0 && sum.n_end == 0) {
                // every live trajectory is rejecting at h == min_dt: the reference would spin forever (ode.rs:324-330)
                finish_result(s, &acc);
                acc.state = VO_STATE_ERR;
                if (res) *res = acc;
                return vo_fail(c, VO_ERR_STATE, "vo_run: all remaining trajectories are rejected at h == min_dt");
            }
            batch = std::min(batch * 2, 64);
        }
    }
    finish_result(s, &acc);
    if (res) *res = acc;
    return VO_OK;
}

int32_t vo_solver_enable_snapshots(vo_solver s) {
    if (!s) return VO_ERR_BAD_ARG;
    DeviceGuard g(s->ctx->device);
    return alloc_snapshots(s);
}

int32_t vo_solver_snapshot(vo_solver s, int32_t k, vo_ens* out) {
    if (!s || !out) return VO_ERR_BAD_ARG;
    if (!s->snap) return vo_fail(s->ctx, VO_ERR_STATE, "vo_solver_snapshot: snapshots are not enabled");
    if (k < 0 || k >= (int32_t)s->t_list.size()) return vo_fail(s->ctx, VO_ERR_BAD_ARG, "vo_solver_snapshot: index outside t_list");
    return vo_ens_wrap(s->ctx, s->snap + (size_t)k * snap_stride(s), s->d, s->n, out);
}

int32_t vo_step_many(const vo_solver* solvers, int32_t n, int32_t adaptive, int64_t rounds) {
    if (!solvers || n < 1 || rounds < 0) return VO_ERR_BAD_ARG;
    for (int i = 0; i < n; ++i)
        if (!solvers[i] || solvers[i]->ctx != solvers[0]->ctx) return vo_fail(solvers[0] ? solvers[0]->ctx : nullptr, VO_ERR_BAD_ARG, "vo_step_many: solvers must share one ctx");
    DeviceGuard g(solvers[0]->ctx->device);
    for (int i = 0; i < n; ++i) {
        int32_t r = prepare_mode(solvers[i], adaptive != 0);
        if (r != VO_OK) return r;
    }
    for (int64_t rd = 0; rd < rounds; ++rd)
        for (int i = 0; i < n; ++i) {
            vo_solver s = solvers[i];
            int32_t r = do_events(s, adaptive != 0, use_small(s) ? step_fusion(s) : 1, nullptr, nullptr, false);
            if (r != VO_OK) return r;
        }
    return VO_OK;
}

int32_t vo_current(vo_solver s, double* t_min, double* t_max, vo_ens* x) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    if (x) *x = s->x;
    if (t_min || t_max) {
        if (s->uniform) {
            if (t_min) *t_min = s->u_t;
            if (t_max) *t_max = s->u_t;
        } else {
            std::vector<double> t((size_t)s->n);
            VO_CUDA(c, cudaMemcpyAsync(t.data(), s->ca.t, 8 * (size_t)s->n, cudaMemcpyDeviceToHost, c->stream));
            VO_CUDA(c, cudaStreamSynchronize(c->stream));
            const auto mm = std::minmax_element(t.begin(), t.end());
            if (t_min) *t_min = *mm.first;
            if (t_max) *t_max = *mm.second;
        }
    }
    return VO_OK;
}

int32_t vo_solver_stats(vo_solver s, int64_t* accepted, int64_t* rejected, double* t, double* h, double* dx_norm, int32_t* status) {
    if (!s) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    const size_t n = (size_t)s->n;
    if (s->uniform) {
        for (size_t i = 0; i < n; ++i) {
            if (accepted) accepted[i] = s->u_accept;
            if (rejected) rejected[i] = s->u_reject;
            if (t) t[i] = s->u_t;
            if (h) h[i] = s->u_h;
            if (dx_norm) dx_norm[i] = s->u_dx_norm;
            if (status) status[i] = s->u_done ? VO_TRAJ_DONE : 0;
        }
        return VO_OK;
    }
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
    if (status) {
        VO_CUDA(c, cudaMemcpyAsync(tmp.data(), s->ca.word, 4 * n, cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(c, cudaStreamSynchronize(c->stream));
        for (size_t i = 0; i < n; ++i) status[i] = (int32_t)(tmp[i] >> VO_WORD_STATUS_SHIFT);
    }
    if (t) VO_CUDA(c, cudaMemcpyAsync(t, s->ca.t, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    if (h) VO_CUDA(c, cudaMemcpyAsync(h, s->ca.h, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    if (dx_norm) VO_CUDA(c, cudaMemcpyAsync(dx_norm, s->ca.dx_norm, 8 * n, cudaMemcpyDeviceToHost, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

int32_t vo_solver_reset(vo_solver s, vo_ens x0) {
    if (!s || !x0) return VO_ERR_BAD_ARG;
    if (x0->d != s->d || x0->n != s->n) return vo_fail(s->ctx, VO_ERR_SHAPE, "vo_solver_reset: shape mismatch");
    DeviceGuard g(s->ctx->device);
    int32_t r = vo_ens_copy(s->x, x0);
    if (r == VO_OK) r = vo_ens_copy(s->next_x, x0);
    if (r == VO_OK && s->x_err) r = vo_ens_copy(s->x_err, x0);
    if (r != VO_OK) return r;
    s->uniform = true, s->cst.live = false, s->prev_h_stale = false;
    s->u_t = s->t0, s->u_h = s->h_init, s->u_prev_h = s->h_init, s->u_tgt = 0, s->u_done = false;
    s->u_accept = s->u_reject = 0, s->u_dx_norm = 0.0, s->n_done = 0, s->try_pending = false;
    VO_CUDA(s->ctx, cudaMemsetAsync(s->ev_dev, 0, sizeof(EvSlot) * VO_EV_SLOTS, s->ctx->stream));
    std::memset(&s->ev_seen, 0, sizeof s->ev_seen);
    return VO_OK;
}

}  // extern "C"

// group.cu: this shard's totals into device memory, stream-ordered (no synchronisation)
int32_t vo_solver_local_stats(vo_solver s, unsigned long long* sums_dev, double* mm_dev) {
    if (!s || !sums_dev || !mm_dev) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    if (s->uniform) {
        const unsigned long long n = (unsigned long long)s->n;
        const unsigned long long h_sums[6] = {(unsigned long long)s->u_accept * n, (unsigned long long)s->u_reject * n, n, s->u_done ? n : 0ull, 0ull, 0ull};
        const double h_mm[2] = {s->u_t, -s->u_t};
        // small pageable sources are staged by the runtime before the call returns, so stack arrays are safe here
        VO_CUDA(c, cudaMemcpyAsync(sums_dev, h_sums, sizeof h_sums, cudaMemcpyHostToDevice, c->stream));
        VO_CUDA(c, cudaMemcpyAsync(mm_dev, h_mm, sizeof h_mm, cudaMemcpyHostToDevice, c->stream));
        return VO_OK;
    }
    const uint64_t epoch = c->epoch;
    VO_CUDA(c, cudaMemsetAsync(sums_dev, 0, 6 * sizeof(unsigned long long), c->stream));
    const long long lowest = (long long)0x8000000000000000ull;  // below the key of every double
    const long long init[2] = {lowest, lowest};
    VO_CUDA(c, cudaMemcpyAsync(mm_dev, init, sizeof init, cudaMemcpyHostToDevice, c->stream));
    ctl_stats_kernel<<<(unsigned)std::min<int64_t>(ceil_div(s->n, 256), (int64_t)c->sm_count * 4), 256, 0, c->stream>>>(s->ca, s->n, sums_dev, mm_dev);
    VO_CHECK_LAUNCH(c);
    ctl_stats_finish_kernel<<<1, 1, 0, c->stream>>>(sums_dev, mm_dev, (unsigned long long)s->n);
    VO_CHECK_LAUNCH(c);
    c->epoch = epoch;  // read-only with respect to the solver's state
    return VO_OK;
}

extern "C" {

int32_t vo_rk_try_step(vo_solver s, double t, double dt, vo_ens next_x, vo_ens x_err, vo_ens* K) {
    if (!s || !next_x) return VO_ERR_BAD_ARG;
    vo_ctx c = s->ctx;
    DeviceGuard g(c->device);
    if (next_x->d != s->d || next_x->n != s->n || (x_err && (x_err->d != s->d || x_err->n != s->n)))
        return vo_fail(c, VO_ERR_SHAPE, "vo_rk_try_step: shape mismatch");
    if (K)
        for (int j = 0; j < s->tab.s; ++j)
            if (!K[j] || K[j]->d != s->d || K[j]->n != s->n) return vo_fail(c, VO_ERR_SHAPE, "vo_rk_try_step: K must hold s ensembles of the solver's shape");
    return stage_rk_step(s, t, dt, false, next_x->p, (x_err && s->has_x_err) ? x_err->p : nullptr, K, nullptr);
}

int32_t vo_rhs_eval(vo_rhs r, double t, vo_ens x, vo_ens dx) {
    if (!r || !x || !dx) return VO_ERR_BAD_ARG;
    vo_ctx c = r->ctx;
    if (x->d != r->d || dx->d != x->d || dx->n != x->n) return vo_fail(c, VO_ERR_SHAPE, "vo_rhs_eval: shape mismatch");
    DeviceGuard g(c->device);
    // K_0 = f(t, x): stage 0 of the stage path on a throw-away solver view
    vo_solver_s tmp;
    tmp.ctx = c, tmp.rhs = r, tmp.d = x->d, tmp.n = x->n, tmp.x = x;
    tmp.tab.s = 2;
    StageArgs sa;
    std::memset(&sa, 0, sizeof sa);
    sa.s = 2, sa.i = 0, sa.t_i = t;
    int32_t rc = launch_stage_kernel<false>(&tmp, sa, dx->p, nullptr, nullptr);
    tmp.x = nullptr;
    return rc;
}

}  // extern "C"
