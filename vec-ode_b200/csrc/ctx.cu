// ctx.cu — contexts, ensembles (SoA device buffers), tableaux and RHS handles.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <set>
#include <tuple>

#include "common.cuh"

thread_local std::string g_vo_tls_err;

cudaError_t vo_ensure_smem_attr(int device, const void* func, size_t bytes) {
    if (bytes <= 48 * 1024) return cudaSuccess;
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> done;  // largest opt-in made so far per (device, function)
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = done[{device, func}];
    if (have >= bytes) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) have = bytes;
    return e;
}

// ------------------------------------------------------------------------------------------------
// Guarded device allocations (VECODE_GUARD=1), see common.cuh
// ------------------------------------------------------------------------------------------------
namespace {
constexpr size_t GUARD_BYTES = 4096;
constexpr unsigned char GUARD_PATTERN = 0xA5;
struct GuardBlock {
    void* base;
    size_t bytes;
    int device;
};
std::mutex g_guard_mu;
std::map<void*, GuardBlock> g_guard_live;  // user pointer -> block
int64_t g_guard_violations = 0;            // blocks found damaged so far (each block counted once per check)
int64_t g_guard_allocs = 0;

bool guard_on() {
    static const bool on = [] {
        const char* e = getenv("VECODE_GUARD");
        return e && e[0] && e[0] != '0';
    }();
    return on;
}

// Reads both guard zones of one block back; returns the number of damaged bytes and repairs them so that a later check reports new damage only.
size_t guard_damage(void* user, const GuardBlock& b) {
    std::vector<unsigned char> host(2 * GUARD_BYTES);
    DeviceGuard g(b.device);
    cudaDeviceSynchronize();
    unsigned char* lo = (unsigned char*)b.base;
    unsigned char* hi = (unsigned char*)user + b.bytes;
    if (cudaMemcpy(host.data(), lo, GUARD_BYTES, cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(host.data() + GUARD_BYTES, hi, GUARD_BYTES, cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    size_t bad = 0, first = 0;
    for (size_t i = 0; i < host.size(); ++i)
        if (host[i] != GUARD_PATTERN) {
            if (!bad) first = i;
            ++bad;
        }
    if (bad) {
        const long off = first < GUARD_BYTES ? (long)first - (long)GUARD_BYTES : (long)(first - GUARD_BYTES);
        fprintf(stderr, "vecode guard: %zu byte(s) written outside a %zu-byte device block; first at %s%ld\n", bad, b.bytes, first < GUARD_BYTES ? "start" : "end+",
                off);
        cudaMemset(lo, GUARD_PATTERN, GUARD_BYTES), cudaMemset(hi, GUARD_PATTERN, GUARD_BYTES);
    }
    return bad;
}
}  // namespace

cudaError_t vo_dmalloc_impl(void** p, size_t bytes) {
    if (!guard_on()) return cudaMalloc(p, bytes);
    // the user block keeps cudaMalloc's alignment (the front guard is a multiple of 512 bytes); its END is padded to 16 bytes only, so that
    // the rear guard starts as close behind the last element as the bulk-copy granularity of the kernels allows
    const size_t padded = (bytes + 15) & ~(size_t)15;
    void* base = nullptr;
    const cudaError_t e = cudaMalloc(&base, padded + 2 * GUARD_BYTES);
    if (e != cudaSuccess) return e;
    unsigned char* user = (unsigned char*)base + GUARD_BYTES;
    cudaMemset(base, GUARD_PATTERN, GUARD_BYTES);
    cudaMemset(user + bytes, GUARD_PATTERN, padded - bytes + GUARD_BYTES);
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(g_guard_mu);
    g_guard_live[user] = GuardBlock{base, bytes, dev};
    ++g_guard_allocs;
    *p = user;
    return cudaSuccess;
}

cudaError_t vo_dfree(void* p) {
    if (!p || !guard_on()) return cudaFree(p);
    GuardBlock b{};
    {
        std::lock_guard<std::mutex> lock(g_guard_mu);
        auto it = g_guard_live.find(p);
        if (it == g_guard_live.end()) return cudaFree(p);  // not ours (allocated before the switch was read: cannot happen) — plain free
        b = it->second;
        g_guard_live.erase(it);
    }
    if (guard_damage(p, b)) {
        std::lock_guard<std::mutex> lock(g_guard_mu);
        ++g_guard_violations;
    }
    DeviceGuard g(b.device);
    return cudaFree(b.base);
}

extern "C" int32_t vo_guard_enabled(void) { return guard_on() ? 1 : 0; }

// Checks the guard zones of every live block (synchronises the devices) and returns the number of damaged blocks found since the
// library was loaded, freed ones included; 0 when the switch is off. live_blocks (may be NULL): blocks currently allocated.
extern "C" int64_t vo_guard_check(int64_t* live_blocks) {
    if (live_blocks) *live_blocks = 0;
    if (!guard_on()) return 0;
    std::vector<std::pair<void*, GuardBlock>> blocks;
    {
        std::lock_guard<std::mutex> lock(g_guard_mu);
        blocks.assign(g_guard_live.begin(), g_guard_live.end());
    }
    int64_t found = 0;
    for (auto& kv : blocks) found += guard_damage(kv.first, kv.second) ? 1 : 0;
    std::lock_guard<std::mutex> lock(g_guard_mu);
    g_guard_violations += found;
    if (live_blocks) *live_blocks = (int64_t)g_guard_live.size();
    return g_guard_violations;
}

// Small device -> pinned-host read-backs (event counters) as a KERNEL that stores into the mapped host buffer, not as a copy: a
// cudaMemcpyAsync queues on the device-to-host copy engine behind whatever else is there — on the root of a sharded solve the
// 32 MB pieces of the final gather — and a solver's control loop then idles for the length of that transfer at every read-back.
__global__ void vo_small_readback_kernel(const unsigned long long* __restrict__ src, unsigned long long* __restrict__ dst_host, int n_words) {
    for (int i = threadIdx.x; i < n_words; i += blockDim.x) dst_host[i] = src[i];
}
cudaError_t vo_small_readback(vo_ctx c, void* host_pinned, const void* dev, size_t bytes) {
    vo_small_readback_kernel<<<1, 256, 0, c->stream>>>((const unsigned long long*)dev, (unsigned long long*)host_pinned, (int)(bytes / 8));
    return cudaGetLastError();
}

extern "C" {

int32_t vo_version(void) { return VO_VERSION; }

static int32_t ctx_create_impl(int32_t device, void* stream, int32_t urgency, vo_ctx* out);
int32_t vo_ctx_create(int32_t device, void* stream, vo_ctx* out) { return ctx_create_impl(device, stream, 0, out); }
int32_t vo_ctx_create_urgent(int32_t device, int32_t urgency, vo_ctx* out) { return ctx_create_impl(device, nullptr, urgency < 0 ? 0 : urgency, out); }

static int32_t ctx_create_impl(int32_t device, void* stream, int32_t urgency, vo_ctx* out) {
    if (!out) return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_ctx_create: out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return vo_fail(nullptr, VO_ERR_CUDA,
                       std::string("vo_ctx_create: no CUDA device available (") + cudaGetErrorString(e) +
                           "); this library has no CPU fallback");
    if (device < 0 || device >= ndev) return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_ctx_create: bad device ordinal");
    vo_ctx c = new vo_ctx_s();
    c->device = device;
    DeviceGuard g(device);
    if (stream) {
        c->stream = (cudaStream_t)stream;
    } else {
        int lo = 0, hi = 0;  // numerically lower = scheduled first; the range is [greatest, least]
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        const int prio = std::max(hi, lo - urgency);  // urgency 0 = the default (least) priority, each step one level up
        e = urgency > 0 ? cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio) : cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete c;
            return vo_fail(nullptr, VO_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
        }
        c->owns_stream = true;
    }
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    {   // staging buffers of upload/download come from the stream-ordered pool: keep freed blocks cached across
        // synchronisations instead of returning them to the driver every time (the default threshold is 0)
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
    }
    if (cudaMallocHost(&c->pinned, 4096) != cudaSuccess || vo_dmalloc(&c->dscratch, 4096) != cudaSuccess) {
        delete c;
        return vo_fail(nullptr, VO_ERR_ALLOC, "vo_ctx_create: scratch allocation failed");
    }
    *out = c;
    return VO_OK;
}

int32_t vo_ctx_destroy(vo_ctx c) {
    if (!c) return VO_OK;
    DeviceGuard g(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->owns_stream) cudaStreamDestroy(c->stream);
    cudaFreeHost(c->pinned);
    vo_dfree(c->dscratch);
    delete c;
    return VO_OK;
}

int32_t vo_ctx_sync(vo_ctx c) {
    if (!c) return VO_ERR_BAD_ARG;
    DeviceGuard g(c->device);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

// Stream-order `waiter` after everything enqueued so far on `other` (an event recorded on one stream, waited for on the other;
// no host synchronisation). Both contexts may sit on different devices.
int32_t vo_ctx_wait_for(vo_ctx waiter, vo_ctx other) {
    if (!waiter || !other) return VO_ERR_BAD_ARG;
    if (waiter == other || waiter->stream == other->stream) return VO_OK;
    cudaEvent_t ev = nullptr;
    {
        DeviceGuard g(other->device);
        VO_CUDA(other, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        cudaError_t e = cudaEventRecord(ev, other->stream);
        if (e != cudaSuccess) {
            cudaEventDestroy(ev);
            return vo_fail(other, VO_ERR_CUDA, std::string("cudaEventRecord: ") + cudaGetErrorString(e));
        }
    }
    DeviceGuard g(waiter->device);
    cudaError_t e = cudaStreamWaitEvent(waiter->stream, ev, 0);
    cudaEventDestroy(ev);  // released once the recorded work has completed
    vo_touch(waiter);
    if (e != cudaSuccess) return vo_fail(waiter, VO_ERR_CUDA, std::string("cudaStreamWaitEvent: ") + cudaGetErrorString(e));
    return VO_OK;
}

int32_t vo_ctx_fence(vo_ctx c) {
    if (!c) return VO_ERR_BAD_ARG;
    vo_touch(c);
    return VO_OK;
}

void* vo_ctx_stream(vo_ctx c) { return c ? (void*)c->stream : nullptr; }
const char* vo_last_error(vo_ctx c) { return c ? c->err.c_str() : g_vo_tls_err.c_str(); }
int64_t vo_ctx_launch_count(vo_ctx c) { return c ? c->launches : 0; }

int32_t vo_ctx_set_arith(vo_ctx c, int32_t mode) {
    if (!c || (mode != VO_ARITH_STRICT && mode != VO_ARITH_FAST)) return vo_fail(c, VO_ERR_BAD_ARG, "vo_ctx_set_arith: bad mode");
    c->arith = mode;
    return VO_OK;
}

// ---- ensembles -------------------------------------------------------------------------------------
int32_t vo_ens_create(vo_ctx c, int64_t d, int64_t n, vo_ens* out) {
    if (!c || !out || d <= 0 || n <= 0) return vo_fail(c, VO_ERR_BAD_ARG, "vo_ens_create: bad argument");
    DeviceGuard g(c->device);
    vo_ens e = new vo_ens_s();
    e->ctx = c, e->d = d, e->n = n, e->owns = true;
    if (vo_dmalloc(&e->p, sizeof(double) * d * n) != cudaSuccess) {
        cudaGetLastError();
        delete e;
        return vo_fail(c, VO_ERR_ALLOC, "vo_ens_create: cudaMalloc failed");
    }
    VO_CUDA(c, cudaMemsetAsync(e->p, 0, sizeof(double) * d * n, c->stream));
    *out = e;
    return VO_OK;
}

int32_t vo_ens_wrap(vo_ctx c, void* dptr, int64_t d, int64_t n, vo_ens* out) {
    if (!c || !out || !dptr || d <= 0 || n <= 0) return vo_fail(c, VO_ERR_BAD_ARG, "vo_ens_wrap: bad argument");
    if ((uintptr_t)dptr % 16 != 0) return vo_fail(c, VO_ERR_BAD_ARG, "vo_ens_wrap: pointer must be 16-byte aligned");
    vo_ens e = new vo_ens_s();
    e->ctx = c, e->d = d, e->n = n, e->owns = false, e->p = (double*)dptr;
    *out = e;
    return VO_OK;
}

int32_t vo_ens_copy(vo_ens dst, vo_ens src) {
    if (!dst || !src) return VO_ERR_BAD_ARG;
    if (dst->d != src->d || dst->n != src->n) return vo_fail(dst->ctx, VO_ERR_SHAPE, "vo_ens_copy: shape mismatch");
    DeviceGuard g(dst->ctx->device);
    VO_CUDA(dst->ctx, cudaMemcpyAsync(dst->p, src->p, sizeof(double) * src->elems(), cudaMemcpyDeviceToDevice, dst->ctx->stream));
    return VO_OK;
}

int32_t vo_ens_clone(vo_ens src, vo_ens* out) {
    if (!src || !out) return VO_ERR_BAD_ARG;
    int32_t r = vo_ens_create(src->ctx, src->d, src->n, out);
    if (r != VO_OK) return r;
    return vo_ens_copy(*out, src);
}

int32_t vo_ens_destroy(vo_ens e) {
    if (!e) return VO_OK;
    DeviceGuard g(e->ctx->device);
    if (e->owns && e->p) {
        cudaStreamSynchronize(e->ctx->stream);
        vo_dfree(e->p);
    }
    delete e;
    return VO_OK;
}

int32_t vo_ens_dims(vo_ens e, int64_t* d, int64_t* n) {
    if (!e) return VO_ERR_BAD_ARG;
    if (d) *d = e->d;
    if (n) *n = e->n;
    return VO_OK;
}
void* vo_ens_device_ptr(vo_ens e) { return e ? e->p : nullptr; }

}  // extern "C"

// AoS [N][d] <-> SoA [d][N] on the device. One thread per element, indexed so that the SoA side is
// coalesced; the AoS side of a warp covers a contiguous 32*d*8-byte span, so every sector is used.
__global__ void aos_to_soa_kernel(const double* __restrict__ aos, double* __restrict__ soa, int64_t d, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int64_t c = 0; c < d; ++c) soa[c * n + i] = aos[i * d + c];
}
__global__ void soa_to_aos_kernel(const double* __restrict__ soa, double* __restrict__ aos, int64_t d, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int64_t c = 0; c < d; ++c) aos[i * d + c] = soa[c * n + i];
}

extern "C" {

int32_t vo_ens_upload(vo_ens e, const double* host, int32_t layout) {
    if (!e || !host) return VO_ERR_BAD_ARG;
    vo_ctx c = e->ctx;
    DeviceGuard g(c->device);
    const size_t bytes = sizeof(double) * e->elems();
    if (layout == VO_LAYOUT_SOA || e->d == 1 || e->n == 1) {
        VO_CUDA(c, cudaMemcpyAsync(e->p, host, bytes, cudaMemcpyHostToDevice, c->stream));
    } else if (layout == VO_LAYOUT_AOS) {
        double* stage = nullptr;
        VO_CUDA(c, cudaMallocAsync(&stage, bytes, c->stream));
        VO_CUDA(c, cudaMemcpyAsync(stage, host, bytes, cudaMemcpyHostToDevice, c->stream));
        aos_to_soa_kernel<<<(unsigned)ceil_div(e->n, 256), 256, 0, c->stream>>>(stage, e->p, e->d, e->n);
        VO_CHECK_LAUNCH(c);
        VO_CUDA(c, cudaFreeAsync(stage, c->stream));
    } else {
        return vo_fail(c, VO_ERR_BAD_ARG, "vo_ens_upload: bad layout");
    }
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

int32_t vo_ens_download(vo_ens e, double* host, int32_t layout) {
    if (!e || !host) return VO_ERR_BAD_ARG;
    vo_ctx c = e->ctx;
    DeviceGuard g(c->device);
    const size_t bytes = sizeof(double) * e->elems();
    if (layout == VO_LAYOUT_SOA || e->d == 1 || e->n == 1) {
        VO_CUDA(c, cudaMemcpyAsync(host, e->p, bytes, cudaMemcpyDeviceToHost, c->stream));
    } else if (layout == VO_LAYOUT_AOS) {
        double* stage = nullptr;
        VO_CUDA(c, cudaMallocAsync(&stage, bytes, c->stream));
        soa_to_aos_kernel<<<(unsigned)ceil_div(e->n, 256), 256, 0, c->stream>>>(e->p, stage, e->d, e->n);
        VO_CHECK_LAUNCH(c);
        VO_CUDA(c, cudaMemcpyAsync(host, stage, bytes, cudaMemcpyDeviceToHost, c->stream));
        VO_CUDA(c, cudaFreeAsync(stage, c->stream));
    } else {
        return vo_fail(c, VO_ERR_BAD_ARG, "vo_ens_download: bad layout");
    }
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

// ---- tableaux (host-only objects) ------------------------------------------------------------------
int32_t vo_tableau_create(const double* ac, const double* b, const double* b_err, int32_t s, vo_tableau* out) {
    if (!ac || !b || !out || s < 1 || s > VO_MAX_STAGES)
        return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_tableau_create: need 1 <= s <= VO_MAX_STAGES and non-NULL ac, b");
    vo_tableau t = new vo_tableau_s();
    std::memset(t->ac, 0, sizeof t->ac), std::memset(t->b, 0, sizeof t->b), std::memset(t->b_err, 0, sizeof t->b_err);
    t->s = s;
    // stored with row stride s exactly like Array2::from_shape_vec((s,s), ..) (rk.rs:35-36)
    std::memcpy(t->ac, ac, sizeof(double) * s * s);
    std::memcpy(t->b, b, sizeof(double) * s);
    t->has_err = b_err != nullptr;
    if (b_err) std::memcpy(t->b_err, b_err, sizeof(double) * s);
    *out = t;
    return VO_OK;
}

int32_t vo_tableau_builtin(int32_t which, vo_tableau* out) {
    if (which == VO_TABLEAU_RKF45_REF) {
        // src/dat/mod.rs:9-27 as f64 division expressions; `-3544./2526.` is the reference's literal (:19).
        const double ac[36] = {0., 0., 0., 0., 0., 0.,
                               1. / 4., 1. / 4., 0., 0., 0., 0.,
                               3.0 / 32., 9.0 / 32., 3. / 8., 0., 0., 0.,
                               1932. / 2197., -7200. / 2197., 7296. / 2197., 12. / 13., 0., 0.,
                               439. / 216., -8., 3680. / 513., -845. / 4104., 1.0, 0.,
                               -8. / 27., 2., -3544. / 2526., 1859. / 4104., -11. / 40., 1.0 / 2.0};
        const double b[6] = {16. / 135., 0., 6656. / 12825., 28561. / 56430., -9. / 50., 2. / 55.};
        const double be[6] = {25. / 216., 0., 1408. / 2565., 2197. / 4104., -1. / 5., 0.};
        return vo_tableau_create(ac, b, be, 6, out);
    }
    if (which == VO_TABLEAU_RK4) {
        const double ac[16] = {0., 0., 0., 0., 1. / 2., 1. / 2., 0., 0., 0., 1. / 2., 1. / 2., 0., 0., 0., 1., 1.};
        const double b[4] = {1. / 6., 1. / 3., 1. / 3., 1. / 6.};
        return vo_tableau_create(ac, b, nullptr, 4, out);
    }
    if (which == VO_TABLEAU_DOPRI5) {
        const double ac[49] = {0., 0., 0., 0., 0., 0., 0.,
                               1. / 5., 1. / 5., 0., 0., 0., 0., 0.,
                               3. / 40., 9. / 40., 3. / 10., 0., 0., 0., 0.,
                               44. / 45., -56. / 15., 32. / 9., 4. / 5., 0., 0., 0.,
                               19372. / 6561., -25360. / 2187., 64448. / 6561., -212. / 729., 8. / 9., 0., 0.,
                               9017. / 3168., -355. / 33., 46732. / 5247., 49. / 176., -5103. / 18656., 1., 0.,
                               35. / 384., 0., 500. / 1113., 125. / 192., -2187. / 6784., 11. / 84., 1.};
        const double b4[7] = {5179. / 57600., 0., 7571. / 16695., 393. / 640., -92097. / 339200., 187. / 2100., 1. / 40.};
        const double b5[7] = {35. / 384., 0., 500. / 1113., 125. / 192., -2187. / 6784., 11. / 84., 0.};
        return vo_tableau_create(ac, b4, b5, 7, out);
    }
    return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_tableau_builtin: unknown tableau");
}

int32_t vo_tableau_num_stages(vo_tableau t) { return t ? t->s : VO_ERR_BAD_ARG; }

int32_t vo_tableau_get(vo_tableau t, double* ac, double* b, double* b_err, int32_t* has_err) {
    if (!t) return VO_ERR_BAD_ARG;
    if (ac) std::memcpy(ac, t->ac, sizeof(double) * t->s * t->s);
    if (b) std::memcpy(b, t->b, sizeof(double) * t->s);
    if (b_err && t->has_err) std::memcpy(b_err, t->b_err, sizeof(double) * t->s);
    if (has_err) *has_err = t->has_err ? 1 : 0;
    return VO_OK;
}

int32_t vo_tableau_destroy(vo_tableau t) {
    delete t;
    return VO_OK;
}

// ---- RHS handles -----------------------------------------------------------------------------------
static int rhs_num_params(int kind, int d) {
    switch (kind) {
        case VO_RHS_DIAG_LINEAR: return d;
        case VO_RHS_HARMONIC2D: return 1;
        case VO_RHS_LORENZ63: return 3;
        case VO_RHS_VDP: return 1;
        case VO_RHS_HEAT1D: return 1;
    }
    return -1;
}

int32_t vo_rhs_create(vo_ctx c, int32_t kind, int32_t d, vo_rhs* out) {
    if (!c || !out) return vo_fail(c, VO_ERR_BAD_ARG, "vo_rhs_create: bad argument");
    const int np = rhs_num_params(kind, d);
    if (np < 0) return vo_fail(c, VO_ERR_BAD_ARG, "vo_rhs_create: unknown RHS kind");
    const bool dim_ok = (kind == VO_RHS_DIAG_LINEAR && d >= 1 && d <= VO_MAX_PARAMS) || (kind == VO_RHS_HARMONIC2D && d == 2) ||
                        (kind == VO_RHS_LORENZ63 && d == 3) || (kind == VO_RHS_VDP && d == 2) || (kind == VO_RHS_HEAT1D && d >= 3);
    if (!dim_ok) return vo_fail(c, VO_ERR_SHAPE, "vo_rhs_create: dimension does not fit this RHS kind");
    vo_rhs r = new vo_rhs_s();
    r->ctx = c, r->kind = kind, r->d = d, r->np = np;
    for (int i = 0; i < VO_MAX_PARAMS; ++i) r->shared[i] = 0.0, r->per_traj[i] = nullptr, r->per_traj_n[i] = 0;
    // defaults: the textbook constants of each family
    if (kind == VO_RHS_DIAG_LINEAR) for (int i = 0; i < np; ++i) r->shared[i] = -1.0;
    if (kind == VO_RHS_HARMONIC2D) r->shared[0] = 1.0;
    if (kind == VO_RHS_LORENZ63) r->shared[0] = 10.0, r->shared[1] = 28.0, r->shared[2] = 8.0 / 3.0;
    if (kind == VO_RHS_VDP) r->shared[0] = 1.0;
    if (kind == VO_RHS_HEAT1D) r->shared[0] = 1.0;
    *out = r;
    return VO_OK;
}

int32_t vo_rhs_num_params(vo_rhs r) { return r ? r->np : VO_ERR_BAD_ARG; }

int32_t vo_rhs_set_param(vo_rhs r, int32_t idx, double value) {
    if (!r || idx < 0 || idx >= r->np) return vo_fail(r ? r->ctx : nullptr, VO_ERR_BAD_ARG, "vo_rhs_set_param: bad index");
    r->shared[idx] = value;
    if (r->per_traj[idx]) {
        DeviceGuard g(r->ctx->device);
        cudaStreamSynchronize(r->ctx->stream);
        vo_dfree(r->per_traj[idx]);
        r->per_traj[idx] = nullptr, r->per_traj_n[idx] = 0;
    }
    return VO_OK;
}

int32_t vo_rhs_set_param_array(vo_rhs r, int32_t idx, const double* host, int64_t n) {
    if (!r || !host || idx < 0 || idx >= r->np || n <= 0)
        return vo_fail(r ? r->ctx : nullptr, VO_ERR_BAD_ARG, "vo_rhs_set_param_array: bad argument");
    vo_ctx c = r->ctx;
    DeviceGuard g(c->device);
    if (r->per_traj[idx] && r->per_traj_n[idx] != n) {
        cudaStreamSynchronize(c->stream);
        vo_dfree(r->per_traj[idx]);
        r->per_traj[idx] = nullptr;
    }
    if (!r->per_traj[idx]) {
        if (vo_dmalloc(&r->per_traj[idx], sizeof(double) * n) != cudaSuccess) return vo_fail(c, VO_ERR_ALLOC, "vo_rhs_set_param_array: cudaMalloc failed");
        r->per_traj_n[idx] = n;
    }
    VO_CUDA(c, cudaMemcpyAsync(r->per_traj[idx], host, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return VO_OK;
}

int32_t vo_rhs_destroy(vo_rhs r) {
    if (!r) return VO_OK;
    DeviceGuard g(r->ctx->device);
    cudaStreamSynchronize(r->ctx->stream);
    for (int i = 0; i < VO_MAX_PARAMS; ++i)
        if (r->per_traj[i]) vo_dfree(r->per_traj[i]);
    if (r->kind == VO_RHS_CUSTOM) custom_rhs_release(r);
    delete r;
    return VO_OK;
}

}  // extern "C"
