// common.cuh — handle definitions, error plumbing and arithmetic-mode helpers shared by all kernels.
#pragma once
#ifdef __CUDACC_RTC__
// run-time compilation of a user RHS (nvrtc_rhs.cu): device-side definitions only, no host headers
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
#else
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#endif

#include "../../include/vecode_b200.h"

#define VO_MAX_PARAMS 8
#ifndef __CUDACC_RTC__
// ------------------------------------------------------------------------------------------------
// Handles
// ------------------------------------------------------------------------------------------------
struct vo_ctx_s {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    int arith = VO_ARITH_STRICT;
    int sm_count = 148;
    int64_t launches = 0;
    // Bumped by every library call that enqueues work on the stream EXCEPT the chained register-resident launches of
    // solver.cu (and by vo_ctx_fence, for work the caller enqueues on the stream behind the library's back). A solver may
    // chain its next launch to its previous one only while the epoch has not moved in between (pipe::Chain).
    uint64_t epoch = 1;
    std::string err;
    // small pinned scratch for result read-back and a device mirror
    void* pinned = nullptr;   // 4 KiB
    void* dscratch = nullptr; // 4 KiB
};

struct vo_ens_s {
    vo_ctx ctx = nullptr;
    double* p = nullptr;
    int64_t d = 0, n = 0;
    bool owns = true;
    int64_t elems() const { return d * n; }
};

struct vo_tableau_s {
    int s = 0;
    bool has_err = false;
    double ac[VO_MAX_STAGES * VO_MAX_STAGES];
    double b[VO_MAX_STAGES];
    double b_err[VO_MAX_STAGES];
};

struct vo_rhs_s {
    vo_ctx ctx = nullptr;
    int kind = 0, d = 0, np = 0;
    double shared[VO_MAX_PARAMS];      // shared value of each parameter
    double* per_traj[VO_MAX_PARAMS];   // device array or nullptr
    int64_t per_traj_n[VO_MAX_PARAMS];
    std::string body;                  // VO_RHS_CUSTOM: source of the RHS statements
    std::map<int, void*> modules;      // VO_RHS_CUSTOM: compiled modules keyed by (stage count, arithmetic mode)
    int radius = 0;                    // VO_RHS_CUSTOM_STENCIL: the stencil reaches `radius` grid points to each side
    int alias_kind = -1;               // >= 0: a compiled-in family re-compiled at run time (RhsCustom = RhsF<alias_kind, d>) to take a user norm
    std::string norm_src;              // source of the VoUserNorm functor compiled into this RHS's modules (vo_solver_set_norm_custom)
};
// Device allocations of the library (ctx.cu). Ordinary cudaMalloc / cudaFree unless the process runs with VECODE_GUARD=1: then every
// allocation sits between two 4 KiB guard zones filled with a byte pattern, checked when the block is freed and by vo_guard_check —
// a write past either end of a state, control or scratch array by any kernel shows up as a violation (tests/conftest.py asserts zero
// after every GPU test when the switch is on). compute-sanitizer is closed on the GPU pool; this is the library's own bounds check.
cudaError_t vo_dmalloc_impl(void** p, size_t bytes);
cudaError_t vo_dfree(void* p);
template <class T> static inline cudaError_t vo_dmalloc(T** p, size_t bytes) { return vo_dmalloc_impl((void**)p, bytes); }
cudaError_t vo_small_readback(vo_ctx c, void* host_pinned, const void* dev, size_t bytes);  // ctx.cu: bytes % 8 == 0, pinned (mapped) destination
void custom_rhs_release(vo_rhs_s* r);  // nvrtc_rhs.cu
// user-defined norm (nvrtc_rhs.cu, norm_custom.cuh): the functor's source and the reduction kernels compiled from it
struct vo_normfn_s {
    vo_ctx ctx = nullptr;
    std::string map_body, finish_body;
    int join = 0;
    void* module[2] = {nullptr, nullptr};  // per arithmetic mode (strict modules are compiled with --fmad=false)
    void* fn[2][3] = {};                   // small / partial / final
    std::mutex mu;                         // contexts may be driven from several host threads (pipeline.py): the lazy compile is serialised
};
std::string norm_source(const vo_normfn_s* f);
// norm of x = [d][n] (components i_off .. i_off + d of a d_total-component vector) into out_dev[n]; finish = false leaves the accumulator
int32_t norm_custom_device(vo_normfn_s* f, const double* x, int64_t d, int64_t n, int64_t i_off, int64_t d_total, double* out_dev, double* partial_dev,
                           int partial_cap, bool finish);
// a private RHS handle whose run-time modules carry the user's norm (for a compiled-in family: the family re-compiled with it)
vo_rhs_s* custom_rhs_with_norm(const vo_rhs_s* base, const vo_normfn_s* f);
// run-time compiled generator of the exponential integrators (nvrtc_rhs.cu): module + kernel handle for exp_step_kernel<n, M, 16, user GEN>,
// or exp_small_kernel<n, M, user GEN> for n <= VO_EXP_SMALL_MAX_N
#define VO_EXP_SMALL_MAX_N 8
int32_t rtc_exp_module(vo_ctx c, const std::string& body, const std::string& norm_src, int ndim, int M, size_t smem, void** module_out, void** fn_out);
int32_t rtc_exp_launch(vo_ctx c, void* fn, unsigned grid, unsigned block, size_t smem, void** args);
void rtc_exp_unload(void* module);

#endif  // !__CUDACC_RTC__

// Device-side view of the RHS parameters, passed by value to kernels.
struct RhsParams {
    double shared[VO_MAX_PARAMS];
    const double* per_traj[VO_MAX_PARAMS];
};

// Device-side tableau, passed by value (constant bank): compile-time-unrolled indices become c[0x0][..] operands.
struct TableauDev {
    double ac[VO_MAX_STAGES * VO_MAX_STAGES];
    double b[VO_MAX_STAGES];
    double b_err[VO_MAX_STAGES];
    int s;
    int has_err;
    // First-same-as-last structure, detected on the host bit for bit: bit 0 set <=> b_err[j] == ac[s-1][j] for every j < s-1,
    // bit 1 the same for b. The first s-1 terms of that final combination are then the very operations that formed the last
    // stage's argument, in the same order, so the kernels reuse that partial sum instead of recomputing it (Dormand-Prince:
    // the propagated 5th-order solution is stage 7's argument plus the term b_err[6] * K_7 — kept, zero or not).
    int reuse;
};

#ifndef __CUDACC_RTC__
// ------------------------------------------------------------------------------------------------
// Errors
// ------------------------------------------------------------------------------------------------
extern thread_local std::string g_vo_tls_err;

static inline int32_t vo_fail(vo_ctx ctx, int32_t code, const std::string& msg) {
    if (ctx) ctx->err = msg;
    g_vo_tls_err = msg;
    return code;
}

static inline void vo_touch(vo_ctx ctx) {
    if (ctx) ctx->epoch++;
}

#define VO_CUDA(ctx, call)                                                                              \
    do {                                                                                                \
        vo_touch(ctx);                                                                                  \
        cudaError_t _e = (call);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return vo_fail((ctx), VO_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));     \
    } while (0)

#define VO_CHECK_LAUNCH(ctx)                                                                            \
    do {                                                                                                \
        cudaError_t _e = cudaGetLastError();                                                            \
        if (_e != cudaSuccess)                                                                          \
            return vo_fail((ctx), VO_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(_e)); \
        (ctx)->launches++;                                                                              \
        (ctx)->epoch++;                                                                                 \
    } while (0)

// the chained register-resident launches themselves: they touch only their own solver's state, so they leave the epoch alone
#define VO_CHECK_LAUNCH_CHAINED(ctx)                                                                    \
    do {                                                                                                \
        cudaError_t _e = cudaGetLastError();                                                            \
        if (_e != cudaSuccess)                                                                          \
            return vo_fail((ctx), VO_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(_e)); \
        (ctx)->launches++;                                                                              \
    } while (0)

// Opt a kernel into more than 48 KB of dynamic shared memory. The attribute is per device and per function, and contexts on
// several devices may be driven from different host threads, so what has been set is remembered per (device, function).
cudaError_t vo_ensure_smem_attr(int device, const void* func, size_t bytes);

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

#endif  // !__CUDACC_RTC__

// ------------------------------------------------------------------------------------------------
// Arithmetic modes. STRICT: explicit round-to-nearest multiply and add (never contracted by nvcc), the
// reference's operation order. FAST: ordinary operators, nvcc is free to emit DFMA.
// ------------------------------------------------------------------------------------------------
template <bool STRICT> struct Ar {
    static __device__ __forceinline__ double mul(double a, double b) { return STRICT ? __dmul_rn(a, b) : a * b; }
    static __device__ __forceinline__ double add(double a, double b) { return STRICT ? __dadd_rn(a, b) : a + b; }
    static __device__ __forceinline__ double sub(double a, double b) { return STRICT ? __dsub_rn(a, b) : a - b; }
    // y + (k*x)   (src/impls/ndarray.rs:23)
    static __device__ __forceinline__ double axpy(double y, double k, double x) {
        return STRICT ? __dadd_rn(y, __dmul_rn(k, x)) : fma(k, x, y);
    }
};

#ifndef __CUDACC_RTC__
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
#endif
