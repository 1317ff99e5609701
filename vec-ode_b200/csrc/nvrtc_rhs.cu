// nvrtc_rhs.cu — user-defined right-hand sides: the C-ABI replacement of the reference's RHS closure
// `f: FnMut(T, &V, &mut V) -> Result<(),()>` (src/base/rk.rs:97; called at rk.rs:111 and :127).
//
// A closure cannot cross a C ABI into device code, so the caller hands over the SOURCE of its statements. It is wrapped
// into a functor with the same shape as the compiled-in families of rhs.cuh and compiled at run time (NVRTC, sm_100a)
// together with the very kernel templates the built-in families use — the headers are embedded in this shared object —
// so a user RHS runs fused inside the register-resident whole-attempt kernels (rk_small.cuh, rk_small2.cuh) and inside
// the stage-path kernel (rk_stage_pointwise.cuh) exactly like a built-in one. One module per (stage count, arithmetic
// mode), compiled on first use and cached on the vo_rhs. VO_ARITH_STRICT modules are compiled with --fmad=false, so a
// plain `a*b + c` in the body stays a separate multiply and add like the reference's Rust.
//
// libnvrtc is dlopen'ed on first use and the CUDA driver entry points are taken from the runtime
// (cudaGetDriverEntryPoint), so the library still loads — and every other path still works — on a machine without them.
#include <cuda.h>
#include <dlfcn.h>
#include <nvrtc.h>

#include <cstring>
#include <mutex>

#include "norm_custom.cuh"
#include "rk_small_launch.cuh"
#include "rk_stage_pointwise.cuh"
#include "rk_stage_stencil.cuh"

namespace {

struct Header {
    const char* name;
    const char* text;
};
const Header RTC_HEADERS[] = {
#include "rtc_headers.inc"
};
constexpr int N_HEADERS = (int)(sizeof(RTC_HEADERS) / sizeof(RTC_HEADERS[0]));

// ---- libnvrtc, loaded lazily -------------------------------------------------------------------------------------
struct Nvrtc {
    void* so = nullptr;
    decltype(&nvrtcCreateProgram) createProgram = nullptr;
    decltype(&nvrtcDestroyProgram) destroyProgram = nullptr;
    decltype(&nvrtcCompileProgram) compileProgram = nullptr;
    decltype(&nvrtcAddNameExpression) addNameExpression = nullptr;
    decltype(&nvrtcGetLoweredName) getLoweredName = nullptr;
    decltype(&nvrtcGetCUBINSize) getCUBINSize = nullptr;
    decltype(&nvrtcGetCUBIN) getCUBIN = nullptr;
    decltype(&nvrtcGetProgramLogSize) getProgramLogSize = nullptr;
    decltype(&nvrtcGetProgramLog) getProgramLog = nullptr;
    decltype(&nvrtcGetErrorString) getErrorString = nullptr;
};

bool nvrtc_load(Nvrtc** out, std::string& err) {
    static Nvrtc nv;
    static std::once_flag once;
    static std::string load_err;
    std::call_once(once, [] {
        const char* names[] = {getenv("VECODE_NVRTC"), "libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"};
        for (const char* n : names) {
            if (!n || !*n) continue;
            nv.so = dlopen(n, RTLD_NOW | RTLD_LOCAL);
            if (nv.so) break;
        }
        if (!nv.so) {
            load_err = "user RHS: libnvrtc could not be loaded (set VECODE_NVRTC to its path)";
            return;
        }
#define VO_NVRTC_SYM(field, sym)                                            \
    nv.field = reinterpret_cast<decltype(nv.field)>(dlsym(nv.so, #sym));    \
    if (!nv.field) load_err = std::string("user RHS: libnvrtc lacks ") + #sym;
        VO_NVRTC_SYM(createProgram, nvrtcCreateProgram)
        VO_NVRTC_SYM(destroyProgram, nvrtcDestroyProgram)
        VO_NVRTC_SYM(compileProgram, nvrtcCompileProgram)
        VO_NVRTC_SYM(addNameExpression, nvrtcAddNameExpression)
        VO_NVRTC_SYM(getLoweredName, nvrtcGetLoweredName)
        VO_NVRTC_SYM(getCUBINSize, nvrtcGetCUBINSize)
        VO_NVRTC_SYM(getCUBIN, nvrtcGetCUBIN)
        VO_NVRTC_SYM(getProgramLogSize, nvrtcGetProgramLogSize)
        VO_NVRTC_SYM(getProgramLog, nvrtcGetProgramLog)
        VO_NVRTC_SYM(getErrorString, nvrtcGetErrorString)
#undef VO_NVRTC_SYM
    });
    if (!load_err.empty()) {
        err = load_err;
        return false;
    }
    *out = &nv;
    return true;
}

// ---- driver entry points through the runtime ---------------------------------------------------------------------
struct Driver {
    decltype(&cuModuleLoadData) moduleLoadData = nullptr;
    decltype(&cuModuleUnload) moduleUnload = nullptr;
    decltype(&cuModuleGetFunction) moduleGetFunction = nullptr;
    decltype(&cuLaunchKernelEx) launchKernelEx = nullptr;
    decltype(&cuFuncSetAttribute) funcSetAttribute = nullptr;
    decltype(&cuOccupancyMaxActiveBlocksPerMultiprocessor) occupancy = nullptr;
    decltype(&cuGetErrorString) getErrorString = nullptr;
};

bool driver_load(Driver** out, std::string& err) {
    static Driver dr;
    static std::once_flag once;
    static std::string load_err;
    std::call_once(once, [] {
        auto get = [&](const char* sym, void** fn) {
            cudaDriverEntryPointQueryResult st;
            if (cudaGetDriverEntryPoint(sym, fn, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess || !*fn)
                load_err = std::string("user RHS: CUDA driver entry point not available: ") + sym;
        };
        get("cuModuleLoadData", (void**)&dr.moduleLoadData);
        get("cuModuleUnload", (void**)&dr.moduleUnload);
        get("cuModuleGetFunction", (void**)&dr.moduleGetFunction);
        get("cuLaunchKernelEx", (void**)&dr.launchKernelEx);
        get("cuFuncSetAttribute", (void**)&dr.funcSetAttribute);
        get("cuOccupancyMaxActiveBlocksPerMultiprocessor", (void**)&dr.occupancy);
        get("cuGetErrorString", (void**)&dr.getErrorString);
        cudaGetLastError();
    });
    if (!load_err.empty()) {
        err = load_err;
        return false;
    }
    *out = &dr;
    return true;
}

std::string cu_msg(Driver* dr, CUresult e) {
    const char* s = nullptr;
    if (dr->getErrorString(e, &s) != CUDA_SUCCESS || !s) return "CUDA driver error " + std::to_string((int)e);
    return s;
}

// ---- one compiled module -----------------------------------------------------------------------------------------
// function tables: a register-resident module's is indexed by SmallKernel (rk_small_launch.cuh), a stage-path module's by
enum { K_STAGE, K_STAGE_TAIL, K_STAGE_COUNT };
// stencil modules: the two plain kernels, then the TMA-staged ones indexed by (tail, number of stage-derivative rows read)
constexpr int K_STENCIL_TMA = 2, K_FN_MAX = 2 + 2 * 8;
static_assert(K_FN_MAX >= SK_COUNT, "CustomModule::fn too small");
constexpr int STAGE_MODULE = -1;  // `S` key of the stage-path module (it does not depend on the stage count)

struct CustomModule {
    CUmodule mod = nullptr;
    CUfunction fn[K_FN_MAX] = {};
    int bps[K_FN_MAX] = {};  // resident CTAs per SM at the shared-memory size last queried
    size_t bps_smem[K_FN_MAX] = {};
};

std::string rtc_source(const vo_rhs_s* r, bool stage_module) {
    const int d = r->d, np = r->np;
    if (r->kind == VO_RHS_CUSTOM_STENCIL) {  // a grid stencil: the fused per-stage kernel of rk_stage_stencil.cuh
        std::string st = "#include \"rk_stage_stencil.cuh\"\nstruct StencilCustom {\n    static constexpr int R = " + std::to_string(r->radius) +
                         ", NP = " + std::to_string(np > 0 ? np : 1) + ";\n";
        st += "    template <bool STRICT> static __device__ __forceinline__ double eval(const double t, const long long j, const long long d, const double (&u)[2 * R + 1], "
              "const double (&p)[NP]) {\n        double du = 0.0;\n        {\n#line 1 \"rhs_body\"\n" + r->body + "\n        }\n        return du;\n    }\n};\n";
        return st;
    }
    std::string s = r->norm_src;  // the VoUserNorm functor, if any: non-dependent in err_norm, so it comes before the templates
    s += stage_module ? "#include \"rk_stage_pointwise.cuh\"\n" : "#include \"rk_small2.cuh\"\n";
    if (r->alias_kind >= 0) return s + "using RhsCustom = RhsF<" + std::to_string(r->alias_kind) + ", " + std::to_string(d) + ">;\n";
    s += "struct RhsCustom {\n    static constexpr int D = " + std::to_string(d) + ", NP = " + std::to_string(np > 0 ? np : 1) + ";\n";
    s += "    template <bool STRICT> static __device__ __forceinline__ void eval(const double t, const double (&x)[D], double (&dx)[D], const double (&p)[NP]) {\n";
    s += "#line 1 \"rhs_body\"\n" + r->body + "\n    }\n};\n";
    return s;
}

std::vector<std::string> kernel_names(int S, bool strict, bool stage_module, bool stencil = false) {
    const std::string st = strict ? "true" : "false", ss = std::to_string(S);
    if (stencil) {
        std::vector<std::string> v = {"stage_stencil_kernel<StencilCustom, " + st + ", false>", "stage_stencil_kernel<StencilCustom, " + st + ", true>"};
        if (S == 1)  // `S` doubles as "with the TMA-staged kernels" for a stencil module (radius <= 4)
            for (int tail = 0; tail < 2; ++tail)
                for (int nk = 0; nk < 8; ++nk)
                    v.push_back("stage_stencil_tma_kernel<StencilCustom, " + st + ", " + (tail ? "true" : "false") + ", " + std::to_string(nk) + ">");
        return v;
    }
    if (stage_module) return {"stage_pointwise_kernel<RhsCustom, " + st + ", false>", "stage_pointwise_kernel<RhsCustom, " + st + ", true>"};
    std::vector<std::string> v(SK_COUNT);
    v[SK_FIXED2W] = S > 0 ? "rk_fixed2w_staged_kernel<RhsCustom, " + ss + ", " + st + ">" : "";  // unrolled stage counts only, as in launch_one
    v[SK_FIXED_STAGED] = "rk_fixed_staged_kernel<RhsCustom, " + ss + ", " + st + ">";
    v[SK_FIXED] = "rk_fixed_kernel<RhsCustom, " + ss + ", " + st + ">";
    v[SK_CTL2W] = S > 0 ? "rk_ctl2w_staged_kernel<RhsCustom, " + ss + ", " + st + ">" : "";
    v[SK_CTL_STAGED_L2] = "rk_ctl_staged_kernel<RhsCustom, " + ss + ", " + st + ", 1>";
    v[SK_CTL_STAGED_GEN] = "rk_ctl_staged_kernel<RhsCustom, " + ss + ", " + st + ", 0>";
    v[SK_CTL] = "rk_ctl_kernel<RhsCustom, " + ss + ", " + st + ">";
    return v;
}

// Source -> cubin. Needs no GPU. `lowered[i]` is the mangled name of names[i] ("" where names[i] is "").
struct RtcCached {
    std::vector<char> cubin;
    std::vector<std::string> lowered;
};
int32_t rtc_compile_uncached(const std::string& src, const std::vector<std::string>& names, bool fmad_off, std::vector<char>& cubin,
                             std::vector<std::string>& lowered, std::string& log);

// Process-wide cache of compiled sources: a pipelined solve builds one handle per chunk from the same body, tests build many.
int32_t rtc_compile(const std::string& src, const std::vector<std::string>& names, bool fmad_off, std::vector<char>& cubin,
                    std::vector<std::string>& lowered, std::string& log) {
    static std::map<std::string, RtcCached> cache;
    static std::mutex mu;
    std::string key = fmad_off ? "S\n" : "F\n";
    for (const std::string& n : names) key += n + "\n";
    key += src;
    {
        std::lock_guard<std::mutex> lock(mu);
        auto it = cache.find(key);
        if (it != cache.end()) {
            cubin = it->second.cubin, lowered = it->second.lowered;
            return VO_OK;
        }
    }
    const int32_t rc = rtc_compile_uncached(src, names, fmad_off, cubin, lowered, log);
    if (rc == VO_OK) {
        std::lock_guard<std::mutex> lock(mu);
        if (cache.size() < 256) cache[key] = RtcCached{cubin, lowered};
    }
    return rc;
}

int32_t rtc_compile_uncached(const std::string& src, const std::vector<std::string>& names, bool fmad_off, std::vector<char>& cubin,
                             std::vector<std::string>& lowered, std::string& log) {
    Nvrtc* nv = nullptr;
    if (!nvrtc_load(&nv, log)) return VO_ERR_UNSUPPORTED;
    const char* hdr_text[N_HEADERS];
    const char* hdr_name[N_HEADERS];
    for (int i = 0; i < N_HEADERS; ++i) hdr_text[i] = RTC_HEADERS[i].text, hdr_name[i] = RTC_HEADERS[i].name;
    nvrtcProgram prog;
    nvrtcResult r = nv->createProgram(&prog, src.c_str(), "vo_user_rhs.cu", N_HEADERS, hdr_text, hdr_name);
    if (r != NVRTC_SUCCESS) {
        log = std::string("nvrtcCreateProgram: ") + nv->getErrorString(r);
        return VO_ERR_CUDA;
    }
    for (const std::string& n : names)
        if (!n.empty()) nv->addNameExpression(prog, n.c_str());
    std::vector<const char*> opts = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo",
                                      "-default-device"};  // the C-ABI prototypes in vecode_b200.h are declarations only; JIT mode rejects host functions
    if (fmad_off) opts.push_back("--fmad=false");
    r = nv->compileProgram(prog, (int)opts.size(), opts.data());
    if (r != NVRTC_SUCCESS) {
        size_t n = 0;
        nv->getProgramLogSize(prog, &n);
        std::string l(n, '\0');
        if (n) nv->getProgramLog(prog, &l[0]);
        if (l.size() > 4000) l.resize(4000), l += "\n[...]";
        log = std::string("user source does not compile (") + nv->getErrorString(r) + "):\n" + l.c_str();
        nv->destroyProgram(&prog);
        return VO_ERR_BAD_ARG;
    }
    size_t n = 0;
    nv->getCUBINSize(prog, &n);
    cubin.resize(n);
    nv->getCUBIN(prog, cubin.data());
    lowered.assign(names.size(), "");
    for (size_t i = 0; i < names.size(); ++i) {
        if (names[i].empty()) continue;
        const char* low = nullptr;
        if (nv->getLoweredName(prog, names[i].c_str(), &low) != NVRTC_SUCCESS || !low) {
            log = "user RHS: no lowered name for " + names[i];
            nv->destroyProgram(&prog);
            return VO_ERR_CUDA;
        }
        lowered[i] = low;
    }
    nv->destroyProgram(&prog);
    return VO_OK;
}

int32_t compile_custom(const vo_rhs_s* r, int S, bool strict, std::vector<char>& cubin, std::vector<std::string>& lowered, std::string& log) {
    const bool stage_module = S == STAGE_MODULE;
    const bool stencil = r->kind == VO_RHS_CUSTOM_STENCIL;
    return rtc_compile(rtc_source(r, stage_module), kernel_names(stencil ? (r->radius <= 4 ? 1 : 0) : S, strict, stage_module, stencil), strict, cubin, lowered, log);
}

int module_key(int S, bool strict) { return (S + 1) * 2 + (strict ? 1 : 0); }

int32_t get_module(vo_rhs_s* r, int S, bool strict, Driver** drv, CustomModule** out) {
    vo_ctx c = r->ctx;
    std::string err;
    if (!driver_load(drv, err)) return vo_fail(c, VO_ERR_UNSUPPORTED, err);
    auto it = r->modules.find(module_key(S, strict));
    if (it != r->modules.end()) {
        *out = static_cast<CustomModule*>(it->second);
        return VO_OK;
    }
    std::vector<char> cubin;
    std::vector<std::string> lowered;
    int32_t rc = compile_custom(r, S, strict, cubin, lowered, err);
    if (rc != VO_OK) return vo_fail(c, rc, err);
    cudaFree(0);  // make sure the primary context the runtime uses is current before the first driver call
    CustomModule* m = new CustomModule();
    CUresult e = (*drv)->moduleLoadData(&m->mod, cubin.data());
    if (e != CUDA_SUCCESS) {
        delete m;
        return vo_fail(c, VO_ERR_CUDA, "user RHS: cuModuleLoadData: " + cu_msg(*drv, e));
    }
    for (size_t i = 0; i < lowered.size(); ++i) {
        if (lowered[i].empty()) continue;
        e = (*drv)->moduleGetFunction(&m->fn[i], m->mod, lowered[i].c_str());
        if (e != CUDA_SUCCESS) {
            (*drv)->moduleUnload(m->mod);
            delete m;
            return vo_fail(c, VO_ERR_CUDA, "user RHS: cuModuleGetFunction(" + lowered[i] + "): " + cu_msg(*drv, e));
        }
    }
    r->modules[module_key(S, strict)] = m;
    *out = m;
    return VO_OK;
}

// Persistent grid of rk_small_launch.cuh::persistent_grid for a driver-API function.
int32_t custom_grid(vo_ctx c, Driver* drv, CustomModule* m, int k, int64_t N, size_t smem, int tile, unsigned* grid) {
    if (m->bps[k] == 0 || m->bps_smem[k] != smem) {
        if (smem > 48 * 1024) {
            CUresult e = drv->funcSetAttribute(m->fn[k], CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem);
            if (e != CUDA_SUCCESS) return vo_fail(c, VO_ERR_CUDA, "user RHS: shared-memory attribute: " + cu_msg(drv, e));
        }
        int bps = 0;
        if (drv->occupancy(&bps, m->fn[k], RK_SMALL_THREADS, smem) != CUDA_SUCCESS || bps < 1) bps = 1;
        m->bps[k] = bps, m->bps_smem[k] = smem;
    }
    *grid = grid_for(ceil_div(N, tile), c->sm_count, m->bps[k]);
    return VO_OK;
}

int32_t custom_launch(vo_ctx c, Driver* drv, CUfunction fn, unsigned grid, unsigned block, size_t smem, bool pdl, void** args) {
    CUlaunchConfig cfg;
    std::memset(&cfg, 0, sizeof cfg);
    cfg.gridDimX = grid, cfg.gridDimY = 1, cfg.gridDimZ = 1, cfg.blockDimX = block, cfg.blockDimY = 1, cfg.blockDimZ = 1;
    cfg.sharedMemBytes = (unsigned)smem, cfg.hStream = (CUstream)c->stream;
    CUlaunchAttribute at[1];
    std::memset(at, 0, sizeof at);
    at[0].id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
    at[0].value.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = pdl ? 1 : 0;
    CUresult e = drv->launchKernelEx(&cfg, fn, args, nullptr);
    if (e != CUDA_SUCCESS) return vo_fail(c, VO_ERR_CUDA, "user RHS: kernel launch: " + cu_msg(drv, e));
    return VO_OK;
}

int stage_count_key(int s) { return (s == 4 || s == 6 || s == 7) ? s : 0; }  // the unrolled instantiations of launch_family

}  // namespace

// The register-resident path for a user RHS: the kernel small_plan chooses, as launch_one (rk_small_launch.cuh) does.
int32_t launch_small_custom(const SmallLaunch& L, vo_rhs_s* r) {
    vo_ctx c = L.ctx;
    const bool strict = c->arith == VO_ARITH_STRICT;
    const int S = stage_count_key(L.tb->s);
    Driver* drv = nullptr;
    CustomModule* m = nullptr;
    int32_t rc = get_module(r, S, strict, &drv, &m);
    if (rc != VO_OK) return rc;
    double* x = L.x;
    int64_t N = L.N;
    TableauDev tb = *L.tb;
    RhsParams rp = *L.rp;
    CtlArrays ca = L.ca;
    EvSlot* ev = L.ev;
    const SmallPlan P = small_plan(N, S > 0, r->d + per_traj_rows(rp, r->np), L.cs);
    // grid, then the chain decision (same kernel and same grid as this solver's previous launch), then the launch
    unsigned grid = 0;
    rc = custom_grid(c, drv, m, P.k, N, P.smem, P.tile, &grid);
    if (rc != VO_OK) return rc;
    pipe::Chain ch = L.cst->next((const void*)m->fn[P.k], grid, P.staged);
    // The driver takes the number of parameters from the kernel image: the unstaged kernels (SK_FIXED, SK_CTL) have no
    // trailing pipe::Chain and read one pointer less of the list.
    auto go = [&](void** args) { return custom_launch(c, drv, m->fn[P.k], grid, RK_SMALL_THREADS, P.smem, ch.chained != 0, args); };
    if (L.sl) {
        StepList sl = *L.sl;
        void* args[] = {&x, &N, &tb, &rp, &sl, &ch};
        return go(args);
    }
    CtlShared cs = *L.cs;
    void* args[] = {&x, &N, &tb, &rp, &ca, &cs, &ev, &ch};
    return go(args);
}

// The stage path for a user RHS (vo_rk_try_step, vo_rhs_eval, vo_solver_set_path(1)).
int32_t launch_stage_custom(vo_ctx c, vo_rhs_s* r, bool tail, const double* x0, int64_t N, const StageArgs& sa_in, const RhsParams& rp_in, double* k_out,
                            double* nx, double* xe) {
    Driver* drv = nullptr;
    CustomModule* m = nullptr;
    int32_t rc = get_module(r, STAGE_MODULE, c->arith == VO_ARITH_STRICT, &drv, &m);
    if (rc != VO_OK) return rc;
    StageArgs sa = sa_in;
    RhsParams rp = rp_in;
    void* args[] = {&x0, &N, &sa, &rp, &k_out, &nx, &xe};
    return custom_launch(c, drv, m->fn[tail ? K_STAGE_TAIL : K_STAGE], (unsigned)ceil_div(N, 128), 128, 0, false, args);
}

// The stage path for a user stencil on one grid state (rk_stage_stencil.cuh). Large even grids with radius <= 4 take the TMA-staged
// kernel (the K's this launch reads compacted exactly as for the compiled-in heat equation, solver.cu: launch_heat_tma); everything
// else the plain kernel with persistent CTAs over 256-point tiles.
int32_t launch_stage_stencil_custom(vo_ctx c, vo_rhs_s* r, bool tail, const double* x0, int64_t d, const StageArgs& sa_in, const RhsParams& rp_in, double* k_out,
                                    double* nx, double* xe) {
    Driver* drv = nullptr;
    CustomModule* m = nullptr;
    const bool strict = c->arith == VO_ARITH_STRICT;
    int32_t rc = get_module(r, STAGE_MODULE, strict, &drv, &m);
    if (rc != VO_OK) return rc;
    StageArgs sa = sa_in;
    RhsParams rp = rp_in;
    const int S = sa.s;
    if (r->radius <= 4 && d % 2 == 0 && d >= 4 * SX_TILE && S <= 8 && !getenv("VECODE_STENCIL_PLAIN")) {
        StencilArgs ha;
        std::memset(&ha, 0, sizeof ha);
        ha.dt = sa.dt, ha.t_i = sa.t_i, ha.use_err = sa.use_err;
        const int nload = tail ? S - 1 : sa.i;
        int nk = 0;
        for (int j = 0; j < nload; ++j) {
            if (!(strict || tail || sa.a[j] != 0.0)) continue;  // FAST non-tail stages drop zero coefficients; STRICT keeps them, like the reference
            ha.K[nk] = sa.K[j], ha.a[nk] = j < sa.i ? sa.a[j] : 0.0, ha.b[nk] = sa.b[j], ha.b_err[nk] = sa.b_err[j];
            ++nk;
        }
        ha.nterm = (strict || tail) ? sa.i : nk;
        ha.b_last = sa.b[S - 1], ha.b_err_last = sa.b_err[S - 1];
        const int HL = (r->radius + 1) & ~1, bps = (nk <= 3 && r->radius <= 2) ? 2 : 1;
        const size_t row_bytes = (size_t)(nk + 1) * (SX_TILE + 2 * HL) * sizeof(double);
        ha.nst = (int)std::max<size_t>(2, std::min<size_t>(SX_STAGES_MAX, (size_t)(208 * 1024 / bps) / row_bytes));
        const size_t smem = (size_t)ha.nst * row_bytes;
        const int k = K_STENCIL_TMA + (tail ? 8 : 0) + nk;
        if (m->bps_smem[k] < smem) {
            CUresult e = drv->funcSetAttribute(m->fn[k], CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, 216 * 1024);
            if (e != CUDA_SUCCESS) return vo_fail(c, VO_ERR_CUDA, "user stencil: shared-memory attribute: " + cu_msg(drv, e));
            m->bps_smem[k] = 216 * 1024;
        }
        const int64_t tiles = ceil_div(d, SX_TILE);
        const int64_t iters = ceil_div(tiles, (int64_t)c->sm_count * bps);
        void* args[] = {&x0, &d, &ha, &rp, &k_out, &nx, &xe};
        return custom_launch(c, drv, m->fn[k], (unsigned)ceil_div(tiles, iters), SX_THREADS, smem, false, args);
    }
    void* args[] = {&x0, &d, &sa, &rp, &k_out, &nx, &xe};
    const int64_t tiles = ceil_div(d, ST_THREADS);
    const unsigned grid = (unsigned)std::min<int64_t>(tiles, (int64_t)c->sm_count * 8);
    return custom_launch(c, drv, m->fn[tail ? K_STAGE_TAIL : K_STAGE], grid, ST_THREADS, 0, false, args);
}

void custom_rhs_release(vo_rhs_s* r) {
    std::string err;
    Driver* drv = nullptr;
    const bool have = driver_load(&drv, err);
    for (auto& kv : r->modules) {
        CustomModule* m = static_cast<CustomModule*>(kv.second);
        if (have && m->mod) drv->moduleUnload(m->mod);
        delete m;
    }
    r->modules.clear();
}

// ---- the same machinery for the generator closure of the exponential integrators (exp.cu) -------------------------------
// The functor wraps statements that assign g[1] .. g[M_gen-1], the real coefficients of L(t) = B_0 + sum_m g[m] B_m, from the
// time `t` and this system's parameter row `p` (the 3 (M_gen - 1) doubles per system handed to vo_exp_create).
int32_t rtc_exp_compile(const std::string& body, const std::string& norm_src, int ndim, int M, std::vector<char>& cubin, std::string& lowered, std::string& log) {
    const bool small = ndim <= VO_EXP_SMALL_MAX_N;  // exp_small_kernel for 1 <= n <= 8, the tensor-core tiles above
    std::string src = norm_src + (small ? "#include \"exp_small_kernels.cuh\"\n" : "#include \"exp_kernels.cuh\"\n");
    const bool user_gen = !body.empty();
    if (user_gen)
        src += "struct GenCustom {\n"
               "    template <int M> static __device__ __forceinline__ void coef(const double* __restrict__ p, int M_gen, const double t, double (&c)[M]) {\n"
               "        double g[M];\n#pragma unroll\n        for (int m = 0; m < M; ++m) g[m] = 0.0;\n        {\n#line 1 \"generator_body\"\n" +
               body +
               "\n        }\n#pragma unroll\n        for (int m = 0; m < M; ++m) c[m] = (m >= 1 && m < M_gen) ? g[m] : 0.0;\n        c[0] = 1.0;\n    }\n};\n";
    const std::string shape = std::to_string(ndim) + ", " + std::to_string(M) + (small ? ", " : ", 16, ");
    std::vector<std::string> names = {(small ? "exp_small_kernel<" : "exp_step_kernel<") + shape + (user_gen ? "GenCustom" : "GenCos") + ">"}, low;
    const int32_t rc = rtc_compile(src, names, false, cubin, low, log);
    if (rc == VO_OK) lowered = low[0];
    return rc;
}

int32_t rtc_exp_module(vo_ctx c, const std::string& body, const std::string& norm_src, int ndim, int M, size_t smem, void** module_out, void** fn_out) {
    std::string err, lowered;
    Driver* drv = nullptr;
    if (!driver_load(&drv, err)) return vo_fail(c, VO_ERR_UNSUPPORTED, err);
    std::vector<char> cubin;
    int32_t rc = rtc_exp_compile(body, norm_src, ndim, M, cubin, lowered, err);
    if (rc != VO_OK) return vo_fail(c, rc, err);
    cudaFree(0);
    CUmodule mod = nullptr;
    CUfunction fn = nullptr;
    CUresult e = drv->moduleLoadData(&mod, cubin.data());
    if (e == CUDA_SUCCESS) e = drv->moduleGetFunction(&fn, mod, lowered.c_str());
    if (e == CUDA_SUCCESS) e = drv->funcSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem);
    if (e != CUDA_SUCCESS) {
        if (mod) drv->moduleUnload(mod);
        return vo_fail(c, VO_ERR_CUDA, "user generator: module load: " + cu_msg(drv, e));
    }
    *module_out = mod, *fn_out = fn;
    return VO_OK;
}

int32_t rtc_exp_launch(vo_ctx c, void* fn, unsigned grid, unsigned block, size_t smem, void** args) {
    std::string err;
    Driver* drv = nullptr;
    if (!driver_load(&drv, err)) return vo_fail(c, VO_ERR_UNSUPPORTED, err);
    return custom_launch(c, drv, (CUfunction)fn, grid, block, smem, false, args);
}

void rtc_exp_unload(void* module) {
    std::string err;
    Driver* drv = nullptr;
    if (module && driver_load(&drv, err)) drv->moduleUnload((CUmodule)module);
}


// ---- user-defined norms (norm_custom.cuh) ------------------------------------------------------------------------------------
std::string norm_source(const vo_normfn_s* f) {
    std::string s = "#define VO_USER_NORM 1\nstruct VoUserNorm {\n    static constexpr int JOIN = " + std::to_string(f->join) + ";\n";
    s += "    static __device__ __forceinline__ double map(const double e, const double im, const int i, const int n) {\n        double m = 0.0;\n        {\n"
         "#line 1 \"norm_map_body\"\n" + f->map_body + "\n        }\n        return m;\n    }\n";
    s += "    static __device__ __forceinline__ double finish(const double acc, const int n) {\n        double r = acc;\n        {\n"
         "#line 1 \"norm_finish_body\"\n" + f->finish_body + "\n        }\n        return r;\n    }\n};\n";
    return s;
}

namespace {
int32_t norm_compile(const vo_normfn_s* f, bool strict, std::vector<char>& cubin, std::vector<std::string>& lowered, std::string& log) {
    const std::string src = norm_source(f) + "#include \"norm_custom.cuh\"\n";
    return rtc_compile(src, {"norm_small_custom_kernel<VoUserNorm>", "norm_partial_custom_kernel<VoUserNorm>", "norm_final_custom_kernel<VoUserNorm>"}, strict, cubin,
                       lowered, log);
}
}  // namespace

int32_t norm_custom_device(vo_normfn_s* f, const double* x, int64_t d, int64_t n, int64_t i_off, int64_t d_total, double* out_dev, double* partial_dev,
                           int partial_cap, bool finish) {
    vo_ctx c = f->ctx;
    const int am = c->arith == VO_ARITH_STRICT ? 0 : 1;
    std::string err;
    Driver* drv = nullptr;
    if (!driver_load(&drv, err)) return vo_fail(c, VO_ERR_UNSUPPORTED, err);
    std::unique_lock<std::mutex> lock(f->mu);
    if (!f->module[am]) {
        std::vector<char> cubin;
        std::vector<std::string> lowered;
        int32_t rc = norm_compile(f, am == 0, cubin, lowered, err);
        if (rc != VO_OK) return vo_fail(c, rc, err);
        cudaFree(0);
        CUmodule mod = nullptr;
        CUresult e = drv->moduleLoadData(&mod, cubin.data());
        for (int k = 0; k < 3 && e == CUDA_SUCCESS; ++k) e = drv->moduleGetFunction((CUfunction*)&f->fn[am][k], mod, lowered[k].c_str());
        if (e != CUDA_SUCCESS) {
            if (mod) drv->moduleUnload(mod);
            return vo_fail(c, VO_ERR_CUDA, "user norm: module load: " + cu_msg(drv, e));
        }
        f->module[am] = mod;
    }
    lock.unlock();
    int fin = finish ? 1 : 0;
    if (d <= 64) {  // one thread per trajectory, left to right (the order of a sequential norm), like the built-in norms
        void* args[] = {&x, &d, &n, &out_dev, &fin};
        // (the small kernel numbers components from 0; a window of a larger vector goes through the partial kernel below)
        if (i_off == 0 && d == d_total) {
            int32_t r = custom_launch(c, drv, (CUfunction)f->fn[am][0], (unsigned)ceil_div(n, 256), 256, 0, false, args);
            if (r != VO_OK) return r;
            VO_CHECK_LAUNCH(c);
            return VO_OK;
        }
    }
    int chunks = (int)std::min<int64_t>(std::max<int64_t>(1, d / 4096), std::max<int64_t>(1, (int64_t)c->sm_count * 4 / std::max<int64_t>(1, n)));
    chunks = std::max(1, std::min(chunks, partial_cap / (int)std::max<int64_t>(1, n)));
    if ((int64_t)chunks * n > partial_cap) return vo_fail(c, VO_ERR_UNSUPPORTED, "user norm: too many trajectories for the large-d path");
    {
        void* args[] = {&x, &d, &n, &i_off, &d_total, &partial_dev};
        CUlaunchConfig cfg;
        std::memset(&cfg, 0, sizeof cfg);
        cfg.gridDimX = (unsigned)chunks, cfg.gridDimY = (unsigned)n, cfg.gridDimZ = 1, cfg.blockDimX = 256, cfg.blockDimY = 1, cfg.blockDimZ = 1;
        cfg.hStream = (CUstream)c->stream;
        CUresult e = drv->launchKernelEx(&cfg, (CUfunction)f->fn[am][1], args, nullptr);
        if (e != CUDA_SUCCESS) return vo_fail(c, VO_ERR_CUDA, "user norm: kernel launch: " + cu_msg(drv, e));
        VO_CHECK_LAUNCH(c);
    }
    void* args[] = {&partial_dev, &chunks, &d_total, &out_dev, &fin};
    int32_t r = custom_launch(c, drv, (CUfunction)f->fn[am][2], (unsigned)n, 32, 0, false, args);
    if (r != VO_OK) return r;
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}

vo_rhs_s* custom_rhs_with_norm(const vo_rhs_s* base, const vo_normfn_s* f) {
    vo_rhs_s* r = new vo_rhs_s();
    r->ctx = base->ctx, r->kind = VO_RHS_CUSTOM, r->d = base->d, r->np = base->np, r->body = base->body;
    r->alias_kind = base->kind == VO_RHS_CUSTOM ? -1 : base->kind;
    r->norm_src = norm_source(f);
    for (int i = 0; i < VO_MAX_PARAMS; ++i) r->shared[i] = 0.0, r->per_traj[i] = nullptr, r->per_traj_n[i] = 0;  // parameters stay with the solver's own RHS
    return r;
}

extern "C" {

int32_t vo_normfn_create(vo_ctx c, const char* map_body, int32_t join, const char* finish_body, vo_normfn* out) {
    if (!c || !map_body || !out || (join != VO_NORM_JOIN_SUM && join != VO_NORM_JOIN_MAX)) return vo_fail(c, VO_ERR_BAD_ARG, "vo_normfn_create: bad argument");
    vo_normfn f = new vo_normfn_s();
    f->ctx = c, f->map_body = map_body, f->finish_body = finish_body ? finish_body : "", f->join = join;
    std::vector<char> cubin;
    std::vector<std::string> lowered;
    std::string log;
    const int32_t rc = norm_compile(f, c->arith == VO_ARITH_STRICT, cubin, lowered, log);  // a source error is reported here, not at the first step
    if (rc != VO_OK) {
        delete f;
        return vo_fail(c, rc, log);
    }
    *out = f;
    return VO_OK;
}

int32_t vo_normfn_destroy(vo_normfn f) {
    if (!f) return VO_OK;
    std::string err;
    Driver* drv = nullptr;
    const bool have = driver_load(&drv, err);
    for (int a = 0; a < 2; ++a)
        if (have && f->module[a]) drv->moduleUnload((CUmodule)f->module[a]);
    delete f;
    return VO_OK;
}

int32_t vo_normfn_check(const char* map_body, int32_t join, const char* finish_body, char* log, int64_t log_cap) {
    if (log && log_cap > 0) log[0] = '\0';
    if (!map_body || (join != VO_NORM_JOIN_SUM && join != VO_NORM_JOIN_MAX)) return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_normfn_check: bad argument");
    vo_normfn_s f;
    f.map_body = map_body, f.finish_body = finish_body ? finish_body : "", f.join = join;
    std::vector<char> cubin;
    std::vector<std::string> lowered;
    std::string msg;
    const int32_t rc = norm_compile(&f, true, cubin, lowered, msg);
    if (rc != VO_OK) {
        if (log && log_cap > 0) std::strncpy(log, msg.c_str(), (size_t)log_cap - 1), log[log_cap - 1] = '\0';
        return vo_fail(nullptr, rc, msg);
    }
    return (int32_t)std::min<size_t>(cubin.size(), 0x7fffffff);
}

int32_t vo_normfn_check_kernels(const char* map_body, int32_t join, const char* finish_body, int32_t rhs_kind, int32_t d, int32_t stages, int32_t arith, int32_t exp_n,
                                int32_t exp_M, char* log, int64_t log_cap) {
    if (log && log_cap > 0) log[0] = '\0';
    if (!map_body || (join != VO_NORM_JOIN_SUM && join != VO_NORM_JOIN_MAX)) return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_normfn_check_kernels: bad argument");
    vo_normfn_s f;
    f.map_body = map_body, f.finish_body = finish_body ? finish_body : "", f.join = join;
    std::string msg;
    size_t total = 0;
    int32_t rc = VO_OK;
    if (rhs_kind >= 0) {  // the register-resident kernels of a compiled-in family, re-compiled with the norm in them
        vo_rhs_s base;
        base.kind = rhs_kind, base.d = d, base.np = 0;
        vo_rhs_s* r = custom_rhs_with_norm(&base, &f);
        std::vector<char> cubin;
        std::vector<std::string> lowered;
        rc = compile_custom(r, stage_count_key(stages), arith == VO_ARITH_STRICT, cubin, lowered, msg);
        total += cubin.size();
        delete r;
    }
    if (rc == VO_OK && exp_n > 0) {
        std::vector<char> cubin;
        std::string lowered;
        if (exp_n > 64 || (exp_n > VO_EXP_SMALL_MAX_N && exp_n % 8) || exp_M < 1 || exp_M > 4)
            rc = VO_ERR_BAD_ARG, msg = "vo_normfn_check_kernels: exp_n must be 1 <= n <= 8 or a multiple of 8 up to 64, and 1 <= exp_M <= 4";
        else
            rc = rtc_exp_compile("", norm_source(&f), exp_n, exp_M, cubin, lowered, msg);
        total += cubin.size();
    }
    if (rc != VO_OK) {
        if (log && log_cap > 0) std::strncpy(log, msg.c_str(), (size_t)log_cap - 1), log[log_cap - 1] = '\0';
        return vo_fail(nullptr, rc, msg);
    }
    return (int32_t)std::min<size_t>(total, 0x7fffffff);
}

int32_t vo_norm_custom(vo_ens e, vo_normfn f, double* out_host) {
    if (!e || !f || !out_host) return vo_fail(e ? e->ctx : nullptr, VO_ERR_BAD_ARG, "vo_norm_custom: bad argument");
    vo_ctx c = e->ctx;
    if (f->ctx != c) return vo_fail(c, VO_ERR_BAD_ARG, "vo_norm_custom: the norm belongs to another ctx");
    DeviceGuard g(c->device);
    double *out_dev = nullptr, *partial = nullptr;
    const int cap = 1 << 16;
    VO_CUDA(c, cudaMallocAsync(&out_dev, sizeof(double) * e->n, c->stream));
    VO_CUDA(c, cudaMallocAsync(&partial, sizeof(double) * cap, c->stream));
    int32_t r = norm_custom_device(f, e->p, e->d, e->n, 0, e->d, out_dev, partial, cap, true);
    if (r == VO_OK) {
        cudaError_t ce = cudaMemcpyAsync(out_host, out_dev, sizeof(double) * e->n, cudaMemcpyDeviceToHost, c->stream);
        if (ce != cudaSuccess) r = vo_fail(c, VO_ERR_CUDA, cudaGetErrorString(ce));
    }
    cudaFreeAsync(out_dev, c->stream), cudaFreeAsync(partial, c->stream);
    VO_CUDA(c, cudaStreamSynchronize(c->stream));
    return r;
}

int32_t vo_exp_generator_check(const char* body, int32_t n, int32_t M, char* log, int64_t log_cap) {
    if (log && log_cap > 0) log[0] = '\0';
    if (!body || n < 1 || n > 64 || (n > VO_EXP_SMALL_MAX_N && n % 8) || M < 1 || M > 4)
        return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_exp_generator_check: need 1 <= n <= 8 or n a multiple of 8 up to 64, and 1 <= M <= 4");
    std::vector<char> cubin;
    std::string lowered, msg;
    const int32_t rc = rtc_exp_compile(body, "", n, M, cubin, lowered, msg);
    if (rc != VO_OK) {
        if (log && log_cap > 0) std::strncpy(log, msg.c_str(), (size_t)log_cap - 1), log[log_cap - 1] = '\0';
        return vo_fail(nullptr, rc, msg);
    }
    return (int32_t)std::min<size_t>(cubin.size(), 0x7fffffff);
}

int32_t vo_rhs_create_custom(vo_ctx c, const char* body, int32_t d, int32_t n_params, vo_rhs* out) {
    if (!c || !body || !out) return vo_fail(c, VO_ERR_BAD_ARG, "vo_rhs_create_custom: NULL argument");
    if (d < 1 || d > 32 || n_params < 0 || n_params > VO_MAX_PARAMS) return vo_fail(c, VO_ERR_SHAPE, "vo_rhs_create_custom: needs 1 <= d <= 32 and 0 <= n_params <= 8");
    DeviceGuard g(c->device);
    vo_rhs r = new vo_rhs_s();
    r->ctx = c, r->kind = VO_RHS_CUSTOM, r->d = d, r->np = n_params, r->body = body;
    for (int i = 0; i < VO_MAX_PARAMS; ++i) r->shared[i] = 0.0, r->per_traj[i] = nullptr, r->per_traj_n[i] = 0;
    // compile the stage-path module now, so that a source error is reported here rather than at the first step
    Driver* drv = nullptr;
    CustomModule* m = nullptr;
    int32_t rc = get_module(r, STAGE_MODULE, c->arith == VO_ARITH_STRICT, &drv, &m);
    if (rc != VO_OK) {
        custom_rhs_release(r);
        delete r;
        return rc;
    }
    *out = r;
    return VO_OK;
}

int32_t vo_rhs_create_custom_stencil(vo_ctx c, const char* body, int64_t d, int32_t radius, int32_t n_params, vo_rhs* out) {
    if (!c || !body || !out) return vo_fail(c, VO_ERR_BAD_ARG, "vo_rhs_create_custom_stencil: NULL argument");
    if (radius < 1 || radius > 8 || n_params < 0 || n_params > VO_MAX_PARAMS || d < 2 * radius + 1 || d > 0x7fffffff)
        return vo_fail(c, VO_ERR_SHAPE, "vo_rhs_create_custom_stencil: needs 1 <= radius <= 8, 0 <= n_params <= 8 and 2 radius + 1 <= d < 2^31");
    DeviceGuard g(c->device);
    vo_rhs r = new vo_rhs_s();
    r->ctx = c, r->kind = VO_RHS_CUSTOM_STENCIL, r->d = (int)d, r->np = n_params, r->body = body, r->radius = radius;
    for (int i = 0; i < VO_MAX_PARAMS; ++i) r->shared[i] = 0.0, r->per_traj[i] = nullptr, r->per_traj_n[i] = 0;
    Driver* drv = nullptr;
    CustomModule* m = nullptr;
    int32_t rc = get_module(r, STAGE_MODULE, c->arith == VO_ARITH_STRICT, &drv, &m);  // a source error is reported here
    if (rc != VO_OK) {
        custom_rhs_release(r);
        delete r;
        return rc;
    }
    *out = r;
    return VO_OK;
}

int32_t vo_rhs_custom_stencil_check(const char* body, int32_t radius, int32_t n_params, int32_t arith, char* log, int64_t log_cap) {
    if (log && log_cap > 0) log[0] = '\0';
    if (!body || radius < 1 || radius > 8 || n_params < 0 || n_params > VO_MAX_PARAMS) return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_rhs_custom_stencil_check: bad argument");
    vo_rhs_s tmp;
    tmp.kind = VO_RHS_CUSTOM_STENCIL, tmp.d = 0, tmp.np = n_params, tmp.body = body, tmp.radius = radius;
    std::vector<char> cubin;
    std::vector<std::string> lowered;
    std::string msg;
    const int32_t rc = compile_custom(&tmp, STAGE_MODULE, arith == VO_ARITH_STRICT, cubin, lowered, msg);
    if (rc != VO_OK) {
        if (log && log_cap > 0) std::strncpy(log, msg.c_str(), (size_t)log_cap - 1), log[log_cap - 1] = '\0';
        return vo_fail(nullptr, rc, msg);
    }
    return (int32_t)std::min<size_t>(cubin.size(), 0x7fffffff);
}

int32_t vo_rhs_custom_check(const char* body, int32_t d, int32_t n_params, int32_t stages, int32_t arith, char* log, int64_t log_cap) {
    if (log && log_cap > 0) log[0] = '\0';
    if (!body || d < 1 || d > (stages < 0 ? 32 : 8) || n_params < 0 || n_params > VO_MAX_PARAMS || stages < -1 || stages > VO_MAX_STAGES)
        return vo_fail(nullptr, VO_ERR_BAD_ARG, "vo_rhs_custom_check: bad argument");
    std::vector<char> cubin;
    std::vector<std::string> lowered;
    std::string msg;
    vo_rhs_s tmp;
    tmp.kind = VO_RHS_CUSTOM, tmp.d = d, tmp.np = n_params, tmp.body = body;
    const int32_t rc = compile_custom(&tmp, stages < 0 ? STAGE_MODULE : stage_count_key(stages), arith == VO_ARITH_STRICT, cubin, lowered, msg);
    if (rc != VO_OK) {
        if (log && log_cap > 0) std::strncpy(log, msg.c_str(), (size_t)log_cap - 1), log[log_cap - 1] = '\0';
        return vo_fail(nullptr, rc, msg);
    }
    return (int32_t)std::min<size_t>(cubin.size(), 0x7fffffff);
}

}  // extern "C"
