// exp_small.cu — launches of exp_small_kernel (exp_small_kernels.cuh) for the compiled-in generator family, 1 <= n <= 8 and
// 1 <= M <= 4. A translation unit of its own: 32 instantiations, compiled next to exp.cu.
#include <algorithm>
#include <cstring>

#include "exp_small_kernels.cuh"

unsigned exp_small_grid(vo_ctx c, int64_t N) {  // grid-stride: at most as many threads as the SMs hold
    return (unsigned)std::min<int64_t>(ceil_div(N, VO_EXP_SMALL_THREADS), (int64_t)c->sm_count * (2048 / VO_EXP_SMALL_THREADS));
}

namespace {
template <int NDIM, int M>
int32_t launch_shape(vo_ctx c, const ExpKP& kp, const double* basis, double2* psi, double2* psi_out, const double* gp, const double2* coef_in, const CtlArrays& ca,
                     EvSlot* ev) {
    SmallBasis<NDIM, M> B;
    static_assert(sizeof B == sizeof(double) * 2 * M * NDIM * NDIM, "SmallBasis is the caller's [M][n][n] complex array");
    std::memcpy(&B, basis, sizeof B);
    exp_small_kernel<NDIM, M, GenCos><<<exp_small_grid(c, kp.N), VO_EXP_SMALL_THREADS, 0, c->stream>>>(kp, B, psi, psi_out, gp, coef_in, ca, ev);
    VO_CHECK_LAUNCH(c);
    return VO_OK;
}
}  // namespace

int32_t launch_exp_small(vo_ctx c, int n, int M, const ExpKP& kp, const double* basis, double2* psi, double2* psi_out, const double* gp, const double2* coef_in,
                         const CtlArrays& ca, EvSlot* ev) {
#define VO_EXP_SMALL_CASE(NDIM, MM) \
    if (n == NDIM && M == MM) return launch_shape<NDIM, MM>(c, kp, basis, psi, psi_out, gp, coef_in, ca, ev);
    VO_EXP_SMALL_CASE(1, 1) VO_EXP_SMALL_CASE(1, 2) VO_EXP_SMALL_CASE(1, 3) VO_EXP_SMALL_CASE(1, 4)
    VO_EXP_SMALL_CASE(2, 1) VO_EXP_SMALL_CASE(2, 2) VO_EXP_SMALL_CASE(2, 3) VO_EXP_SMALL_CASE(2, 4)
    VO_EXP_SMALL_CASE(3, 1) VO_EXP_SMALL_CASE(3, 2) VO_EXP_SMALL_CASE(3, 3) VO_EXP_SMALL_CASE(3, 4)
    VO_EXP_SMALL_CASE(4, 1) VO_EXP_SMALL_CASE(4, 2) VO_EXP_SMALL_CASE(4, 3) VO_EXP_SMALL_CASE(4, 4)
    VO_EXP_SMALL_CASE(5, 1) VO_EXP_SMALL_CASE(5, 2) VO_EXP_SMALL_CASE(5, 3) VO_EXP_SMALL_CASE(5, 4)
    VO_EXP_SMALL_CASE(6, 1) VO_EXP_SMALL_CASE(6, 2) VO_EXP_SMALL_CASE(6, 3) VO_EXP_SMALL_CASE(6, 4)
    VO_EXP_SMALL_CASE(7, 1) VO_EXP_SMALL_CASE(7, 2) VO_EXP_SMALL_CASE(7, 3) VO_EXP_SMALL_CASE(7, 4)
    VO_EXP_SMALL_CASE(8, 1) VO_EXP_SMALL_CASE(8, 2) VO_EXP_SMALL_CASE(8, 3) VO_EXP_SMALL_CASE(8, 4)
#undef VO_EXP_SMALL_CASE
    return vo_fail(c, VO_ERR_UNSUPPORTED, "exp: the one-system-per-thread kernel takes 1 <= n <= 8 and 1 <= M <= 4");
}
