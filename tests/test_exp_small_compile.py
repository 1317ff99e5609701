"""Run-time compilation for systems of 1 to 8 levels without a GPU: a user generator and a user norm go into exp_small_kernel
(one system per thread) exactly as they go into the tensor-core kernel above n = 8."""
import pytest


@pytest.mark.parametrize("n", [1, 2, 8])
@pytest.mark.parametrize("M", [1, 4])
def test_generator_compiles_into_the_small_kernel(vo, n, M):
    assert vo.ExpCFMSolver.check_generator("g[1] = p[0] * cos(p[1] * t + p[2]);", n, M) > 5_000


def test_generator_compile_error_carries_the_log(vo):
    with pytest.raises(vo.VecOdeError) as e:
        vo.ExpCFMSolver.check_generator("g[1] = nope;", 3, 2)
    assert "generator_body(1)" in str(e.value)


def test_generator_check_refuses_the_unsupported_sizes(vo):
    for n in (9, 12, 15):
        with pytest.raises(vo.VecOdeError):
            vo.ExpCFMSolver.check_generator("g[1] = 0.0;", n, 2)


def test_user_norm_compiles_into_the_small_kernel(vo):
    assert vo.NormFn.check_kernels("m = e * e + im * im;", "sum", "r = sqrt(acc);", exp_n=3, exp_M=2) > 5_000
    with pytest.raises(vo.VecOdeError) as e:
        vo.NormFn.check_kernels("m = nope;", "max", "", exp_n=3, exp_M=2)
    assert "norm_map_body" in str(e.value)
