"""User-defined composites without a GPU: NVRTC compiles the user's source together with the kernel template for
sm_100a, so registration, its errors and the Python surface are all checked on a CPU-only host."""
import os
import subprocess

import numpy as np
import pytest

from tests.user_composites import COUPLED_QUADRATIC, RESTATED, SOFTMIN


@pytest.fixture(scope="module")
def lib(built_library):
    from bocf_b200 import _lib
    return _lib


@pytest.mark.parametrize("m", [1, 4, 16, 64])
def test_register_compiles_every_instantiation(lib, m):
    # registration compiles all 7 modes x 3 launch shapes of mc_acq_user_kernel and both utility kernels, and fails
    # if any of them does not compile or has no lowered name
    cid = lib.register_composite(COUPLED_QUADRATIC, m, -1)
    assert cid >= lib.COMPOSITE_USER_BASE
    assert lib.register_composite(COUPLED_QUADRATIC, m, -1) == cid


def test_register_dedups_on_source_m_and_theta_len(lib):
    src = RESTATED["sumsq_target"][1]
    a = lib.register_composite(src, 3, -1)
    assert lib.register_composite(src, 3, -1) == a
    assert lib.register_composite(src, 2, -1) != a
    assert lib.register_composite(src, 3, 3) != a
    assert lib.register_composite(SOFTMIN, 3, 0) not in (a,)


def test_syntax_error_carries_nvrtc_log(lib):
    bad = RESTATED["sumsq_target"][1].replace("y[j] - th[j];", "y[j] - not_declared_here[j];")
    with pytest.raises(lib.BocfError) as ei:
        lib.register_composite(bad, 4, -1)
    assert ei.value.code == -1
    assert "not_declared_here" in str(ei.value) and "undefined" in str(ei.value)


def test_missing_gradient_fails(lib):
    only_u = "__device__ double bocf_U(const double* th, const double* y) { return y[0]; }\n"
    with pytest.raises(lib.BocfError) as ei:
        lib.register_composite(only_u, 2, 0)
    assert "bocf_dU" in str(ei.value)


@pytest.mark.parametrize("m", [0, 65, -3])
def test_outputs_out_of_range_rejected(lib, m):
    with pytest.raises(lib.BocfError) as ei:
        lib.register_composite(COUPLED_QUADRATIC, m, -1)
    assert ei.value.code == -1


def test_theta_len_below_minus_one_rejected(lib):
    with pytest.raises(lib.BocfError):
        lib.register_composite(SOFTMIN, 2, -2)


def test_no_link_time_nvrtc_dependency(built_library):
    out = subprocess.run(["readelf", "-d", built_library], capture_output=True, text=True).stdout
    needed = [ln for ln in out.splitlines() if "NEEDED" in ln]
    assert needed and not any("nvrtc" in ln for ln in needed), needed


def test_cuda_composite_needs_host_callables():
    import bocf_b200
    pd = bocf_b200.ParameterDistribution(support=np.ones((1, 2)), prob_dist=np.ones(1))
    comp = bocf_b200.CudaComposite(COUPLED_QUADRATIC)
    with pytest.raises(ValueError):
        bocf_b200.Utility(parameter_dist=pd, composite=comp)
    with pytest.raises(ValueError):
        bocf_b200.Utility(func=lambda th, y: 0.0, parameter_dist=pd, composite=comp)
    with pytest.raises(ValueError):
        bocf_b200.Utility(func=lambda th, y: 0.0, parameter_dist=pd)
    u = bocf_b200.Utility(func=lambda th, y: 1.5, dfunc=lambda th, y: y, parameter_dist=pd, composite=comp)
    assert u.eval_func(None, None) == 1.5 and u.composite is comp and not u.linear


@pytest.mark.parametrize("theta_len", ["x", -1, 1.5, True, None])
def test_cuda_composite_rejects_bad_theta_len(theta_len):
    import bocf_b200
    with pytest.raises(ValueError):
        bocf_b200.CudaComposite(COUPLED_QUADRATIC, theta_len=theta_len)


def test_theta_matrix_honours_theta_len():
    import bocf_b200
    from bocf_b200.utility import theta_matrix
    pd = bocf_b200.ParameterDistribution(support=np.ones((1, 2)), prob_dist=np.ones(1))

    def util(tl):
        return bocf_b200.Utility(func=lambda th, y: 0.0, dfunc=lambda th, y: y, parameter_dist=pd,
                                 composite=bocf_b200.CudaComposite(SOFTMIN, theta_len=tl))

    flat = np.arange(6.0)
    assert theta_matrix(util("m"), flat).shape == (1, 6)
    assert theta_matrix(util(1), flat).shape == (6, 1)
    assert theta_matrix(util(0), flat).shape == (6, 1)
    assert theta_matrix(util(3), flat).shape == (2, 3)
    assert theta_matrix(util(2), flat.reshape(3, 2)).shape == (3, 2)
    assert util(3).theta_len == 3 and util("m").theta_len == "m"
    # catalogued composites keep their shapes
    sumsq = bocf_b200.Utility(parameter_dist=pd, composite="sumsq_target")
    rosen = bocf_b200.Utility(parameter_dist=pd, composite="rosen_composite")
    assert theta_matrix(sumsq, flat).shape == (1, 6) and theta_matrix(rosen, flat).shape == (6, 1)


def test_nvrtc_preload_finds_a_library():
    from bocf_b200 import _lib
    assert _lib.preload_nvrtc() is not None
    assert os.path.basename(_lib._nvrtc._name) == "libnvrtc.so.12"
