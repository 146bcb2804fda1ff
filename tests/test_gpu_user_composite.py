"""User-defined composites (CudaComposite) on the GPU: the NVRTC-compiled kernels against the built-in ones for the five
catalogued composites restated as user source, and against the CPU oracle for composites that are not separable."""
import ctypes

import numpy as np
import pytest
import torch

from tests.helpers import assert_close, make_problem, oracle_model, product_model, rel_err, tol
from tests.user_composites import (COUPLED_QUADRATIC, RESTATED, SOFTMIN, coupled_quadratic_U, coupled_quadratic_dU,
                                   softmin_U, softmin_dU)

pytestmark = pytest.mark.gpu

SAME = 1e-12          # user kernel vs built-in kernel on the same composite: same operations in the same order


def _user_utility(name, P):
    import bocf_b200
    from bocf_b200.utility import _host_funcs
    tl, src = RESTATED[name]
    U, dU = _host_funcs(name)
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    return bocf_b200.Utility(func=U, dfunc=dU, parameter_dist=pd, composite=bocf_b200.CudaComposite(src, tl))


def _builtin_utility(P):
    import bocf_b200
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    return bocf_b200.Utility(parameter_dist=pd, composite=P.composite)


def _acq(model, util, P, Xc, grad, variant="uEI_noiseless", parallel=True):
    import bocf_b200
    model.set_hyperparameters(0)
    acq = getattr(bocf_b200, variant)(model, None, utility=util)
    acq.W_samples = P.Z
    if grad:
        a, g = acq._compute_acq_withGradients(Xc)
        return a[:, 0], g
    return acq._compute_acq(Xc, parallel=parallel)[:, 0]


def _utility_eval(cid, m, Y, theta, grad):
    from bocf_b200 import _lib
    lib = _lib.load_library()
    L, p = theta.shape
    N = Y.shape[1]
    Yd = torch.from_numpy(np.ascontiguousarray(Y)).cuda()
    out = torch.empty((L, m, N) if grad else (L, N), dtype=torch.float64, device="cuda")
    th = np.ascontiguousarray(theta)
    fn = lib.bocf_utility_grad_eval if grad else lib.bocf_utility_eval
    _lib.check(fn(cid, m, ctypes.c_void_p(Yd.data_ptr()), N, th.ctypes.data_as(ctypes.c_void_p), L, p,
                  ctypes.c_void_p(out.data_ptr()), None))
    return out.cpu().numpy()


@pytest.mark.parametrize("name", sorted(RESTATED))
def test_restated_utility_eval(cuda_device, name):
    from bocf_b200 import _lib
    m, N = 5, 301
    rng = np.random.default_rng(4)
    Y = rng.standard_normal((m, N))
    theta = rng.standard_normal((3, m))
    tl, src = RESTATED[name]
    cid = _lib.register_composite(src, m, -1 if tl == "m" else tl)
    for grad in (False, True):
        ref = _utility_eval(_lib.COMPOSITES[name], m, Y, theta, grad)
        got = _utility_eval(cid, m, Y, theta, grad)
        assert rel_err(got, ref) <= SAME, (name, grad)


@pytest.mark.parametrize("name", sorted(RESTATED))
@pytest.mark.parametrize("N", [17, 600, 5000])      # block / warp / 4 candidates per warp
def test_restated_composite_matches_builtin(cuda_device, name, N):
    P = make_problem(m=4, d=3, n=60, H=2, kind="matern52", composite=name, N=N, S=1000, L=3, seed=N % 7)
    model = product_model(P, cuda_device)
    ub, uu = _builtin_utility(P), _user_utility(name, P)
    # EI-CF value: the single-candidate path and the pool branch (f* per hyper-sample)
    for Xc, par in ((P.Xc[:1], True), (P.Xc, True), (P.Xc, False)):
        assert rel_err(_acq(model, uu, P, Xc, False, parallel=par), _acq(model, ub, P, Xc, False, parallel=par)) <= SAME
    # EI-CF gradient (fused path in the tensor-core mode)
    a_b, g_b = _acq(model, ub, P, P.Xc, True)
    a_u, g_u = _acq(model, uu, P, P.Xc, True)
    assert np.count_nonzero(g_b) > 0
    assert rel_err(a_u, a_b) <= SAME and rel_err(g_u, g_b) <= SAME
    # uPI: the same counts
    assert np.array_equal(_acq(model, uu, P, P.Xc, False, "uPI"), _acq(model, ub, P, P.Xc, False, "uPI"))
    # mean utility (the MC branch of the marginal argmax), value and gradient, summed over both hyper-samples
    Z = np.random.default_rng(5).standard_normal((50, P.m))
    v_b, dv_b = model.expected_utility(P.Xc, name, P.theta[0], 2, Z=Z, grad=True)
    v_u, dv_u = model.expected_utility(P.Xc, uu.composite, P.theta[0], 2, Z=Z, grad=True)
    assert rel_err(v_u, v_b) <= SAME and rel_err(dv_u, dv_b) <= SAME


def _oracle_acq(P, func, dfunc, Xc, grad):
    from oracle import acquisitions as A
    from oracle.utility import ParameterDistribution, Utility
    mod = oracle_model(P)
    mod.set_hyperparameters(0)
    U = Utility(func, dfunc, ParameterDistribution(support=P.theta, prob_dist=P.prob))
    acq = A.uEI_noiseless(mod, utility=U, W_samples=P.Z, vectorised=True)
    if grad:
        a, g = acq._compute_acq_withGradients(Xc)
        return a[:, 0], g
    return acq._compute_acq(Xc)[:, 0], None


COUPLED = ("coupled", COUPLED_QUADRATIC, "m", coupled_quadratic_U, coupled_quadratic_dU)
SOFT = ("softmin", SOFTMIN, 0, softmin_U, softmin_dU)


@pytest.mark.parametrize("comp", [COUPLED, SOFT], ids=lambda c: c[0])
@pytest.mark.parametrize("m,d", [(1, 1), (4, 16), (64, 3)])
def test_non_separable_composite_matches_oracle(cuda_device, comp, m, d):
    import bocf_b200
    _, src, tl, func, dfunc = comp
    # n = 15 in one dimension: 50 points on [0, 1] make the Gram matrix too ill-conditioned for an fp64 parity bar
    P = make_problem(m=m, d=d, n=15 if d == 1 else 50, H=2, kind="rbf", composite="sumsq_target", N=300, S=256, L=2,
                     seed=m + d)
    if tl == 0:
        P.theta = np.zeros((2, 1))
    model = product_model(P, cuda_device)
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    util = bocf_b200.Utility(func=func, dfunc=dfunc, parameter_dist=pd, composite=bocf_b200.CudaComposite(src, tl))
    a, g = _acq(model, util, P, P.Xc, True)
    a_o, g_o = _oracle_acq(P, func, dfunc, P.Xc, True)
    assert np.count_nonzero(a_o) > 10
    assert_close(a, a_o, tol(1e-7), "acq")
    assert_close(g, g_o, tol(1e-6), "grad acq")
    v = _acq(model, util, P, P.Xc, False)                          # pool branch: f* per hyper-sample, as the oracle
    v_o, _ = _oracle_acq(P, func, dfunc, P.Xc, False)
    assert_close(v, v_o, tol(1e-7), "acq value")


def test_chunking_does_not_change_user_composite_results(cuda_device):
    """Across a chunk border (a small scratch limit): the oracle agrees, and the results equal the one-chunk ones
    bitwise."""
    import bocf_b200
    from bocf_b200 import _lib
    P = make_problem(m=3, d=5, n=300, H=2, kind="se", composite="sumsq_target", N=5000, S=64, L=1, seed=7)
    model = product_model(P, cuda_device)
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    util = bocf_b200.Utility(func=coupled_quadratic_U, dfunc=coupled_quadratic_dU, parameter_dist=pd,
                             composite=bocf_b200.CudaComposite(COUPLED_QUADRATIC))
    a1, g1 = _acq(model, util, P, P.Xc, True)
    _lib.check(model._lib.bocf_model_set_scratch_limit(model._handle, ctypes.c_uint64(64 << 20)))
    chunk = model.chunk_candidates(P.N, grad=True)
    assert chunk < P.N
    a2, g2 = _acq(model, util, P, P.Xc, True)
    assert np.array_equal(a1, a2) and np.array_equal(g1, g2)
    idx = np.unique(np.concatenate([np.arange(chunk - 40, chunk + 40), np.arange(0, P.N, 97)]))
    a_o, g_o = _oracle_acq(P, coupled_quadratic_U, coupled_quadratic_dU, P.Xc[idx], True)
    assert_close(a2[idx], a_o, tol(1e-7), "acq")
    assert_close(g2[idx], g_o, tol(1e-6), "grad acq")


def test_user_composite_errors(cuda_device):
    import bocf_b200
    from bocf_b200 import _lib
    P = make_problem(m=5, d=2, n=30, H=1, N=40, S=64, L=1, seed=2)
    model = product_model(P, cuda_device)
    comp = bocf_b200.CudaComposite(COUPLED_QUADRATIC)
    cid4 = comp.composite_id(4)
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    util = bocf_b200.Utility(func=coupled_quadratic_U, dfunc=coupled_quadratic_dU, parameter_dist=pd, composite=comp)
    acq = bocf_b200.uEI_noiseless(model, None, utility=util)
    acq.W_samples = P.Z
    acq._compute_acq(P.Xc)                                        # compiled for m = 5 at first use: runs
    lib = model._lib
    Xd = torch.from_numpy(P.Xc).cuda()
    Zt = torch.from_numpy(np.ascontiguousarray(P.Z.T)).cuda()
    out = torch.empty(P.N, dtype=torch.float64, device="cuda")
    one, zero = np.ones(1), np.zeros((1, 1))

    def call(cid, variant="ei_cf", p=5):
        th = np.zeros((1, max(p, 1)))
        return lib.bocf_acq_eval(model._handle, _lib.VARIANTS[variant], cid, ctypes.c_void_p(Xd.data_ptr()), P.N,
                                 ctypes.c_void_p(Zt.data_ptr()), P.S, th.ctypes.data_as(ctypes.c_void_p), 1, p,
                                 one.ctypes.data_as(ctypes.c_void_p), zero.ctypes.data_as(ctypes.c_void_p), 1, 0,
                                 ctypes.c_void_p(out.data_ptr()), None, None)
    assert call(cid4) == -1                                       # registered for m = 4, model has m = 5
    cid5 = comp.composite_id(5)
    assert call(cid5) == 0
    assert call(cid5, p=4) == -1                                  # theta shorter than theta_len = m
    assert call(cid5, variant="psi") == -5                        # no closed form
    assert call(cid5 + 1000) == -1                                # never registered
    with pytest.raises(_lib.BocfError):
        model.expected_utility(P.Xc, comp, np.zeros(5), 1, Z=None)
    # a CudaComposite whose device code disagrees with func / dfunc is refused at first use
    wrong = bocf_b200.Utility(func=lambda th, y: coupled_quadratic_U(th, y) + 1e-3, dfunc=coupled_quadratic_dU,
                              parameter_dist=pd, composite=comp)
    acq2 = bocf_b200.uEI_noiseless(model, None, utility=wrong)
    with pytest.raises(ValueError):
        acq2._compute_acq(P.Xc)


def _cbo(composite, cuda_device, iters=3):
    import bocf_b200 as B
    from bocf_b200.utility import _host_funcs
    rng = np.random.default_rng(3)
    d, m = 2, 3
    W = rng.standard_normal((m, d))

    def f(X):
        X = np.atleast_2d(X)
        return np.stack([np.sin(3 * X @ W[j]) + 0.3 * j * X[:, 0] for j in range(m)], axis=0)
    theta = f(np.array([[0.3, 0.7]])).T
    np.random.seed(0)
    space = B.Design_space(space=[{'name': 'var', 'type': 'continuous', 'domain': (0, 1), 'dimensionality': d}])
    objective = B.MultiObjective(f, as_list=False, output_dim=m)
    acq_opt = B.AcquisitionOptimizer(optimizer='lbfgs2', inner_optimizer='lbfgs2', space=space, n_starting=64, n_anchor=4)
    X_init = B.initial_design('random', space, 2 * (d + 1))
    model = B.multi_outputGP(m, n_samples=1, device=cuda_device)
    model.set_hyperparameter_samples(np.full((1, m), 1.0), np.full((1, m, d), 0.4), np.full((1, m), 1e-4), kind="matern52")
    pd = B.ParameterDistribution(support=theta, prob_dist=np.ones(1))
    if composite == "sumsq_target":
        U = B.Utility(parameter_dist=pd, composite="sumsq_target")
    else:
        fu, dfu = _host_funcs("sumsq_target")
        U = B.Utility(func=fu, dfunc=dfu, parameter_dist=pd, composite=B.CudaComposite(RESTATED["sumsq_target"][1]))
    acq = B.uEI_noiseless(model, space, optimizer=acq_opt, utility=U)
    bo = B.CBO(model, space, objective, acq, B.Sequential(acq), X_init, expectation_utility=None)
    bo.run_optimization(max_iter=iters)
    return bo


def test_cbo_loop_with_restated_composite_matches_builtin(cuda_device):
    bo_b = _cbo("sumsq_target", cuda_device)
    bo_u = _cbo("user", cuda_device)
    assert len(bo_u.suggested_points) == 3
    np.testing.assert_allclose(np.asarray(bo_u.suggested_points), np.asarray(bo_b.suggested_points), atol=1e-6)


def test_cbo_user_composite_with_expectation_utility_raises(cuda_device):
    import bocf_b200 as B
    from bocf_b200.cbo import CBO
    pd = B.ParameterDistribution(support=np.zeros((1, 3)), prob_dist=np.ones(1))
    U = B.Utility(func=coupled_quadratic_U, dfunc=coupled_quadratic_dU, parameter_dist=pd,
                  composite=B.CudaComposite(COUPLED_QUADRATIC))
    P = make_problem(m=3, d=2, n=20, H=1, N=8, S=16, seed=1)
    model = product_model(P, cuda_device)
    bo = CBO.__new__(CBO)
    bo.model, bo.utility, bo.n_attributes = model, U, 3
    bo.expectation_utility = B.ExpectationUtility(lambda th, mu, v: 0.0, lambda th, mu, v: 0.0)
    bo._n_hyps = lambda: 1
    with pytest.raises(ValueError, match="no closed-form expectation"):
        bo._current_marginal_argmax(np.zeros(3))
