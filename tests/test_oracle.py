"""Oracle self-checks, modelled on the nearest pins in the reference's own test-suite (SURVEY.md section 4/8c):
GPy/testing/model_tests.py:63-82 (posterior vs the direct pinv formula), kernel_tests.py:366-422 (finite-difference
gradients_X for RBF / Matern32 / Matern52), cython_tests.py:34-51 (_grad_X C vs numpy), linalg_test.py:18-37
(jitchol jitter schedule), GPyOpt/testing/acquisitions_tests/test_ei_acquisition.py:18-37 (analytic EI known answers).
"""
import ctypes
import os

import numpy as np
import pytest

from oracle import linalg as ol
from oracle.kern import Kern, grad_X
from oracle.gp import GPRegression
from tests.helpers import make_problem, oracle_model, oracle_acq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("kind", ["se", "rbf", "matern52", "matern32"])
def test_posterior_matches_pinv_formula(kind):
    # model_tests.py:63-82 test_raw_predict
    rng = np.random.default_rng(0)
    X = rng.uniform(size=(25, 3))
    Y = rng.standard_normal((25, 1))
    k = Kern(kind, 3, 1.3, [0.4, 0.7, 0.5], ARD=True)
    g = GPRegression(X, Y, k, noise_var=0.05)
    Xs = rng.uniform(size=(7, 3))
    Kinv = np.linalg.pinv(k.K(X) + np.eye(25) * (0.05 + 1e-8))
    mu_hat = k.K(Xs, X).dot(Kinv).dot(Y - Y.mean()) + Y.mean()
    var_hat = k.Kdiag(Xs) - np.sum(k.K(Xs, X).dot(Kinv) * k.K(Xs, X), axis=1)
    np.testing.assert_allclose(g.posterior_mean(Xs), mu_hat, rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(g.posterior_variance_noiseless(Xs)[:, 0], var_hat, rtol=1e-7, atol=1e-10)
    np.testing.assert_allclose(g.posterior_variance(Xs)[:, 0], var_hat + 0.05, rtol=1e-7, atol=1e-10)


@pytest.mark.parametrize("kind", ["se", "rbf", "matern52", "matern32"])
def test_gradients_X_finite_difference(kind):
    # kernel_tests.py check_kernel_gradient_functions pattern
    rng = np.random.default_rng(1)
    X, X2 = rng.uniform(size=(6, 4)), rng.uniform(size=(9, 4))
    D = rng.standard_normal((6, 9))
    k = Kern(kind, 4, 0.8, [0.5, 0.9, 0.3, 0.6], ARD=True)
    g = k.gradients_X(D, X, X2)
    eps = 1e-6
    for i in range(6):
        for q in range(4):
            Xp, Xm = X.copy(), X.copy()
            Xp[i, q] += eps
            Xm[i, q] -= eps
            fd = (np.sum(D * k.K(Xp, X2)) - np.sum(D * k.K(Xm, X2))) / (2 * eps)
            assert abs(fd - g[i, q]) < 1e-6 * max(1.0, abs(fd))


def test_grad_X_matches_reference_C_routine():
    # cython_tests.py:34-51, against the C routine's output stored in tests/golden (make_golden_grad_x.py); when
    # oracle/Makefile has built the reference's stationary_utils.c, the routine itself is held to the same vectors
    z = np.load(os.path.join(ROOT, "tests", "golden", "grad_x_stationary_utils.npz"))
    X, X2, tmp, want = z["X"], z["X2"], z["tmp"], z["grad"]
    assert np.array_equal(grad_X(X, X2, tmp), want)           # same summation order -> bit identical
    so = os.path.join(ROOT, "oracle", "_ref", "libstationary_utils.so")
    if os.path.exists(so):
        lib = ctypes.CDLL(so)
        dp = ctypes.POINTER(ctypes.c_double)
        lib._grad_X.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, dp, dp, dp, dp]
        (N, D), M = X.shape, X2.shape[0]
        out = np.zeros((N, D))
        lib._grad_X(N, D, M, X.ctypes.data_as(dp), X2.ctypes.data_as(dp), tmp.ctypes.data_as(dp), out.ctypes.data_as(dp))
        assert np.array_equal(out, want)


def test_jitchol_jitter_schedule():
    # linalg_test.py:18-37: a matrix that is not PD until enough jitter is added; and the failure message
    A = np.array([[1.0, 1.0 + 3e-5], [1.0 + 3e-5, 1.0]])      # eigenvalue -3e-5: needs jitter > 3e-5
    L, jit = ol.jitchol(A, return_jitter=True)
    assert jit == pytest.approx(np.diag(A).mean() * 1e-6 * 100)    # 1e-6, 1e-5 fail; 1e-4 succeeds
    np.testing.assert_allclose(L @ L.T, A + jit * np.eye(2), atol=1e-12)
    B = np.array([[1.0, 2.0], [2.0, 1.0]])
    with pytest.raises(np.linalg.LinAlgError, match="not positive definite, even with jitter"):
        ol.jitchol(B)
    with pytest.raises(np.linalg.LinAlgError, match="non-positive diagonal"):
        ol.jitchol(np.array([[1.0, 2.0], [2.0, -1.0]]))


def test_analytic_ei_known_answers():
    # GPyOpt/testing/acquisitions_tests/test_ei_acquisition.py:18-37: m=1, s=3, fmin=0.1, jitter=0.01 gives
    # EI = 0.79646919 (GPyOpt minimises: u = (fmin - m - jitter)/s).  maEI maximises theta^T y, so the same
    # phi/Phi algebra is reached with mu = -(m + jitter), best = -fmin.
    from oracle.acquisitions import maEI
    phi, Phi, u = maEI._get_quantiles(maEI.__new__(maEI), -0.1, -(1.0 + 0.01), 3.0)
    ei = 3.0 * (u * Phi + phi)
    assert ei == pytest.approx(0.79646919, abs=1e-7)
    # :28-37: m = 1, s = 1, dmdx = dsdx = 0.1 -> EI = 0.0986038, dEI = dsdx*phi - Phi*dmdx = 0.00822768.
    # In maEI's convention dmu = -dmdx, so  Phi*dmu + phi*dsigma  (maEI.py:120-122) is the same number.
    phi, Phi, u = maEI._get_quantiles(maEI.__new__(maEI), -0.1, -(1.0 + 0.01), 1.0)
    assert 1.0 * (u * Phi + phi) == pytest.approx(0.0986038, abs=1e-7)
    assert Phi * (-0.1) + phi * 0.1 == pytest.approx(0.00822768, abs=1e-8)


def test_uEI_linear_converges_to_maEI():
    # MC EI-CF with the linear utility must approach the closed form of maEI as S grows (SURVEY.md 7.0)
    P = make_problem(m=3, d=3, n=25, H=1, kind="rbf", composite="linear", N=12, S=20000, L=1, seed=21)
    om = oracle_model(P)
    a_mc, _ = oracle_acq(P, grad=False, variant="uEI_noiseless", model=om)
    a_an, _ = oracle_acq(P, grad=False, variant="maEI", model=om)
    assert np.max(np.abs(a_mc - a_an)) < 0.05 * np.max(a_an) + 2e-3


def test_literal_and_vectorised_twins_agree():
    P = make_problem(m=4, d=5, n=40, H=2, kind="matern52", composite="exp_cos", N=30, S=12, L=2, seed=5)
    a1, g1 = oracle_acq(P, grad=True, vectorised=False)
    a2, g2 = oracle_acq(P, grad=True, vectorised=True)
    np.testing.assert_allclose(a1, a2, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(g1, g2, rtol=1e-12, atol=1e-14)
    v1, _ = oracle_acq(P, grad=False, vectorised=False)
    v2, _ = oracle_acq(P, grad=False, vectorised=True)
    np.testing.assert_allclose(v1, v2, rtol=1e-13, atol=1e-15)


def test_variance_nonnegative_many_points():
    # model_tests.py:25-61 pattern: clipped predictive variance stays >= 1e-10 on many random points
    P = make_problem(m=2, d=2, n=60, H=1, kind="se", N=20000, S=4, noise=1e-10, seed=3, focus=0.0)
    om = oracle_model(P)
    assert np.all(om.posterior_variance(P.Xc) >= 1e-10)
