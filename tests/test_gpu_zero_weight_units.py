"""The fused acquisition gradient skips the units (output, 128-candidate tile) of the second contraction whose gradient
weights are all zero: no base sample of those candidates improves on the incumbent.  A candidate's value and gradient
must not depend on whether its tile-mates are active, the partial sums a skipped unit left from an earlier chunk must
never be read, and every weight producer (built-in MC kernel, user composite, maEI) must still agree with the oracle."""
import ctypes

import numpy as np
import pytest

from tests.helpers import assert_close, make_problem, oracle_acq, product_model, product_utility, rel_err, tol

pytestmark = pytest.mark.gpu


def _problem(H=1, L=1, N=4000, seed=3, composite="sumsq_target"):
    return make_problem(m=4, d=5, n=200, H=H, kind="matern52", composite=composite, N=N, S=256, L=L, seed=seed,
                        focus=0.5)


def _sweep(P, model, Xc, variant="uEI_noiseless", utility=None):
    import bocf_b200
    acq = getattr(bocf_b200, variant)(model, None, utility=product_utility(P) if utility is None else utility)
    if hasattr(acq, "W_samples"):
        acq.W_samples = P.Z
    model.set_hyperparameters(0)
    a, g = acq._compute_acq_withGradients(np.ascontiguousarray(Xc))
    return np.asarray(a)[:, 0], np.asarray(g)


def _pools(P, model):
    """Candidates with a non-zero EI (focused draws) and with an exactly zero one (uniform draws)."""
    a, g = _sweep(P, model, P.Xc)
    k = P.N // 2                                             # make_problem puts the focused draws first
    act = P.Xc[:k][a[:k] > 0]
    idle = P.Xc[k:][a[k:] == 0]
    assert np.all(g[a == 0] == 0)
    assert len(act) > 200 and len(idle) > 200
    return act, idle


def _small_chunks(model, N):
    from bocf_b200 import _lib
    _lib.check(model._lib.bocf_model_set_scratch_limit(model._handle, ctypes.c_uint64(64 << 20)))
    chunk = model.chunk_candidates(N, grad=True)
    assert chunk % 128 == 0 and chunk >= 512
    return chunk


def test_result_independent_of_tile_mates(cuda_device):
    """Fixed active candidates at a tile's first and last row, both sides of a chunk border and in the ragged last chunk:
    bitwise the same whether their tile-mates are active or not; the inactive candidates get exactly zero."""
    P = _problem()
    model = product_model(P, cuda_device)
    act, idle = _pools(P, model)
    chunk = _small_chunks(model, 10 ** 6)
    N = 2 * chunk + chunk // 2 + 37                          # several chunks and a ragged last one
    assert model.chunk_candidates(N, grad=True) == chunk
    fixed = np.unique([0, 127, 128, 255, 384 + 64, chunk - 1, chunk, chunk + 127, 2 * chunk - 129, 2 * chunk,
                       N - 37, N - 1])
    rng = np.random.default_rng(5)
    X_fixed = act[rng.choice(len(act), len(fixed), replace=False)]
    XA = act[rng.integers(0, len(act), N)]
    XB = idle[rng.integers(0, len(idle), N)]
    XA[fixed] = X_fixed
    XB[fixed] = X_fixed
    aA, gA = _sweep(P, model, XA)
    aB, gB = _sweep(P, model, XB)
    assert np.all(aA > 0) and np.all(aB[fixed] > 0)
    assert np.array_equal(aA[fixed], aB[fixed]) and np.array_equal(gA[fixed], gB[fixed])
    rest = np.setdiff1d(np.arange(N), fixed)
    assert np.all(aB[rest] == 0) and np.all(gB[rest] == 0)


def test_skipped_unit_reads_no_stale_partials(cuda_device):
    """Chunk k is all active, chunk k+1 all inactive except one tile: every tile position of chunk k+1 that was active in
    chunk k now gets an exactly zero gradient; the one active tile matches its result in a sweep of its own size."""
    P = _problem()
    model = product_model(P, cuda_device)
    act, idle = _pools(P, model)
    chunk = _small_chunks(model, 10 ** 6)
    N = 3 * chunk
    rng = np.random.default_rng(6)
    X = idle[rng.integers(0, len(idle), N)]
    X[:chunk] = act[rng.integers(0, len(act), chunk)]
    X[2 * chunk + 256:2 * chunk + 384] = act[rng.integers(0, len(act), 128)]     # one tile of chunk 2
    a, g = _sweep(P, model, X)
    assert np.all(a[:chunk] > 0) and np.all(np.any(g[:chunk] != 0, axis=1))
    quiet = np.r_[chunk:2 * chunk + 256, 2 * chunk + 384:N]
    assert np.all(a[quiet] == 0) and np.all(g[quiet] == 0)
    # the same tile again, with the first two chunks inactive: the same bits
    Y = idle[rng.integers(0, len(idle), N)]
    Y[2 * chunk + 256:2 * chunk + 384] = X[2 * chunk + 256:2 * chunk + 384]
    a2, g2 = _sweep(P, model, Y)
    t = np.s_[2 * chunk + 256:2 * chunk + 384]
    assert np.array_equal(a2[t], a[t]) and np.array_equal(g2[t], g[t])
    assert np.all(a2[:2 * chunk] == 0) and np.all(g2[:2 * chunk] == 0)


def _margin(P, model, h):
    """max over utility parameters l and base samples s of U(theta_l, mu + sigma z_s) - f*_l under hyper-sample h (f* of
    hyper-sample 0): > 0 where the candidate has an improving sample under h.  Only picks the candidates to check."""
    model.set_hyperparameters(0)
    fX = np.asarray(model.posterior_mean_at_evaluated_points())                       # (m, n)
    fstar = np.max(-((fX.T[None, :, :] - P.theta[:, None, :]) ** 2).sum(-1), axis=1)   # (L,)
    model.set_hyperparameters(h)
    mu = np.asarray(model.posterior_mean(P.Xc)).T                                     # (N, m)
    sd = np.sqrt(np.asarray(model.posterior_variance_noiseless(P.Xc))).T
    y = mu[:, None, :] + sd[:, None, :] * P.Z[None, :, :]                              # (N, S, m)
    return np.max([np.max(-((y - t) ** 2).sum(-1), axis=1) - f for t, f in zip(P.theta, fstar)], axis=0)


def test_accumulation_over_hyper_samples(cuda_device):
    """H = 2 hyper-samples, L = 3 utility parameters: the sweep agrees with the oracle on candidates that improve under
    one hyper-sample only, under both and under neither, and a zero EI has an exactly zero gradient."""
    P = _problem(H=2, L=3, N=1200)
    model = product_model(P, cuda_device)
    a, g = _sweep(P, model, P.Xc)
    assert np.all(g[a == 0] == 0)
    mg = [_margin(P, model, h) for h in range(2)]
    one = np.nonzero((mg[0] > 0) != (mg[1] > 0))[0]
    both = np.nonzero((mg[0] > 0) & (mg[1] > 0))[0]
    none = np.nonzero((mg[0] <= 0) & (mg[1] <= 0))[0]
    assert len(one) >= 5 and len(both) >= 5 and len(none) >= 5, (len(one), len(both), len(none))
    rng = np.random.default_rng(8)
    idx = np.unique(np.concatenate([rng.choice(s_, min(30, len(s_)), replace=False) for s_ in (one, both, none)]))
    a_o, g_o = oracle_acq(P, grad=True, Xc=P.Xc[idx])
    assert np.count_nonzero(a_o) > 10 and np.count_nonzero(a_o == 0) > 5
    assert_close(a[idx], a_o, tol(1e-7), "acq")
    assert_close(g[idx], g_o, tol(1e-6), "grad acq")


def test_user_composite_weights(cuda_device):
    """The NVRTC-compiled MC kernel leaves the weights for a user composite: sumsq_target restated as user source."""
    import bocf_b200
    from bocf_b200.utility import _host_funcs
    from tests.user_composites import RESTATED
    P = _problem(N=2000)
    model = product_model(P, cuda_device)
    tl, src = RESTATED["sumsq_target"]
    U, dU = _host_funcs("sumsq_target")
    pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
    util = bocf_b200.Utility(func=U, dfunc=dU, parameter_dist=pd, composite=bocf_b200.CudaComposite(src, tl))
    a, g = _sweep(P, model, P.Xc, utility=util)
    a_b, g_b = _sweep(P, model, P.Xc)
    assert np.mean(a == 0) > 0.3 and np.all(g[a == 0] == 0)
    assert rel_err(a, a_b) < 1e-12 and rel_err(g, g_b) < 1e-12          # same operations as the built-in kernel
    rng = np.random.default_rng(9)
    idx = np.unique(np.concatenate([rng.choice(np.nonzero(a > 0)[0], 40, replace=False), rng.choice(P.N, 40, replace=False)]))
    a_o, g_o = oracle_acq(P, grad=True, Xc=P.Xc[idx])
    assert_close(a[idx], a_o, tol(1e-7), "acq")
    assert_close(g[idx], g_o, tol(1e-6), "grad acq")


def test_maei_weights(cuda_device):
    """maEI (linear scalarisation) leaves a non-zero weight for every candidate: every unit is walked."""
    from oracle import acquisitions as OA
    from tests.helpers import oracle_model, oracle_utility
    P = _problem(N=1500, composite="linear", seed=4)
    model = product_model(P, cuda_device)
    a, g = _sweep(P, model, P.Xc, variant="maEI")
    rng = np.random.default_rng(10)
    idx = np.unique(np.concatenate([np.arange(0, 130), rng.choice(P.N, 100, replace=False)]))
    om = oracle_model(P)
    om.set_hyperparameters(0)
    a_o, g_o = OA.maEI(om, utility=oracle_utility(P))._compute_acq_withGradients(P.Xc[idx])
    assert_close(a[idx], a_o[:, 0], tol(1e-8), "maEI")
    assert_close(g[idx], g_o, tol(1e-7), "grad maEI")
