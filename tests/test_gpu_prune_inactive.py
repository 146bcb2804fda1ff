"""Calls of at least 16384 candidates evaluate EI-CF / PI-CF only where the posterior mean cannot prove the acquisition
zero (api.cu: pruned sweep, acq.cu: prune_bound_kernel).  The results must be the full sweep's, bit for bit (+0 and -0
aside): the same candidates in slices below that size take the full sweep, so a pruned call is compared against slices.
Composites without a closed-form bound, user composites and the other variants must stay on the full sweep."""
import ctypes

import numpy as np
import pytest

from tests.helpers import make_problem, product_model, product_utility

pytestmark = pytest.mark.gpu

PRUNE_MIN_N = 16384                      # api.cu


def _problem(composite, seed=3, n=200):
    """m = 16 outputs (with few outputs hardly any uniform candidate can be proven inactive).  Except for sumsq_target,
    training point 0 is made clearly the best observation, and the first half of P.Xc are draws next to it."""
    P = make_problem(m=16, d=6, n=n, H=2, kind="matern52", composite=composite, N=4000, S=256, L=3, seed=seed,
                     focus=0.5)
    if composite != "sumsq_target":
        for j in range(P.m):
            y = P.Y[j]
            if composite == "linear":
                y[0, 0] += 6.0
            elif composite == "neg_sum_exp":
                y[0, 0] -= 6.0
            elif composite == "rosen_composite":
                y[0, 0] = 1.0 if j < P.m // 2 else 0.0
        rng = np.random.default_rng(40 + seed)
        P.Xc[:P.N // 2] = np.clip(P.X[0] + 0.05 * rng.standard_normal((P.N // 2, P.d)), 0, 1)
    return P


def _acq(P, model, variant, utility=None):
    import bocf_b200
    cls = {"ei": bocf_b200.uEI_noiseless, "pi": bocf_b200.uPI}[variant]
    acq = cls(model, None, utility=product_utility(P) if utility is None else utility)
    acq.W_samples = P.Z
    return acq


def _eval(acq, X, grad):
    """One bocf_acq_eval call over X (every hyper-sample, f* per hyper-sample); numpy (acq, grad acq or None)."""
    import torch
    from bocf_b200.utility import theta_matrix
    theta = theta_matrix(acq.utility, acq.utility.parameter_dist.support)
    fstar = acq._fstar(theta, per_hyper_sample=True)
    assert fstar.shape[0] == 2
    Zt = acq._Zt()
    Xd = torch.from_numpy(np.ascontiguousarray(X)).to(acq.model.device)
    a, g = acq._eval_device(acq._variant, Xd, theta, acq._weights(len(theta)), fstar, grad, Zt, Zt.shape[1], 0)
    torch.cuda.synchronize()
    return a.cpu().numpy(), (None if g is None else g.cpu().numpy())


def _profiled(fn):
    from bocf_b200 import _lib
    _lib.profile_enable(True)
    try:
        out = fn()
        prof = _lib.profile_report()
    finally:
        _lib.profile_enable(False)
    return out, prof


def _chunked(model):
    """Small chunks (several per call); returns (chunk, N, slice): a ragged last chunk, and slices below the pruning
    size.  Slices hold more than 1024 candidates, so that a slice's chunks take K*'s K-split (posterior.cu: chunks of
    <= 1024 candidates) exactly when the whole call's do: the K-split sums the mean in another order."""
    from bocf_b200 import _lib
    _lib.check(model._lib.bocf_model_set_scratch_limit(model._handle, ctypes.c_uint64(64 << 20)))
    chunk = model.chunk_candidates(10 ** 6, grad=True)
    assert 512 <= chunk < PRUNE_MIN_N // 2
    N = (40000 // chunk + 1) * chunk + chunk // 3 + 37
    return chunk, N, 6144


def _pool(P, model, N, chunk, kind, seed=5):
    """uniform: U[0,1]^d with a few improving candidates; focused: draws next to the best training points;
    training: a mix of training inputs, points next to them and uniform ones.  In uniform / training the first chunk is
    mostly uniform (the probe prunes), and the improving candidates sit at tile edges, chunk borders and the tail."""
    rng = np.random.default_rng(seed)
    X = rng.uniform(size=(N, P.d))
    focused = P.Xc[:P.N // 2]
    if kind == "focused":
        return focused[rng.integers(0, len(focused), N)]
    pos = np.unique(np.r_[[0, 127, 128, 255, chunk - 1, chunk, chunk + 127, 3 * chunk - 1, 3 * chunk, N - 37, N - 1],
                          rng.choice(np.arange(chunk, N), N // 10, replace=False)])
    if kind == "uniform":
        X[pos] = focused[rng.integers(0, len(focused), len(pos))]
    else:
        tr = P.X[rng.integers(0, P.n, len(pos))]
        near = np.clip(tr + 1e-7 * rng.standard_normal(tr.shape), 0, 1)
        X[pos] = np.where(rng.uniform(size=(len(pos), 1)) < 0.5, tr, near)
    return X


def _sliced(acq, X, sl, grad):
    bounds = list(range(0, len(X), sl)) + [len(X)]
    if bounds[-1] - bounds[-2] < 2048:                       # no short last slice
        del bounds[-2]
    assert all(2048 <= b - a < PRUNE_MIN_N for a, b in zip(bounds[:-1], bounds[1:]))
    parts = [_eval(acq, X[a:b], grad) for a, b in zip(bounds[:-1], bounds[1:])]
    a = np.concatenate([p[0] for p in parts])
    g = None if not grad else np.concatenate([p[1] for p in parts])
    return a, g


def _check_equal(full, ref):
    a, g = full
    ar, gr = ref
    assert np.array_equal(a, ar), "acq: %d of %d entries differ" % (np.count_nonzero(a != ar), len(a))
    if g is not None:
        assert np.array_equal(g, gr), "grad acq: %d rows differ" % np.count_nonzero(np.any(g != gr, axis=1))


@pytest.mark.parametrize("composite", ["sumsq_target", "rosen_composite", "neg_sum_exp", "linear"])
@pytest.mark.parametrize("variant,grad", [("ei", False), ("ei", True), ("pi", False)])
def test_pruned_equals_full_sweep(cuda_device, composite, variant, grad):
    """H = 2, L = 3, several chunks and a ragged last one: a pruned call against the same candidates in slices."""
    P = _problem(composite)
    model = product_model(P, cuda_device)
    acq = _acq(P, model, variant)
    chunk, N, sl = _chunked(model)
    X = _pool(P, model, N, chunk, "uniform")
    full, prof = _profiled(lambda: _eval(acq, X, grad))
    assert prof["prune_list_kernel"][0] == 2 and "prune_bound_kernel" in prof, prof     # probe + full list: pruned
    ref = _sliced(acq, X, sl, grad)
    _check_equal(full, ref)
    a = full[0]
    assert np.count_nonzero(a) > 50 and np.count_nonzero(a == 0) > N // 2


def test_smallest_chunk(cuda_device):
    """The smallest chunk the library picks (256 candidates: n = 600 at the 64 MiB scratch floor), H = 2, L = 3, fused
    gradient: a short last survivor chunk is padded to 129 candidates inside the chunk."""
    P = _problem("neg_sum_exp", n=600)
    model = product_model(P, cuda_device)
    acq = _acq(P, model, "ei")
    from bocf_b200 import _lib
    _lib.check(model._lib.bocf_model_set_scratch_limit(model._handle, ctypes.c_uint64(64 << 20)))
    assert model.chunk_candidates(10 ** 6, grad=True) == 256
    N = 160 * 256 + 200                                      # last chunk of the full sweep: 200 > 128 candidates
    X = _pool(P, model, N, 256, "uniform")
    full, prof = _profiled(lambda: _eval(acq, X, True))
    assert prof["prune_list_kernel"][0] == 2, prof
    n, kept = ctypes.c_int64(0), ctypes.c_int64(0)
    _lib.check(model._lib.bocf_model_sweep_stats(model._handle, ctypes.byref(n), ctypes.byref(kept)))
    assert n.value == N and 0 < kept.value < N // 2
    _check_equal(full, _sliced(acq, X, 6144, True))
    assert np.count_nonzero(full[0]) > 50


@pytest.mark.parametrize("kind", ["focused", "training"])
def test_focused_and_training_candidates(cuda_device, kind):
    """Candidates concentrated next to the incumbent (the probe keeps them: full sweep) and candidates at and next to
    training inputs (pruned): the same bits as the slices, value and fused gradient."""
    P = _problem("sumsq_target")
    model = product_model(P, cuda_device)
    acq = _acq(P, model, "ei")
    chunk, N, sl = _chunked(model)
    X = _pool(P, model, N, chunk, kind)
    full, prof = _profiled(lambda: _eval(acq, X, True))
    assert prof["prune_list_kernel"][0] == (1 if kind == "focused" else 2), prof
    _check_equal(full, _sliced(acq, X, sl, True))


@pytest.mark.parametrize("which", ["exp_cos", "user"])
def test_other_composites_stay_dense(cuda_device, which):
    """exp_cos has no closed-form bound and a user composite is opaque: neither runs the bound."""
    import bocf_b200
    from bocf_b200.utility import _host_funcs
    from tests.user_composites import RESTATED
    P = _problem("exp_cos" if which == "exp_cos" else "sumsq_target")
    model = product_model(P, cuda_device)
    util = None
    if which == "user":
        tl, src = RESTATED["sumsq_target"]
        U, dU = _host_funcs("sumsq_target")
        pd = bocf_b200.ParameterDistribution(support=P.theta, prob_dist=P.prob)
        util = bocf_b200.Utility(func=U, dfunc=dU, parameter_dist=pd, composite=bocf_b200.CudaComposite(src, tl))
    acq = _acq(P, model, "ei", utility=util)
    chunk, N, sl = _chunked(model)
    X = _pool(P, model, N, chunk, "uniform")
    full, prof = _profiled(lambda: _eval(acq, X, True))
    assert "prune_bound_kernel" not in prof, prof
    _check_equal(full, _sliced(acq, X, sl, True))


def test_nan_candidate_survives(cuda_device):
    """A candidate with a NaN input cannot be proven inactive, and the others are unaffected by it.  (Its own gradient is
    NaN or zero depending on whether a tile-mate is active, in either sweep, so only its value is compared.)"""
    P = _problem("sumsq_target")
    model = product_model(P, cuda_device)
    acq = _acq(P, model, "ei")
    chunk, N, sl = _chunked(model)
    X = _pool(P, model, N, chunk, "uniform")
    bad = [5, chunk + 3, N - 2]
    X[bad, 1] = np.nan
    full, prof = _profiled(lambda: _eval(acq, X, True))
    assert prof["prune_list_kernel"][0] == 2, prof
    ref = _sliced(acq, X, sl, True)
    ok = np.setdiff1d(np.arange(N), bad)
    _check_equal((full[0][ok], full[1][ok]), (ref[0][ok], ref[1][ok]))
    assert np.array_equal(full[0][bad], ref[0][bad], equal_nan=True)


def test_host_entry_pruned(cuda_device):
    """bocf_acq_eval_host (numpy in, numpy out through the handle's staging) prunes the same way."""
    import bocf_b200
    from bocf_b200.utility import theta_matrix
    P = _problem("sumsq_target")
    model = product_model(P, cuda_device)
    acq = _acq(P, model, "ei")
    chunk, N, sl = _chunked(model)
    X = _pool(P, model, N, chunk, "uniform")
    theta = theta_matrix(acq.utility, acq.utility.parameter_dist.support)
    fstar = acq._fstar(theta, per_hyper_sample=True)
    Zt = acq._Zt()
    args = (acq._variant, np.ascontiguousarray(X), theta, acq._weights(len(theta)), fstar, True, Zt, Zt.shape[1], 0)
    (a, g), prof = _profiled(lambda: acq._eval_host_small(*args))
    assert prof["prune_list_kernel"][0] == 2, prof
    _check_equal((a[:, 0], g), _sliced(acq, X, sl, True))
    assert isinstance(acq, bocf_b200.uEI_noiseless)


@pytest.mark.parametrize("N", [300, 5000])
def test_mean_only_pass_is_bitwise(cuda_device, N):
    """The mean-only K* pass (posterior mean alone) gives the bits of the passes that also write K*, digit planes, G* and
    the mean gradient, with and without the K-split of small chunks."""
    P = make_problem(m=5, d=7, n=300, H=1, kind=["matern52", "matern52", "rbf", "se", "matern32"],
                     composite="sumsq_target", N=N, S=64, seed=4)
    model = product_model(P, cuda_device)
    X = np.concatenate([P.Xc, P.X[:50], P.X[:50] + 1e-9])
    (mu0, _, _, _), prof = _profiled(lambda: model._posterior(X))
    assert "kstar_mean_kernel" in prof and "kstar_kernel" not in prof, prof
    mu1 = model._posterior(X, want_var=True)[0]
    mu2 = model._posterior(X, want_var=True, want_dmean=True, want_dvar=True)[0]
    assert np.array_equal(mu0, mu1) and np.array_equal(mu0, mu2)
