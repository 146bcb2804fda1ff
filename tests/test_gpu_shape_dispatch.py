"""Every shape-dispatched kernel instantiation against the CPU oracle.

Most of the hot path picks a template instantiation on the host, from the problem's shape and the precision mode:
  * the input-dimension bucket DP (d <= 4, 6, 8, 10, 12, 16) of kstar_kernel (posterior.cu launch_kstar_k) and of the
    second contraction, EPI_DVAR and the fused EPI_DACQ (split_gemm.cu launch_grad);
  * the first contraction with the re-split of V, one instantiation per (scheme, S2) pair (split_gemm.cu launch_var);
  * the digit output SPL of kstar_kernel (0 in fp64 mode, 5 or 6 with digit planes);
  * the MC pass shape (acq.cu launch_mc_t: <= 128 candidates, <= 1024, larger) and its gradient weights in one or two
    register words (m <= 32 / <= 64);
  * the K-split of kstar_kernel (chunks of <= 1024 candidates) and the final gradient sum (<= 128 candidates);
  * maEI / maPI: a register path with a fused gradient for m <= 16, a generic loop with per-output dmean / dvar above.
Each section below walks one of these grids at both ends of every bucket, with m and n that are multiples of no tile
(column tiles of 32 / 48 / 64, K chunks of 64, Cholesky tiles of 128).  tests/test_dispatch_tables_cpu.py parses the
dispatch ladders out of the sources and checks that the case lists here still cover them.

Bars are the project's: in fp64 mode 1e-8 on acq and the posterior mean, 1e-7 on grad acq, the variance and its
gradient, norm-wise and element-wise; tests.helpers.tol() widens them to 1e-6 under the default "auto" precision, where
the variance gradient is held norm-wise only (see _check_posterior).
"""
import functools
import os

import numpy as np
import pytest

from tests.helpers import assert_close, make_problem, oracle_acq, oracle_model, product_acq, product_model, rel_err, tol

pytestmark = pytest.mark.gpu

# section a: both ends of every DP bucket; the tiny MC pass (17) and the sweep with a ragged last tile (1300)
BUCKET_DS = [1, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 16]
BUCKET_NS = [17, 1300]
# section b: (precision, (scheme of the variance contraction, scheme of the variance-gradient contraction)), one per
# launch_var instantiation: 3313, 4423, 4424, 5544, 5545, 6655, 6656
SCHEME_CASES = [("split3", (331, 331)), ("mixed", (442, 331)), ("split4", (442, 442)), ("split54", (554, 442)),
                ("split5", (554, 554)), ("split65", (665, 554)), ("split6", (665, 665))]
SCHEME_DS = [4, 12, 16]
# section c: outputs past the 16 of the maEI register path and the 32 of the first MC weight word
WIDE_MS = [17, 32, 33, 64]
WIDE_COMPOSITES = ["sumsq_target", "neg_sum_exp", "linear"]
MA_MS = [16, 17, 64]
# section d: both sides of 128 (tiny MC pass, small final gradient sum) and of 1024 (small MC pass, K* K-split)
BATCH_EDGE_NS = [1, 128, 129, 1024, 1025]


try:
    from threadpoolctl import threadpool_limits
except ImportError:                          # only the oracle's speed depends on it
    threadpool_limits = None


def _oracle(fn):
    """Cache an oracle computation (the cases of both precision modes compare with it) and run it on one BLAS thread:
    its many small LAPACK calls take several times longer with a thread pool."""
    @functools.lru_cache(maxsize=None)
    @functools.wraps(fn)
    def run(*args):
        if threadpool_limits is None:
            return fn(*args)
        with threadpool_limits(limits=1, user_api="blas"):
            return fn(*args)
    return run


def _mode():
    return os.environ.get("BOCF_PRECISION", "auto")


def _posterior_o(om, X, H):
    out = []
    for h in range(H):
        om.set_hyperparameters(h)
        out.append((om.posterior_mean(X), om.posterior_variance(X), om.posterior_mean_gradient(X),
                    om.posterior_variance_gradient(X)))
    return out


def _check_posterior(pm, X, ref, tol_mean, tol_var):
    for h, (mu_o, v_o, dm_o, dv_o) in enumerate(ref):
        pm.set_hyperparameters(h)
        mu, v = pm.posterior_mean(X), pm.posterior_variance(X)
        dm, dv = pm.posterior_mean_gradient(X), pm.posterior_variance_gradient(X)
        assert_close(mu, mu_o, tol_mean, "mean h=%d" % h)
        assert np.max(np.abs(v - v_o) / v_o) < tol_var, ("var h=%d" % h, np.max(np.abs(v - v_o) / v_o))
        assert_close(dm, dm_o, tol_mean, "dmean h=%d" % h)
        assert rel_err(dv, dv_o) < tol_var, ("dvar h=%d" % h, rel_err(dv, dv_o))
        if _mode() == "fp64":
            # With digit planes the variance gradient runs on 13 pairs (442), whose error is ~1e-7 of the LARGEST entry
            # (api.cu apply_precision).  At d = 1 that is 1.3e-5 of the smallest entries above the element-wise floor,
            # measured on a B200; the CPU digit-plane model of tests/test_split_numerics.py gives 1.5e-5 for the same
            # problem.  So the element-wise check of the variance gradient is the fp64 mode's alone.
            assert_close(dv, dv_o, tol_var, "dvar h=%d" % h)


def _check_eicf(a, g, a_o, g_o, tol_a, tol_g):
    assert np.mean(a_o > 0) > 0.02, "degenerate test problem"
    assert_close(a, a_o, tol_a, "acq")
    if g is not None:
        assert_close(g, g_o, tol_g, "grad acq")
    assert int(np.argmax(a)) == int(np.argmax(a_o))


# ---- a. every DP bucket, both ends -------------------------------------------------------------------------------

def _bucket_problem(d, N):
    return make_problem(m=3, d=d, n=150, H=2, kind="matern52", composite="sumsq_target", N=N, S=256, L=2,
                        seed=100 + d)


@_oracle
def _bucket_oracle(d, N):
    P = _bucket_problem(d, N)
    om = oracle_model(P)
    a_o, g_o = oracle_acq(P, grad=True, model=om)
    return _posterior_o(om, P.Xc, P.H), a_o, g_o


@pytest.mark.parametrize("N", BUCKET_NS)
@pytest.mark.parametrize("d", BUCKET_DS)
def test_every_input_dimension_bucket(cuda_device, d, N):
    """kstar_kernel and the second contraction at both ends of every DP bucket: posterior mean / variance and their
    gradients, and the EI-CF value with its fused gradient."""
    P = _bucket_problem(d, N)
    post_o, a_o, g_o = _bucket_oracle(d, N)
    pm = product_model(P, cuda_device)
    _check_posterior(pm, P.Xc, post_o, tol(1e-8), tol(1e-7))
    a, g = product_acq(P, grad=True, device=cuda_device, model=pm)
    _check_eicf(a, g, a_o, g_o, tol(1e-8), tol(1e-7))


# ---- b. every digit-pair scheme x DP bucket ----------------------------------------------------------------------

@pytest.fixture
def split_device(built_library):      # these tests name their precision explicitly: no mode parametrisation
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return "cuda:0"


# split3 (8 digit pairs in both contractions) has no bar of its own: these are 4x the largest errors measured over
# d = 4, 12, 16 on an NVIDIA B200 at a 1000 W power limit -- variance 2.36e-4 (element-wise, at d = 4), variance
# gradient 2.07e-5, acq 1.35e-5, grad acq 1.92e-5 (norm-wise).
SPLIT3_BARS = {"var": 9.44e-4, "dvar": 8.28e-5, "acq": 5.4e-5, "grad": 7.68e-5}
SCHEME_BARS = {"split3": SPLIT3_BARS,
               "mixed": dict.fromkeys(("var", "dvar", "acq", "grad"), 1e-4),
               "split4": dict.fromkeys(("var", "dvar", "acq", "grad"), 1e-4),
               "split54": dict.fromkeys(("var", "dvar", "acq", "grad"), 1e-6),
               "split5": dict.fromkeys(("var", "dvar", "acq", "grad"), 1e-6),
               "split65": dict.fromkeys(("var", "dvar", "acq", "grad"), 1e-6),
               "split6": {"var": 1e-8, "dvar": 1e-7, "acq": 1e-7, "grad": 1e-7}}


def _scheme_problem(d):
    return make_problem(m=4, d=d, n=200, H=1, kind="matern52", composite="sumsq_target", N=600, S=128, seed=200 + d)


@_oracle
def _scheme_oracle(d):
    P = _scheme_problem(d)
    om = oracle_model(P)
    a_o, g_o = oracle_acq(P, grad=True, model=om)
    return _posterior_o(om, P.Xc, P.H)[0], a_o, g_o


@pytest.mark.parametrize("d", SCHEME_DS)
@pytest.mark.parametrize("prec,schemes", SCHEME_CASES)
def test_every_scheme_in_every_bucket(split_device, prec, schemes, d):
    """Both contractions under every digit-pair scheme the library instantiates, at the low, a middle and the top DP
    bucket of the second one.  The mean and its gradient come out of the digit-writing kstar_kernel variants (SPL 5 or
    6) and stay fp64."""
    P = _scheme_problem(d)
    (mu_o, v_o, dm_o, dv_o), a_o, g_o = _scheme_oracle(d)
    bar = SCHEME_BARS[prec]
    pm = product_model(P, split_device, precision=prec)
    assert pm.active_scheme() == schemes, (prec, pm.active_scheme())
    mu, v = pm.posterior_mean(P.Xc), pm.posterior_variance(P.Xc)
    dm, dv = pm.posterior_mean_gradient(P.Xc), pm.posterior_variance_gradient(P.Xc)
    assert_close(mu, mu_o, 1e-8, "mean")
    assert_close(dm, dm_o, 1e-8, "dmean")
    err = {"var": np.max(np.abs(v - v_o) / v_o), "dvar": rel_err(dv, dv_o)}
    a, g = product_acq(P, grad=True, device=split_device, model=pm)
    assert np.mean(a_o > 0) > 0.02, "degenerate test problem"
    err["acq"], err["grad"] = rel_err(a, a_o), rel_err(g, g_o)
    print("scheme errors %s d=%d: %s" % (prec, d, " ".join("%s %.2e" % kv for kv in sorted(err.items()))))
    for k, e in err.items():
        assert e < bar[k], (prec, k, e, bar[k])
    assert int(np.argmax(a)) == int(np.argmax(a_o))


def test_unsupported_split_pairs_are_rejected(split_device, monkeypatch):
    """A (variance, gradient) plane pair without a first-contraction instantiation is refused when it is requested,
    not at the first variance call; a refused request leaves the handle as it was."""
    from bocf_b200 import _lib
    P = make_problem(m=2, d=3, n=60, H=1, kind="matern52", N=40, S=4, seed=5)
    pm = product_model(P, split_device, precision="split54")
    v0 = pm.posterior_variance(P.Xc)
    for slices in (53, 63, 64, 32, 2, 7, 67, 76):
        assert pm._lib.bocf_model_set_precision(pm._handle, 1, slices, None) == -1, slices
        assert pm.active_scheme() == (554, 442)
    assert np.array_equal(pm.posterior_variance(P.Xc), v0)
    for bad in ("split53", "split64", "split7", "fp32", "split"):
        monkeypatch.setenv("BOCF_PRECISION", bad)
        with pytest.raises(_lib.BocfError) as ei:
            product_model(P, split_device)
        assert ei.value.code == -1 and "BOCF_PRECISION" in str(ei.value), bad
    monkeypatch.setenv("BOCF_PRECISION", "split65")
    assert product_model(P, split_device).active_scheme() == (665, 554)


# ---- c. outputs beyond 16 ----------------------------------------------------------------------------------------

def _wide_problem(m, d, N, composite):
    # with tens of outputs, few candidates improve on the incumbent unless they sit close to the best training points
    return make_problem(m=m, d=d, n=100, H=2, kind="matern52", composite=composite, N=N, S=256, L=2,
                        seed=300 + m + d, focus=0.9, focus_scale=0.03)


@_oracle
def _wide_oracle(m, d, N, composite):
    P = _wide_problem(m, d, N, composite)
    om = oracle_model(P)
    a_o, g_o = oracle_acq(P, grad=True, model=om)
    pi_o, _ = oracle_acq(P, grad=False, variant="uPI", model=om)
    return a_o, g_o, pi_o


@pytest.mark.parametrize("N", [17, 300])
@pytest.mark.parametrize("d", [3, 9])
@pytest.mark.parametrize("m", WIDE_MS)
@pytest.mark.parametrize("composite", WIDE_COMPOSITES)
def test_mc_acquisitions_past_16_outputs(cuda_device, composite, m, d, N):
    """EI-CF value and gradient (the second gradient-weight word of the MC pass past 32 outputs) and PI-CF."""
    P = _wide_problem(m, d, N, composite)
    a_o, g_o, pi_o = _wide_oracle(m, d, N, composite)
    pm = product_model(P, cuda_device)
    a, g = product_acq(P, grad=True, device=cuda_device, model=pm)
    _check_eicf(a, g, a_o, g_o, tol(1e-8), tol(1e-7))
    pi, _ = product_acq(P, grad=False, variant="uPI", device=cuda_device, model=pm)
    assert np.mean(pi_o > 0) > 0.02, "degenerate test problem"
    assert np.max(np.abs(pi - pi_o)) < tol(1e-12)       # counts / (H S): exact up to the final scaling


def _ma_problem(m, d, N):
    return make_problem(m=m, d=d, n=100, H=2, kind="matern52", composite="linear", N=N, S=4, L=3, seed=400 + m + d)


@_oracle
def _ma_oracle(variant, m, d, N):
    P = _ma_problem(m, d, N)
    om = oracle_model(P)
    a_o, g_o = oracle_acq(P, grad=True, variant=variant, model=om)
    av_o, _ = oracle_acq(P, grad=False, variant=variant, model=om)
    return a_o, g_o, av_o


@pytest.mark.parametrize("N", [17, 300])
@pytest.mark.parametrize("d", [3, 9])
@pytest.mark.parametrize("m", MA_MS)
@pytest.mark.parametrize("variant", ["maEI", "maPI"])
def test_analytic_acquisitions_both_sides_of_16_outputs(cuda_device, variant, m, d, N):
    """maEI / maPI at 16 outputs (register path; fused gradient with digit planes) and at 17 and 64 (generic loop over
    per-output dmean / dvar, also with digit planes), held to the same bars."""
    P = _ma_problem(m, d, N)
    a_o, g_o, av_o = _ma_oracle(variant, m, d, N)
    pm = product_model(P, cuda_device)
    if _mode() == "auto":
        assert pm.active_slices() > 0            # the digit-plane contractions, fused (m <= 16) or not, are what runs
    a, g = product_acq(P, grad=True, variant=variant, device=cuda_device, model=pm)
    assert_close(a, a_o, tol(1e-8), "acq")
    assert_close(g, g_o, tol(1e-7), "grad acq")
    av, _ = product_acq(P, grad=False, variant=variant, device=cuda_device, model=pm)
    assert_close(av, av_o, tol(1e-8), "acq value only")


@_oracle
def _m65_oracle():
    P = make_problem(m=65, d=3, n=100, H=2, kind="matern52", composite="linear", N=300, S=64, L=2, seed=465)
    om = oracle_model(P)
    post = _posterior_o(om, P.Xc, P.H)
    return P, [(mu, v) for mu, v, _, _ in post], oracle_acq(P, grad=True, variant="maEI", model=om)


def test_65_outputs(cuda_device):
    """Past MAXM = 64 the posterior and maEI (no output limit) still match the oracle; the MC acquisitions refuse the
    call with BOCF_ERR_UNSUPPORTED and leave the device usable."""
    from bocf_b200 import _lib
    P, post_o, (a_o, g_o) = _m65_oracle()
    pm = product_model(P, cuda_device)
    for h, (mu_o, v_o) in enumerate(post_o):
        pm.set_hyperparameters(h)
        assert_close(pm.posterior_mean(P.Xc), mu_o, tol(1e-8), "mean")
        v = pm.posterior_variance(P.Xc)
        assert np.max(np.abs(v - v_o) / v_o) < tol(1e-7)
    for grad, variant in ((True, "uEI_noiseless"), (False, "uEI_noiseless"), (False, "uPI")):
        with pytest.raises(_lib.BocfError) as ei:
            product_acq(P, grad=grad, variant=variant, device=cuda_device, model=pm)
        assert ei.value.code == -5, (variant, grad, str(ei.value))
    a, g = product_acq(P, grad=True, variant="maEI", device=cuda_device, model=pm)
    assert_close(a, a_o, tol(1e-8), "maEI")
    assert_close(g, g_o, tol(1e-7), "grad maEI")


# ---- d. batch-size edges at a large shape ------------------------------------------------------------------------

@_oracle
def _edge_case():
    """One pool of candidates, each batch a prefix of it.  make_problem puts its focused draws first; the first candidate
    that improves on the incumbent is swapped to the front, so that the one-candidate batch is not all zero."""
    P = make_problem(m=20, d=11, n=300, H=2, kind="matern52", composite="sumsq_target", N=max(BATCH_EDGE_NS), S=256,
                     L=2, seed=500, focus=0.9, focus_scale=0.03)
    om = oracle_model(P)
    a_o, g_o = oracle_acq(P, grad=True, model=om)
    perm = np.arange(P.N)
    k = int(np.argmax(a_o > 0))
    perm[[0, k]] = perm[[k, 0]]
    P.Xc = np.ascontiguousarray(P.Xc[perm])
    return P, _posterior_o(om, P.Xc, P.H), a_o[perm], g_o[perm]


@pytest.mark.parametrize("N,on_device", [(N, False) for N in BATCH_EDGE_NS] + [(128, True)])
def test_batch_size_edges(cuda_device, N, on_device):
    """m = 20, d = 11 on both sides of the 128- and 1024-candidate edges.  One case hands the batch over as a device
    tensor (bocf_acq_eval); numpy batches of this size take the host-buffer entry (bocf_acq_eval_host)."""
    import torch
    P, post_o, a_o, g_o = _edge_case()
    X = np.ascontiguousarray(P.Xc[:N])
    pm = product_model(P, cuda_device)
    chunk = pm.chunk_candidates(N, grad=True)
    assert chunk >= N and (chunk <= 1024) == (N <= 1024)       # one chunk; the K* K-split runs iff it is <= 1024
    _check_posterior(pm, X, [tuple(r[:, :N] for r in p) for p in post_o], tol(1e-8), tol(1e-7))
    a, g = product_acq(P, grad=True, device=cuda_device, model=pm, Xc=torch.from_numpy(X).to(cuda_device)
                       if on_device else X)
    if on_device:
        a, g = a.cpu().numpy(), g.cpu().numpy()
    _check_eicf(a, g, a_o[:N], g_o[:N], tol(1e-8), tol(1e-7))
