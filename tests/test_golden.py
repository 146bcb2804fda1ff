"""Golden vectors produced by the REFERENCE's own code (tests/golden/make_golden.py runs the real
uEI_noiseless / uPI / maEI / maPI / EI / PI, multi_outputGP, GPModel, GPy GP / kernels / LAPACK wrappers).

* CPU (-m "not gpu"): pins the oracle restatement to those vectors.
* GPU (-m gpu): the CUDA path against the same vectors, through the plugin classes / C ABI.
"""
import glob
import os

import numpy as np
import pytest

from tests.helpers import tol, Problem, oracle_model, oracle_acq, product_model, product_acq, rel_err

GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.npz"))
                if not os.path.basename(p).startswith(("lml_", "hmc_", "kg_", "grad_x_")))   # lml_*: test_lml.py, hmc_*: test_hmc.py, kg_*: test_kg.py, grad_x_*: test_oracle.py
IDS = [os.path.basename(p)[:-4] for p in GOLDEN]


def load_case(path):
    z = np.load(path, allow_pickle=False)
    P = Problem()
    P.X, P.Xc, P.Z, P.theta, P.prob = z["X"], z["Xc"], z["Z"], z["theta"], z["prob"]
    P.variance, P.lengthscale, P.noise = z["variance"], z["lengthscale"], z["noise"]
    P.kind, P.composite = str(z["kind"]), str(z["composite"])
    P.H, P.m = P.variance.shape
    P.n, P.d = P.X.shape
    P.N, P.S, P.L = P.Xc.shape[0], P.Z.shape[0], P.theta.shape[0]
    P.Y = [z["Y"][j].reshape(-1, 1) for j in range(P.m)]
    return P, z, str(z["acq"])


def test_fixtures_present():
    assert len(GOLDEN) >= 11


@pytest.mark.parametrize("path", GOLDEN, ids=IDS)
def test_oracle_reproduces_reference_posterior(path):
    P, z, _ = load_case(path)
    om = oracle_model(P)
    for h in range(P.H):
        om.set_hyperparameters(h)
        # the restatement follows the reference operation by operation: agreement is at rounding level
        assert rel_err(om.posterior_mean(P.Xc), z["mean_h%d" % h]) < 1e-13
        assert rel_err(om.posterior_variance(P.Xc), z["var_h%d" % h]) < 1e-12
        assert rel_err(om.posterior_mean_gradient(P.Xc), z["dmean_h%d" % h]) < 1e-12
        assert rel_err(om.posterior_variance_gradient(P.Xc), z["dvar_h%d" % h]) < 1e-11
        pm, pv = om.predict(P.Xc)
        assert rel_err(pm, z["pmean_h%d" % h]) < 1e-13 and rel_err(pv, z["pvar_h%d" % h]) < 1e-12
        assert rel_err(om.posterior_variance_noiseless(P.Xc), z["varnl_h%d" % h]) < 1e-11
    om.set_hyperparameters(0)
    assert rel_err(om.posterior_mean_at_evaluated_points(), z["mean_train_h0"]) < 1e-13


@pytest.mark.parametrize("path", GOLDEN, ids=IDS)
@pytest.mark.parametrize("vectorised", [False, True])
def test_oracle_reproduces_reference_acquisition(path, vectorised):
    P, z, acq_name = load_case(path)
    if vectorised and acq_name not in ("uEI_noiseless", "uPI"):
        pytest.skip("analytic variants have a single (literal) restatement")
    a, _ = oracle_acq(P, grad=False, variant=acq_name, vectorised=vectorised, parallel=False)
    assert rel_err(a, z["acq_value"][:, 0]) < 1e-12
    if "acq_value_pool" in z.files:     # pathos branch: f* re-evaluated per hyper-sample (differs when H > 1)
        a, _ = oracle_acq(P, grad=False, variant=acq_name, vectorised=vectorised, parallel=True)
        assert rel_err(a, z["acq_value_pool"][:, 0]) < 1e-12
    if "acq_grad" in z.files:
        a, g = oracle_acq(P, grad=True, variant=acq_name, vectorised=vectorised)
        assert rel_err(a, z["acq_grad_value"][:, 0]) < 1e-12
        assert rel_err(g, z["acq_grad"]) < 1e-11


# ---- the CUDA path against the reference's vectors ----------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=IDS)
def test_cuda_matches_reference_golden(cuda_device, path):
    P, z, acq_name = load_case(path)
    pm = product_model(P, cuda_device)
    for h in range(P.H):
        pm.set_hyperparameters(h)
        assert rel_err(pm.posterior_mean(P.Xc), z["mean_h%d" % h]) < 1e-6       # north-star fp64 bar
        assert rel_err(pm.posterior_variance(P.Xc), z["var_h%d" % h]) < 1e-6
        assert rel_err(pm.posterior_mean(P.Xc), z["mean_h%d" % h]) < tol(1e-9)
        assert rel_err(pm.posterior_variance(P.Xc), z["var_h%d" % h]) < tol(1e-8)
        assert rel_err(pm.posterior_mean_gradient(P.Xc), z["dmean_h%d" % h]) < tol(1e-8)
        assert rel_err(pm.posterior_variance_gradient(P.Xc), z["dvar_h%d" % h]) < tol(1e-7)
        mp, vp = pm.predict(P.Xc)
        assert rel_err(mp, z["pmean_h%d" % h]) < tol(1e-9) and rel_err(vp, z["pvar_h%d" % h]) < tol(1e-8)
    a, _ = product_acq(P, grad=False, variant=acq_name, device=cuda_device, model=pm, parallel=False)
    assert rel_err(a, z["acq_value"][:, 0]) < tol(1e-8)
    assert np.argmax(a) == np.argmax(z["acq_value"][:, 0])
    if "acq_value_pool" in z.files:
        a, _ = product_acq(P, grad=False, variant=acq_name, device=cuda_device, model=pm, parallel=True)
        assert rel_err(a, z["acq_value_pool"][:, 0]) < tol(1e-8)
    if "acq_grad" in z.files:
        a, g = product_acq(P, grad=True, variant=acq_name, device=cuda_device, model=pm)
        assert rel_err(a, z["acq_grad_value"][:, 0]) < tol(1e-8)
        assert rel_err(g, z["acq_grad"]) < tol(1e-7)
