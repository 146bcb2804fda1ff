"""Utility / ParameterDistribution with the reference's interface (utility.py:6-48,
parameter_distribution.py:5-29).

The reference passes arbitrary Python callables ``func`` / ``dfunc``; the device path needs the
composite as device code instead, selected by ``composite=``: either the name of one of the catalogued
device functions (the U(theta, y) found in the reference's experiment scripts, SURVEY.md Appendix A) or
a ``CudaComposite``, the user's own U and dU/dy in CUDA C++, compiled at run time.  ``func``/``dfunc``
stay available as host callables for the parts of the BO loop that evaluate the true objective.
"""
import ctypes

import numpy as np

from . import _lib
from ._lib import COMPOSITES


def _host_funcs(name):
    if name == "sumsq_target":       # test_1a.py:89-96
        return (lambda th, y: -np.sum(np.square((np.asarray(y).T - th).T), axis=0),
                lambda th, y: -2 * (np.squeeze(y) - th))
    if name == "neg_sum_exp":        # test_2a.py:60-65
        return (lambda th, y: np.sum(-np.exp(y), axis=0), lambda th, y: -np.exp(y))
    if name == "exp_cos":            # test_3a.py:53-67
        c = np.array([1., 2., 5., 2., 3.])

        def U(th, y):
            y = np.asarray(y)
            return -np.tensordot(c[np.arange(y.shape[0]) % 5], np.exp(-y / np.pi) * np.cos(np.pi * y), axes=1)

        def dU(th, y):
            y = np.squeeze(y)
            aux = -np.pi * np.exp(-y / np.pi) * np.sin(np.pi * y) - np.exp(-y / np.pi) * np.cos(np.pi * y) / np.pi
            return -c[np.arange(len(y)) % 5] * aux
        return U, dU
    if name == "rosen_composite":    # test_5a.py:48-59
        def U(a, y):
            y = np.asarray(y)
            h = y.shape[0] // 2
            a = float(np.asarray(a).reshape(-1)[0])
            return -np.sum((a - y[:h]) ** 2 + 100 * y[h:2 * h] ** 2, axis=0)

        def dU(a, y):
            y = np.squeeze(y)
            h = len(y) // 2
            a = float(np.asarray(a).reshape(-1)[0])
            g = np.zeros(len(y))
            g[:h] = 2 * (a - y[:h])
            g[h:2 * h] = -200 * y[h:2 * h]
            return g
        return U, dU
    if name == "linear":             # test_1b.py:89-93
        return (lambda th, y: np.dot(th, y), lambda th, y: th)
    raise ValueError("unknown composite %r (known: %s)" % (name, sorted(COMPOSITES)))


# length of one utility parameter: "m" = one entry per output, 1 = a scalar
THETA_DIM = {"sumsq_target": "m", "linear": "m", "neg_sum_exp": 1, "exp_cos": 1, "rosen_composite": 1}


def theta_matrix(utility, samples):
    """Utility parameters as an (L, p) matrix.  A 1-D support is L scalar parameters for the composites that take a
    scalar or none (test_5a.py:41: np.atleast_1d([1.]) -- the reference iterates len(support)), L parameters of a
    fixed length k > 1 laid end to end, or one vector for a composite with one entry per output."""
    th = np.asarray(samples, dtype=np.float64)
    tl = utility.theta_len
    if th.ndim == 0:
        th = th.reshape(1, 1)
    elif th.ndim == 1:
        if tl == "m":
            th = th.reshape(1, -1)
        else:
            th = th.reshape(-1, max(1, tl))
    return np.ascontiguousarray(th)


class CudaComposite(object):
    """A user-defined composite U(theta, y) in CUDA C++: ``source`` defines ``bocf_U`` and ``bocf_dU`` for BOCF_M
    outputs (the contract next to ``enum bocf_composite`` in include/bocf_b200.h).  ``theta_len``: entries of one
    utility parameter, "m" for one per output or a fixed count >= 0.

    The source is compiled by NVRTC for sm_100a once per number of outputs, the first time a model with that many
    outputs uses it (bocf_composite_register).  Pass it as ``Utility(func=..., dfunc=..., composite=...)``."""

    def __init__(self, source, theta_len="m"):
        if not isinstance(source, str) or not source.strip():
            raise ValueError("CudaComposite: source must be a non-empty string of CUDA C++")
        if not (theta_len == "m" or (isinstance(theta_len, (int, np.integer)) and not isinstance(theta_len, bool)
                                     and theta_len >= 0)):
            raise ValueError('CudaComposite: theta_len must be "m" or an int >= 0, got %r' % (theta_len,))
        self.source = source
        self.theta_len = theta_len if theta_len == "m" else int(theta_len)
        self._ids = {}

    def param_len(self, m):
        return m if self.theta_len == "m" else self.theta_len

    def composite_id(self, m):
        """The library's id of this composite for m outputs; compiles it on the first call for each m."""
        cid = self._ids.get(m)
        if cid is None:
            cid = _lib.register_composite(self.source, m, -1 if self.theta_len == "m" else self.theta_len)
            self._ids[m] = cid
        return cid

    def __repr__(self):
        return "CudaComposite(<%d chars of CUDA>, theta_len=%r)" % (len(self.source), self.theta_len)


def composite_id(composite, m):
    """Device id of a composite: the catalogued enum of a name, the registered id of a CudaComposite."""
    if isinstance(composite, CudaComposite):
        return composite.composite_id(m)
    return COMPOSITES[composite]


def _host_psi(name):
    """Closed-form E[U(theta, y)], y_j ~ N(mu_j, v_j), as (psi, dpsi/d(mu, v)) -- the pairs the reference's scripts pass
    as ExpectationUtility; the device enum of acq.cu (psi_acq_kernel) restates the same formulas."""
    if name == "sumsq_target":       # test_1a.py:100-113
        return (lambda th, mu, v: -np.sum(np.square((np.asarray(mu).T - th).T), axis=0) - np.sum(v, axis=0),
                lambda th, mu, v: -np.concatenate((2 * (np.squeeze(mu) - th), np.ones(len(np.squeeze(v))))))
    if name == "neg_sum_exp":        # test_2a.py:70-83
        return (lambda th, mu, v: -np.sum(np.exp(np.squeeze(mu) + 0.5 * np.squeeze(v))),
                lambda th, mu, v: -np.concatenate((np.exp(np.squeeze(mu) + 0.5 * np.squeeze(v)),
                                                   0.5 * np.exp(np.squeeze(mu) + 0.5 * np.squeeze(v)))))
    if name == "rosen_composite":    # test_5a.py:64-77
        def psi(a, mu, v):
            mu, v = np.squeeze(mu), np.squeeze(v)
            h = len(mu) // 2
            a = float(np.asarray(a).reshape(-1)[0])
            return -np.sum((a - mu[:h]) ** 2 + 100 * mu[h:2 * h] ** 2 + v[:h] + 100 * v[h:2 * h])

        def dpsi(a, mu, v):
            mu = np.squeeze(mu)
            m, h = len(mu), len(mu) // 2
            a = float(np.asarray(a).reshape(-1)[0])
            g = np.zeros(2 * m)
            g[:h] = 2 * (a - mu[:h])
            g[h:2 * h] = -200 * mu[h:2 * h]
            g[m:m + h] = -1.0
            g[m + h:m + 2 * h] = -100.0
            return g
        return psi, dpsi
    if name == "linear":             # cbo.py:126-168: E[theta . y] = theta . mu
        return (lambda th, mu, v: np.dot(th, np.squeeze(mu)),
                lambda th, mu, v: np.concatenate((np.atleast_1d(th), np.zeros(len(np.squeeze(mu))))))
    return None


class Utility(object):
    """utility.py:6-48 plus ``composite``: the device-side U(theta, y), a catalogued name or a CudaComposite."""

    def __init__(self, func=None, dfunc=None, parameter_dist=None, linear=False, composite=None):
        if composite is None:
            raise ValueError(
                "bocf_b200.Utility needs composite=<one of %s, or a CudaComposite>: Python callables cannot run inside "
                "the CUDA kernels (and there is no CPU fallback)." % sorted(COMPOSITES))
        self.composite = composite
        self.parameter_dist = parameter_dist
        self.linear = linear or composite == "linear"
        if isinstance(composite, CudaComposite):
            if func is None or dfunc is None:
                raise ValueError("Utility with a CudaComposite needs func and dfunc: the host side of the loop "
                                 "evaluates them, and the device code is checked against them")
            self.func, self.dfunc = func, dfunc
            self._device_checked = set()
            return
        if composite not in COMPOSITES:
            raise ValueError("unknown composite %r" % (composite,))
        hf, hdf = _host_funcs(composite)
        self.func = func if func is not None else hf
        self.dfunc = dfunc if dfunc is not None else hdf
        if func is not None or dfunc is not None:
            self._check_callables(hf, hdf)

    @property
    def theta_len(self):
        """Entries of one utility parameter: "m" (one per output) or a fixed count."""
        c = self.composite
        return c.theta_len if isinstance(c, CudaComposite) else THETA_DIM[c]

    def composite_id(self, m, device=None):
        """The library's id of the composite for a model with m outputs.  A CudaComposite is compiled for m on first
        use and its device U / dU/dy are then checked against func / dfunc on `device` (default: the current CUDA
        device) at 16 random (theta, y) points."""
        cid = composite_id(self.composite, m)
        if isinstance(self.composite, CudaComposite) and m not in self._device_checked:
            self._check_device(cid, m, device)
            self._device_checked.add(m)
        return cid

    def _check_device(self, cid, m, device, n=16):
        import torch
        rng = np.random.default_rng(0x5eed)        # private: the reference's global RNG stream must not move
        p = self.composite.param_len(m)
        th = np.ascontiguousarray(rng.standard_normal((n, p)))
        Y = rng.standard_normal((m, n))
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        lib = _lib.load_library()
        th_p = th.ctypes.data_as(ctypes.c_void_p) if p > 0 else None
        with torch.cuda.device(dev):
            Yd = torch.from_numpy(Y).to(dev)
            U = torch.empty((n, n), dtype=torch.float64, device=dev)
            G = torch.empty((n, m, n), dtype=torch.float64, device=dev)
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(lib.bocf_utility_eval(cid, m, ctypes.c_void_p(Yd.data_ptr()), n, th_p, n, p,
                                             ctypes.c_void_p(U.data_ptr()), st))
            _lib.check(lib.bocf_utility_grad_eval(cid, m, ctypes.c_void_p(Yd.data_ptr()), n, th_p, n, p,
                                                  ctypes.c_void_p(G.data_ptr()), st))
            U, G = U.cpu().numpy(), G.cpu().numpy()
        for k in range(n):
            u_ref = np.asarray(self.func(th[k], Y[:, k]), dtype=float).reshape(-1)
            g_ref = np.asarray(self.dfunc(th[k], Y[:, k]), dtype=float).reshape(-1)
            ok = (u_ref.size == 1 and g_ref.size == m and
                  np.allclose(U[k, k], u_ref[0], rtol=1e-9, atol=1e-12, equal_nan=True) and
                  np.allclose(G[k, :, k], g_ref, rtol=1e-9, atol=1e-12, equal_nan=True))
            if not ok:
                raise ValueError(
                    "Utility: the CudaComposite disagrees with func / dfunc at theta=%s, y=%s: device U=%r dU=%s, "
                    "host U=%s dU=%s" % (th[k], Y[:, k], U[k, k], G[k, :, k], u_ref, g_ref))

    def _check_callables(self, hf, hdf, m=4):
        """A user-supplied func / dfunc must be the catalogued composite: the device evaluates the enum, the loop's
        reporting path the callable -- two different utilities would silently optimise one and report the other."""
        rng = np.random.default_rng(0)
        y = rng.standard_normal(m)
        th = rng.standard_normal(m) if THETA_DIM[self.composite] == "m" else np.array([0.7])
        try:
            ok = np.allclose(np.asarray(self.func(th, y), dtype=float), np.asarray(hf(th, y), dtype=float), rtol=1e-9, atol=1e-12)
            if self.dfunc is not None:
                ok = ok and np.allclose(np.asarray(self.dfunc(th, y), dtype=float).reshape(-1),
                                        np.asarray(hdf(th, y), dtype=float).reshape(-1), rtol=1e-9, atol=1e-12)
        except Exception:            # callables written for one fixed m (test_5a.py) cannot be probed at m = 4
            return
        if not ok:
            raise ValueError("Utility: func / dfunc disagree with composite=%r (the CUDA kernels evaluate the composite)"
                             % (self.composite,))

    def evaluate_w_gradient(self, parameter, y):
        return self.eval_func(parameter, y), self.eval_gradient(parameter, y)

    def eval_func(self, parameter, y):
        return self.func(parameter, y)

    def eval_gradient(self, parameter, y):
        return self.dfunc(parameter, y)


class ParameterDistribution(object):
    """parameter_distribution.py:5-29 (discrete support + probabilities, or a continuous sampler)."""

    def __init__(self, continuous=False, support=None, prob_dist=None, sample_generator=None):
        if continuous is True and sample_generator is None:
            pass
        else:
            self.continuous = continuous
            self.support = support
            self.prob_dist = prob_dist
            self.sample_generator = sample_generator
        if support is not None and len(support) < 20:
            self.use_full_support = True
        else:
            self.use_full_support = False

    def sample(self, n_samples):
        if self.continuous:
            parameter_samples = self.sample_generator(n_samples)
        else:
            indices = np.random.choice(int(len(self.support)), size=n_samples, p=self.prob_dist)
            parameter_samples = self.support[indices, :]
        return parameter_samples
