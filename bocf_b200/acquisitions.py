"""Acquisition classes with the reference's plugin surface, backed by the CUDA library.

AcquisitionBase  GPyOpt/acquisitions/base.py:6-74
uEI_noiseless    uEI_noiseless.py:9-175   (EI-CF)
uPI              uPI.py                   (no gradient)
maEI / maPI      maEI.py / maPI.py        (analytic, linear scalarisation)
EI / PI          EI.py / PI.py            (single-output, single hyper-sample)

Same constructor arguments, method names, shapes and sign conventions; ``_compute_acq`` /
``_compute_acq_withGradients`` take numpy (N,d) and return numpy ((N,1), (N,d)), or take CUDA torch
tensors and return CUDA torch tensors.  The reference's pathos pool (uEI_noiseless.py:85-97) is gone:
all candidates of a call are evaluated by one fused device sweep.

Reference behaviours kept on purpose (SURVEY.md 8a quirks): f* is computed once per call with
whichever hyper-sample is currently selected and the model is left on the last hyper-sample (q2);
the gradient call draws ONE fresh theta when the parameter distribution is sampled (q4); the value
uses max(.,0) while the gradient indicator is a strict > (q10); uPI/maPI add 1e-6 to f* (q11).
One deviation: with ``fixed_hyps=True`` the reference averages 10 identical passes (q6); here the
identical passes are evaluated once.
"""
import ctypes
import threading

import numpy as np
import torch

from . import _lib
from .utility import theta_matrix


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _host(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(ctypes.c_void_p)


class AcquisitionBase(object):
    """GPyOpt/acquisitions/base.py:6-74."""
    analytical_gradient_prediction = False

    def __init__(self, model, space, optimizer, cost_withGradients=None):
        self.model = model
        self.space = space
        self.optimizer = optimizer
        self.analytical_gradient_acq = self.analytical_gradient_prediction and self.model.analytical_gradient_prediction
        self.cost_withGradients = cost_withGradients

    def acquisition_function(self, x):
        # base.py:33-44: the optimiser minimises, so the sign is flipped
        return self._negated(self._compute_acq, x)

    def acquisition_function_withGradients(self, x):
        # base.py:47-56
        return self._negated(self._compute_acq_withGradients, x)

    def _negated(self, fn, x):
        """-fn(x).  The flip is applied on the device, before the results leave it (`_run` honours `_sign`): negating a
        (1M, d) gradient on the host costs more than the whole D2H copy.  Results that did not come out of `_run` are
        negated here.  The pending flip is per THREAD (the batched multistart optimiser runs one scipy L-BFGS state
        machine per thread, optimization.py), and every call into the model handle is serialised by the model's lock."""
        tls = self._tls
        tls.sign, tls.applied = -1.0, False
        try:
            out = fn(x)
        finally:
            applied = tls.applied
            tls.sign, tls.applied = 1.0, False
        if applied:
            return out
        return tuple(-o for o in out) if isinstance(out, tuple) else -out

    @property
    def _tls(self):
        t = self.__dict__.get("_tls_obj")
        if t is None:
            t = self.__dict__.setdefault("_tls_obj", threading.local())
        return t

    @property
    def _sign(self):
        return getattr(self._tls, "sign", 1.0)

    def _mark_sign_applied(self):
        self._tls.applied = True

    def optimize(self, duplicate_manager=None, x_baseline=None):
        if not self.analytical_gradient_acq:
            out = self.optimizer.optimize(f=self.acquisition_function, duplicate_manager=duplicate_manager,
                                          x_baseline=x_baseline)
        else:
            out = self.optimizer.optimize(f=self.acquisition_function, f_df=self.acquisition_function_withGradients,
                                          duplicate_manager=duplicate_manager, x_baseline=x_baseline)
        return out

    def _compute_acq(self, x):
        raise NotImplementedError('')

    def _compute_acq_withGradients(self, x):
        raise NotImplementedError('')

    # ---- shared device plumbing -----------------------------------------------------------------------
    def _n_hyps_effective(self):
        H_loaded = self.model.n_hyper_samples_loaded()
        return 1 if (self.model.fixed_hyps or H_loaded == 1) else min(self.n_hyps_samples, H_loaded)

    HOST_ENTRY_MAX = 4096       # numpy inputs up to this long go through ONE C call (bocf_acq_eval_host)
    PIPELINE_MIN = 1 << 17      # numpy inputs at least this long are streamed through the device in slabs
    PIPELINE_SLABS = 4

    def _run(self, variant, X, theta, weight, fstar, grad, Zt=None, S=0, form=0):
        model = self.model
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        if not isinstance(X, torch.Tensor):
            Xn = np.atleast_2d(np.asarray(X, dtype=np.float64))
            if Xn.shape[0] >= self.PIPELINE_MIN:
                return self._run_pipelined(variant, np.ascontiguousarray(Xn), theta, weight, fstar, grad, Zt, S, form)
            if Xn.shape[0] <= self.HOST_ENTRY_MAX:
                return self._eval_host_small(variant, np.ascontiguousarray(Xn), theta, weight, fstar, grad, Zt, S, form)
        Xd, is_t = model._dev_in(X)
        acq, dacq = self._eval_device(variant, Xd, theta, weight, fstar, grad, Zt, S, form)
        acq = acq.reshape(-1, 1)
        if not is_t:
            acq = self._to_host(acq)
            dacq = None if dacq is None else self._to_host(dacq)
        return (acq, dacq) if grad else acq

    def _eval_host_small(self, variant, Xn, theta, weight, fstar, grad, Zt, S, form):
        """Small numpy batches (the L-BFGS rounds of the acquisition optimiser): one C call does the H2D copy, the sweep
        and the D2H copies with a single stream synchronisation (bocf_acq_eval_host), no torch tensors in between."""
        model = self.model
        N, d = Xn.shape
        L = theta.shape[0]
        th_h, th_p = _host(theta)
        w_h, w_p = _host(weight)
        f_h, f_p = _host(fstar)
        if w_h.size != L or f_h.ndim != 2 or f_h.shape[1] != L:
            raise ValueError("need one weight and one incumbent column per utility parameter: L=%d, %d weights, f* %s"
                             % (L, w_h.size, f_h.shape))
        acq = np.empty((N, 1))
        dacq = np.empty((N, d)) if grad else None
        cid = self.utility.composite_id(model.output_dim, model.device)
        with model._lock:
            # self-contained call (copies in, sweep, copies out, one synchronisation) on the handle's own stream: no
            # torch device / stream bookkeeping on this latency-bound path.  Everything it depends on (factor, digit
            # planes, base samples) was synchronised when it was produced.
            st = model._side_stream_ptr()
            _lib.check(model._lib.bocf_acq_eval_host(
                model._handle, _lib.VARIANTS[variant], cid,
                Xn.ctypes.data_as(ctypes.c_void_p), N, _ptr(Zt), S, th_p, L, theta.shape[1], w_p, f_p, f_h.shape[0], form,
                acq.ctypes.data_as(ctypes.c_void_p), None if dacq is None else dacq.ctypes.data_as(ctypes.c_void_p), st))
        if self._sign < 0:
            np.negative(acq, out=acq)
            if dacq is not None:
                np.negative(dacq, out=dacq)
        self._mark_sign_applied()
        return (acq, dacq) if grad else acq

    def _eval_device(self, variant, Xd, theta, weight, fstar, grad, Zt, S, form):
        """One bocf_acq_eval call on device-resident candidates; applies the pending sign flip on the device."""
        model = self.model
        N, d = Xd.shape
        L = theta.shape[0]
        th_h, th_p = _host(theta)
        w_h, w_p = _host(weight)
        f_h, f_p = _host(fstar)
        if w_h.size != L or f_h.ndim != 2 or f_h.shape[1] != L:
            raise ValueError("need one weight and one incumbent column per utility parameter: L=%d, %d weights, f* %s"
                             % (L, w_h.size, f_h.shape))
        H_use = f_h.shape[0]
        cid = self.utility.composite_id(model.output_dim, model.device)
        with model._lock, torch.cuda.device(model.device):
            acq = torch.empty((N,), dtype=torch.float64, device=model.device)
            dacq = torch.empty((N, d), dtype=torch.float64, device=model.device) if grad else None
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(model._lib.bocf_acq_eval(model._handle, _lib.VARIANTS[variant], cid, _ptr(Xd), N, _ptr(Zt), S,
                                                th_p, L, theta.shape[1], w_p, f_p, H_use, form, _ptr(acq), _ptr(dacq),
                                                st))
            if self._sign < 0:
                acq.neg_()
                if dacq is not None:
                    dacq.neg_()
        self._mark_sign_applied()
        return acq, dacq

    def _run_pipelined(self, variant, Xn, theta, weight, fstar, grad, Zt, S, form):
        """Host candidates in, host results out, in slabs: the H2D copy of slab k+1 and the D2H copy of slab k-1 run on a
        side stream while slab k is evaluated (candidates are independent, so slab results equal the one-shot ones)."""
        model = self.model
        dev = model.device
        N, d = Xn.shape
        step = -(-N // self.PIPELINE_SLABS)
        step = ((step + 127) // 128) * 128
        bounds = [(a, min(a + step, N)) for a in range(0, N, step)]
        Xh = torch.from_numpy(Xn)
        with torch.cuda.device(dev):
            main = torch.cuda.current_stream()
            if getattr(self, "_copy_stream", None) is None:
                self._copy_stream = torch.cuda.Stream(device=dev)
            side = self._copy_stream
            acq_h = torch.empty((N, 1), dtype=torch.float64, device="cpu", pin_memory=True)
            dacq_h = torch.empty((N, d), dtype=torch.float64, device="cpu", pin_memory=True) if grad else None
            side.wait_stream(main)
            slabs, ready = [], []
            with torch.cuda.stream(side):
                for a, b in bounds:
                    slabs.append(Xh[a:b].to(dev, non_blocking=True))
                    ev = torch.cuda.Event()
                    ev.record(side)
                    ready.append(ev)
            keep = []
            for (a, b), Xd, ev in zip(bounds, slabs, ready):
                main.wait_event(ev)
                acq, dacq = self._eval_device(variant, Xd, theta, weight, fstar, grad, Zt, S, form)
                done = torch.cuda.Event()
                done.record(main)
                with torch.cuda.stream(side):
                    side.wait_event(done)
                    acq_h[a:b, 0].copy_(acq, non_blocking=True)
                    if grad:
                        dacq_h[a:b].copy_(dacq, non_blocking=True)
                keep.append((Xd, acq, dacq))
            side.synchronize()
            main.wait_stream(side)
        del keep
        return (acq_h.numpy(), dacq_h.numpy()) if grad else acq_h.numpy()

    @staticmethod
    def _to_host(t):
        """Device -> numpy.  Large results are copied straight into a pinned host buffer (torch's caching host
        allocator recycles it) and returned as the numpy array that owns that buffer: one DMA, no pageable bounce."""
        if t.numel() < (1 << 16):
            return t.cpu().numpy()
        pin = torch.empty(t.shape, dtype=t.dtype, device="cpu", pin_memory=True)
        pin.copy_(t, non_blocking=True)
        torch.cuda.current_stream(t.device).synchronize()
        return pin.numpy()


class uEI_noiseless(AcquisitionBase):
    """EI-CF (uEI_noiseless.py:9-175)."""
    analytical_gradient_prediction = True
    _variant = "ei_cf"

    def __init__(self, model, space, optimizer=None, cost_withGradients=None, utility=None):
        self.optimizer = optimizer
        self.utility = utility
        super(uEI_noiseless, self).__init__(model, space, optimizer, cost_withGradients=cost_withGradients)
        self.n_attributes = self.model.output_dim
        self.W_samples = np.random.normal(size=(25, self.n_attributes))        # uEI_noiseless.py:31
        self.n_hyps_samples = min(10, self.model.number_of_hyps_samples())     # :32
        self.use_full_support = self.utility.parameter_dist.use_full_support   # :33
        if self.use_full_support:
            self.utility_params_samples = self.utility.parameter_dist.support
            self.utility_prob_dist = np.atleast_1d(self.utility.parameter_dist.prob_dist)
        else:
            self.utility_params_samples = self.utility.parameter_dist.sample(10)
        self._Zt_cache = (None, None)

    def _Zt(self):
        """Transposed base samples (m, S) on the device; refreshed when W_samples is replaced."""
        key, Zt = self._Zt_cache
        W = self.W_samples
        if key is None or key[0] is not W or key[1] != W.shape:
            W = np.ascontiguousarray(np.asarray(W, dtype=np.float64))
            Zt = torch.from_numpy(np.ascontiguousarray(W.T)).to(self.model.device)
            self._Zt_cache = ((self.W_samples, W.shape), Zt)
        return Zt

    def _fstar_current(self, theta):
        """max_n U(theta_l, mu(X_n)) under the CURRENTLY selected hyper-sample: (L,).

        The reference recomputes it in every call (uEI_noiseless.py:66,76,141,155); it depends only on the factorised
        model, the selected hyper-sample and theta, so it is cached on exactly those (the L-BFGS rounds of one
        acquisition optimisation call this ~100 times with the same model: a 1000-candidate posterior mean, a utility
        sweep and a device->host sync each)."""
        model = self.model
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        key = (id(model), model._version, model._current_h, self.utility.composite, theta.shape, theta.tobytes())
        cache = self.__dict__.setdefault("_fstar_cache", {})
        hit = cache.get(key)
        if hit is not None:
            return hit.copy()
        if len(cache) > 64:
            cache.clear()
        val = self._fstar_compute(theta)
        cache[key] = val
        return val.copy()

    def _fstar_compute(self, theta):
        model = self.model
        fX = model._posterior_mean_at_evaluated_points_dev()                  # (m, n) on device
        theta = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        L, p = theta.shape
        th_h, th_p = _host(theta)
        n = fX.shape[1]
        cid = self.utility.composite_id(model.output_dim, model.device)
        with torch.cuda.device(model.device):
            U = torch.empty((L, n), dtype=torch.float64, device=model.device)
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(model._lib.bocf_utility_eval(cid, model.output_dim, _ptr(fX.contiguous()), n, th_p, L, p, _ptr(U),
                                                    st))
            return U.max(dim=1).values.cpu().numpy()

    def _fstar(self, theta, per_hyper_sample=False):
        """Incumbent f*_l as an (H_use, L) table.

        per_hyper_sample=False: evaluated ONCE, before the h loop, with whichever hyper-sample is current
        (uEI_noiseless.py:66,76 and :141,155 -- the sequential value path and the gradient path, quirk q2).
        per_hyper_sample=True: re-evaluated inside every pass h, as the pool helper does
        (uEI_noiseless.py:99-109, the branch _compute_acq takes for more than one candidate)."""
        H_use = self._n_hyps_effective()
        if not per_hyper_sample:
            return np.tile(self._fstar_current(theta)[None, :], (H_use, 1))
        rows = []
        for h in range(H_use):
            self.model.set_hyperparameters(h)
            rows.append(self._fstar_current(theta))
        return np.stack(rows, axis=0)

    def _weights(self, L):
        if self.use_full_support:
            return np.asarray(self.utility_prob_dist, dtype=np.float64).reshape(-1)
        return np.full(L, 1.0 / L)

    def _finish(self):
        # the reference leaves the model on its last hyper-sample after the h loop
        self.model.set_hyperparameters(self._n_hyps_effective() - 1)

    def _compute_acq(self, X, parallel=True):
        # uEI_noiseless.py:40-61 (+ :63-83 / :85-116)
        theta = theta_matrix(self.utility, self.utility_params_samples)
        n_cand = X.shape[0] if hasattr(X, "shape") and len(X.shape) == 2 else len(np.atleast_2d(X))
        fstar = self._fstar(theta, per_hyper_sample=bool(parallel and n_cand > 1))     # :43-46
        Zt = self._Zt()
        out = self._run(self._variant, X, theta, self._weights(len(theta)), fstar, False, Zt, Zt.shape[1])
        self._finish()
        return out

    def _compute_acq_withGradients(self, X):
        # uEI_noiseless.py:118-170
        if self.use_full_support:
            theta = self.utility.parameter_dist.support
        else:
            theta = self.utility.parameter_dist.sample(1)                     # :126 (quirk q4)
        theta = theta_matrix(self.utility, theta)
        fstar = self._fstar(theta)
        Zt = self._Zt()
        out = self._run(self._variant, X, theta, self._weights(len(theta)), fstar, True, Zt, Zt.shape[1])
        self._finish()
        return out

    def update_Z_samples(self, n_samples=None):
        # uEI_noiseless.py:172-174
        self.W_samples = np.random.normal(size=self.W_samples.shape)


class uPI(uEI_noiseless):
    """uPI.py: MC probability of improvement of the composite; value only (uPI.py:19)."""
    analytical_gradient_prediction = False
    _variant = "pi_cf"

    def __init__(self, *a, **kw):
        super(uPI, self).__init__(*a, **kw)
        self.jitter = 1e-6                 # uPI.py:40; added to f* inside the kernel

    def _compute_acq_withGradients(self, X):
        raise NotImplementedError("uPI has no analytical gradient (uPI.py:19)")


class maEI(AcquisitionBase):
    """maEI.py: analytic EI of theta^T y, averaged over theta and hyper-samples."""
    analytical_gradient_prediction = True
    _variant = "ma_ei"
    _n_theta_value = 3                     # maEI.py:46
    _n_theta_grad = 3                      # maEI.py:65

    def __init__(self, model, space, optimizer=None, cost_withGradients=None, utility=None):
        self.optimizer = optimizer
        self.utility = utility
        super(maEI, self).__init__(model, space, optimizer, cost_withGradients=cost_withGradients)
        self.use_full_support = self.utility.parameter_dist.use_full_support
        self.n_hyps_samples = min(10, self.model.number_of_hyps_samples())

    def _theta(self, k):
        if self.use_full_support:
            self.utility_params_samples = self.utility.parameter_dist.support
            self.utility_param_dist = np.atleast_1d(self.utility.parameter_dist.prob_dist)
            w = np.asarray(self.utility_param_dist, dtype=np.float64).reshape(-1)
        else:
            self.utility_params_samples = self.utility.parameter_dist.sample(k)
            w = np.full(len(self.utility_params_samples), 1.0 / len(self.utility_params_samples))
        return theta_matrix(self.utility, self.utility_params_samples), w

    def _best(self, theta):
        """best_l = max_n theta_l^T mu_h(X_n), recomputed per hyper-sample (maEI.py:88,129-136): (H_use, L)."""
        model = self.model
        H_use = self._n_hyps_effective()
        th = torch.from_numpy(theta).to(model.device)
        best = np.empty((H_use, theta.shape[0]))
        for h in range(H_use):
            model.set_hyperparameters(h)
            mu = model._posterior_mean_at_evaluated_points_dev()             # (m, n)
            best[h] = (th @ mu).max(dim=1).values.cpu().numpy()
        return best

    def _compute_acq(self, X):
        theta, w = self._theta(self._n_theta_value)
        out = self._run(self._variant, X, theta, w, self._best(theta), False, form=0)
        return out

    def _compute_acq_withGradients(self, X):
        theta, w = self._theta(self._n_theta_grad)
        return self._run(self._variant, X, theta, w, self._best(theta), True, form=1)


class maPI(maEI):
    """maPI.py: analytic PI of theta^T y (jitter 1e-6 on the incumbent, maPI.py:35,151)."""
    _variant = "ma_pi"
    _n_theta_value = 10                    # maPI.py:45
    _n_theta_grad = 3                      # maPI.py:63

    def __init__(self, *a, **kw):
        super(maPI, self).__init__(*a, **kw)
        self.jitter = 1e-6


class EI(maEI):
    """EI.py: single-output twin of maEI; n_hyps_samples = 1 (EI.py:36)."""

    def __init__(self, *a, **kw):
        super(EI, self).__init__(*a, **kw)
        self.n_hyps_samples = 1


class PI(maPI):
    """PI.py: single-output twin of maPI; n_hyps_samples = 1."""

    def __init__(self, *a, **kw):
        super(PI, self).__init__(*a, **kw)
        self.n_hyps_samples = 1
