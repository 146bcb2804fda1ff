"""multi_outputGP with the reference's interface (multi_outputGP.py:9-348), backed by the CUDA library.

m independent single-output exact GPs.  The prediction methods keep the reference's names, argument
meaning and output shapes ((m,N) / (m,N,d) float64); numpy in -> numpy out, CUDA torch tensors in ->
CUDA torch tensors out (no host round trip).  All arithmetic runs in libbocf_b200 (fp64, sm_100a);
there is no CPU fallback.

Hyper-parameters: ``fixed_hyps=True`` keeps the kernels' initial values (gpmodel_fixed_hyps.py); explicit
hyper-samples are loaded with ``set_hyperparameter_samples``; otherwise ``updateModel`` does what
GPModel.updateModel does (gpmodel.py:102-128): ML-II, then an HMC chain whose sub-sampled states become
the ``n_samples`` hyper-sample instances -- all outputs in lockstep on the device likelihood (hmc.py).
"""
import ctypes
import threading

import numpy as np
import torch

from . import _lib
from . import kern as _kern
from .utility import composite_id


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class multi_outputGP(object):
    analytical_gradient_prediction = True

    def __init__(self, output_dim, kernel=None, noise_var=None, exact_feval=None, n_samples=10, ARD=None,
                 fixed_hyps=False, device=None, precision=None, n_burnin=100, subsample_interval=10, step_size=1e-1,
                 leapfrog_steps=20, max_iters=200, hyper_inference=None):
        self.output_dim = int(output_dim)
        self.kernel = [None] * output_dim if kernel is None else list(kernel)
        self.noise_var = [None] * output_dim if noise_var is None else list(noise_var)
        self.exact_feval = [False] * output_dim if exact_feval is None else list(exact_feval)
        self.n_samples = n_samples
        self.ARD = [True] * output_dim if ARD is None else list(ARD)
        self.fixed_hyps = fixed_hyps
        if device is None:
            device = "cuda:%d" % torch.cuda.current_device() if torch.cuda.is_available() else "cuda:0"
        self.device = torch.device(device)
        self._lib = _lib.load_library()
        # arithmetic of the two candidate-side contractions: None (library default / BOCF_PRECISION), "fp64",
        # "auto", or "split3".."split6" (tcgen05 int8 digit planes, include/bocf_b200.h: enum bocf_precision)
        self.precision = precision
        # the C handle is stream-ordered and NOT thread-safe (shared scratch, selected hyper-sample): every call into it
        # takes this lock (the batched multistart optimiser runs one L-BFGS state machine per thread)
        self._lock = threading.RLock()
        self._version = 0           # bumped whenever the factorised state changes (data, hyper-samples, append): cache key
        # GPModel's sampler settings (gpmodel.py:31: n_burnin=100, subsample_interval=10, step_size=1e-1, leapfrog_steps=20)
        self.n_burnin, self.subsample_interval = n_burnin, subsample_interval
        self.step_size, self.leapfrog_steps, self.max_iters = step_size, leapfrog_steps, max_iters
        # "hmc": updateModel fits and samples the hyper-parameters like GPModel.updateModel; "none": keep the initial values
        self.hyper_inference = ("none" if fixed_hyps else "hmc") if hyper_inference is None else hyper_inference
        if self.hyper_inference not in ("hmc", "none"):
            raise ValueError("hyper_inference must be 'hmc' or 'none'")
        self._inference = None
        self.incremental_updates = True     # one-point updateModel calls with unchanged hypers use the O(n^2) append
        self.last_update = None
        self._handle = None
        self._handle_sig = None
        self._explicit_hyp = False
        self._hyp = None            # (kind, variance (H,m), lengthscale (H,m,d), noise (H,m))
        self._current_h = 0
        self.X = None
        self.Y = None
        self.input_dim = None
        self.jitter_added = None

    # ---- hyper-parameters ---------------------------------------------------------------------------
    def set_hyperparameter_samples(self, variance, lengthscale, noise, kind=None):
        """Load H hyper-samples: variance (H,m), lengthscale (H,m,d), noise (H,m).

        Stands in for the per-sample GPRegression instances GPModel.updateModel fills from HMC
        (gpmodel.py:121-126).  ``kind`` in {'se','rbf','matern52','matern32'}, or a sequence with one such name per
        output.
        """
        variance = np.ascontiguousarray(variance, dtype=np.float64)
        lengthscale = np.ascontiguousarray(lengthscale, dtype=np.float64)
        noise = np.ascontiguousarray(noise, dtype=np.float64)
        H, m = variance.shape
        assert m == self.output_dim and lengthscale.shape[:2] == (H, m) and noise.shape == (H, m)
        if kind is None:
            kind = self._kernel_kind()
        elif not isinstance(kind, str):
            kind = tuple(kind)
            assert len(kind) == m, "one kernel family per output"
            if len(set(kind)) == 1:
                kind = kind[0]
        self._hyp = (kind, variance, lengthscale, noise)
        self._explicit_hyp = True
        if self.X is not None:
            self._upload_and_factorize()

    def _kernel_kind(self):
        """Kernel family of the model: one name when every output uses the same family, else a tuple with one name per
        output (multi_outputGP.py:23,38-44 builds output j from kernel[j]; an output without a kernel gets the
        reference's default SE, gpmodel.py:57-58)."""
        kinds = tuple("se" if k is None else k.kind for k in self.kernel)
        return kinds[0] if len(set(kinds)) == 1 else kinds

    def _default_hypers(self, d, Y_all):
        """Initial hyper-parameters of the reference's model constructors, as one hyper-sample (H = 1)."""
        m = self.output_dim
        var = np.empty((1, m))
        ls = np.empty((1, m, d))
        noise = np.empty((1, m))
        for j in range(m):
            k = self.kernel[j]
            if k is None:
                if self.fixed_hyps:     # gpmodel_fixed_hyps.py:49-50
                    k = _kern.SE(d, variance=2., lengthscale=0.3)
                else:                   # gpmodel.py:57-58
                    k = _kern.SE(d, variance=1., ARD=self.ARD[j])
            var[0, j] = k.variance[0]
            ls[0, j, :] = k.lengthscale_vector()
            if self.fixed_hyps:         # gpmodel_fixed_hyps.py:56
                noise[0, j] = 1e-10 if self.noise_var[j] is None else self.noise_var[j]
            elif self.exact_feval[j]:   # gpmodel.py:72-73
                noise[0, j] = 1e-6
            else:                       # gpmodel.py:64
                noise[0, j] = np.var(Y_all[j]) * 0.01 if self.noise_var[j] is None else self.noise_var[j]
        return (self._kernel_kind(), var, ls, noise)

    # ---- data -----------------------------------------------------------------------------------------
    def updateModel(self, X_all, Y_all):
        """multi_outputGP.py:97-102.  X_all (n,d); Y_all list of m arrays (n,1)."""
        X = np.ascontiguousarray(X_all, dtype=np.float64)
        Y = np.ascontiguousarray(np.stack([np.asarray(y, dtype=np.float64).reshape(-1) for y in Y_all], axis=0))
        assert Y.shape == (self.output_dim, X.shape[0])
        old_X, old_Y, old_hyp = self.X, self.Y, self._hyp
        self.X = X
        self.Y = Y
        self.input_dim = X.shape[1]
        if not self._explicit_hyp and not self.fixed_hyps and self.hyper_inference == "hmc":
            self._infer_hyperparameters(Y_all)
            return
        if self._hyp is None or not getattr(self, "_explicit_hyp", False):
            self._hyp = self._default_hypers(self.input_dim, Y_all)
        if self._try_append(old_X, old_Y, old_hyp):
            return
        self._upload_and_factorize()

    # ---- hyper-parameter inference (gpmodel.py:102-128, all outputs in lockstep) --------------------------------------
    def _infer_hyperparameters(self, Y_all):
        from . import hmc as _hmc
        kind = self._kernel_kind()
        d, m = self.input_dim, self.output_dim
        if self._inference is None:
            kernels, noises, fixes, inst = [], [], [], []
            for j in range(m):
                k = self.kernel[j]
                if k is None:                               # gpmodel.py:57-58
                    k = _kern.SE(d, variance=1., ARD=self.ARD[j])
                kernels.append((float(k.variance[0]), np.array(k.lengthscale, dtype=float)))
                if self.exact_feval[j]:                     # gpmodel.py:70-71
                    noises.append(1e-6); fixes.append(True); inst.append(1e-6)
                elif self.noise_var[j] is not None:         # gpmodel.py:72-73
                    noises.append(float(self.noise_var[j])); fixes.append(True); inst.append(float(self.noise_var[j]))
                else:                                       # gpmodel.py:64,74-75
                    nv = float(np.var(Y_all[j])) * 0.01
                    noises.append(nv); fixes.append(False); inst.append(nv)

            def evaluate(variance, lengthscale, noise):
                self._hyp = (kind, np.ascontiguousarray(variance[None, :]), np.ascontiguousarray(lengthscale[None, :, :]),
                             np.ascontiguousarray(noise[None, :]))
                self._upload_and_factorize(upload_data=self._fit_needs_data)
                self._fit_needs_data = False
                lml, gv, gl, gn = self.log_likelihood_and_gradients()
                return lml[0], gv[0], gl[0], gn[0]

            self._inference = _hmc.HyperInference(evaluate, d, kernels, noises, fixes, inst, n_samples=self.n_samples,
                                                  n_burnin=self.n_burnin, subsample_interval=self.subsample_interval,
                                                  step_size=self.step_size, leapfrog_steps=self.leapfrog_steps,
                                                  max_iters=self.max_iters)
        self._fit_needs_data = True
        variance, lengthscale, noise = self._inference.update()
        self._hyp = (kind, variance, lengthscale, noise)
        self._upload_and_factorize()
        self.last_update = "hmc"

    def get_hyperparameters_samples(self):
        """(variance (H,m), lengthscale (H,m,d), noise (H,m)) currently loaded (None before the first updateModel)."""
        return None if self._hyp is None else tuple(np.array(a) for a in self._hyp[1:])

    def _try_append(self, old_X, old_Y, old_hyp):
        """One new observation and unchanged hyper-parameters: O(n^2) bordered update on the device
        (bocf_model_append_point) instead of a refactorisation.  Falls back (returns False) whenever it does not apply."""
        if (not self.incremental_updates or self._handle is None or old_X is None or old_hyp is None or
                self.X.shape[0] != old_X.shape[0] + 1 or self.X.shape[1] != old_X.shape[1] or
                not np.array_equal(self.X[:-1], old_X) or not np.array_equal(self.Y[:, :-1], old_Y)):
            return False
        if old_hyp[0] != self._hyp[0] or any(not np.array_equal(a, b) for a, b in zip(old_hyp[1:], self._hyp[1:])):
            return False
        with torch.cuda.device(self.device):
            xn = torch.from_numpy(np.ascontiguousarray(self.X[-1])).to(self.device)
            yn = torch.from_numpy(np.ascontiguousarray(self.Y[:, -1])).to(self.device)
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            self._version += 1
            rc = self._lib.bocf_model_append_point(self._handle, _ptr(xn), _ptr(yn), st)
            if rc == -5:                       # BOCF_ERR_UNSUPPORTED: buffers full / pivot not positive
                return False
            _lib.check(rc)
            self._X_dev = torch.from_numpy(self.X).to(self.device)
        self._current_h = 0
        self.last_update = "append"
        return True

    def _upload_and_factorize(self, upload_data=True):
        self._version += 1
        kind, variance, lengthscale, noise = self._hyp
        lib = self._lib
        d = self.input_dim
        if lengthscale.shape[2] != d:
            assert lengthscale.shape[2] == 1
            lengthscale = np.ascontiguousarray(np.broadcast_to(lengthscale, lengthscale.shape[:2] + (d,)))
        if self._handle is None or self._handle_sig != (kind, d):
            self._destroy()
            h = ctypes.c_void_p()
            kinds = [kind] * self.output_dim if isinstance(kind, str) else list(kind)
            _lib.check(lib.bocf_model_create(ctypes.byref(h), self.output_dim, d, _lib.KERNELS[kinds[0]],
                                             self.device.index or 0))
            self._handle = h
            self._handle_sig = (kind, d)
            if len(set(kinds)) > 1:             # a kernel family per output
                codes = (ctypes.c_int * self.output_dim)(*[_lib.KERNELS[k] for k in kinds])
                _lib.check(lib.bocf_model_set_kernels(self._handle, codes, self.output_dim))
            upload_data = True
            if self.precision is not None:
                mode, slices = _lib.parse_precision(self.precision)
                _lib.check(lib.bocf_model_set_precision(self._handle, mode, slices, None))
        with torch.cuda.device(self.device):
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            if upload_data or getattr(self, "_X_dev", None) is None:
                Xd = torch.from_numpy(self.X).to(self.device)
                Yd = torch.from_numpy(self.Y).to(self.device)
                _lib.check(lib.bocf_model_set_data(self._handle, self.X.shape[0], _ptr(Xd), _ptr(Yd), st))
                self._X_dev = Xd
            _lib.check(lib.bocf_model_set_hypers(self._handle, variance.shape[0],
                                                 variance.ctypes.data_as(ctypes.c_void_p),
                                                 lengthscale.ctypes.data_as(ctypes.c_void_p),
                                                 noise.ctypes.data_as(ctypes.c_void_p)))
            jit = np.zeros(variance.shape, dtype=np.float64)
            _lib.check(lib.bocf_model_factorize(self._handle, jit.ctypes.data_as(ctypes.c_void_p), st))
            self.jitter_added = jit
        self._current_h = 0
        self.last_update = "factorize"

    def set_precision(self, precision):
        """Switch the contraction arithmetic ("fp64" | "auto" | "split3".."split6"); rebuilds the digit planes."""
        self.precision = precision
        if self._handle is not None:
            mode, slices = _lib.parse_precision(precision)
            with torch.cuda.device(self.device):
                st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
                _lib.check(self._lib.bocf_model_set_precision(self._handle, mode, slices, st))

    def active_slices(self):
        """Digit planes the tensor-core contraction currently uses (0 = fp64 DMMA)."""
        return int(self._lib.bocf_model_active_slices(self._handle)) if self._handle is not None else 0

    def _side_stream_ptr(self):
        """A non-blocking stream owned by this model for self-contained host-entry calls (created once)."""
        st = getattr(self, "_side_stream", None)
        if st is None:
            with torch.cuda.device(self.device):
                st = self._side_stream = torch.cuda.Stream(device=self.device)
            self._side_stream_c = ctypes.c_void_p(st.cuda_stream)
        return self._side_stream_c

    def chunk_candidates(self, N, grad=True):
        """Candidates per internal chunk of a call with N candidates (results never depend on it)."""
        return int(self._lib.bocf_model_chunk_candidates(self._handle, int(N), 1 if grad else 0))

    def active_scheme(self):
        """(scheme of the variance contraction, scheme of the variance-gradient contraction), a scheme being
        100 SA + 10 SB + LMIN (include/bocf_b200.h); (0, 0) = fp64 DMMA."""
        code = int(self._lib.bocf_model_active_scheme(self._handle)) if self._handle is not None else 0
        return (code // 1000, code % 1000) if code > 0 else (0, 0)

    def _destroy(self):
        if getattr(self, "_handle", None) is not None:
            self._lib.bocf_model_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._destroy()
        except Exception:
            pass

    # ---- bookkeeping (multi_outputGP.py:109-135) ----------------------------------------------------
    def number_of_hyps_samples(self):
        return self.n_samples

    def n_hyper_samples_loaded(self):
        return 1 if self._hyp is None else int(self._hyp[1].shape[0])

    def set_hyperparameters(self, n):
        # GPModel.set_hyperparameters selects instance n (gpmodel.py:136-137);
        # GPModelFixedHyps.set_hyperparameters is a no-op (gpmodel_fixed_hyps.py:76-77)
        H = self.n_hyper_samples_loaded()
        self._current_h = 0 if (self.fixed_hyps or H == 1) else int(n)
        if self._current_h >= H:
            raise IndexError("hyper-sample %d not loaded (H = %d)" % (n, H))

    def get_evaluated_points(self):
        return np.copy(self.X)

    # ---- prediction ---------------------------------------------------------------------------------
    def _dev_in(self, X):
        if isinstance(X, torch.Tensor):
            Xd = X.to(device=self.device, dtype=torch.float64)
            if Xd.dim() == 1:
                Xd = Xd[None, :]
            return Xd.contiguous(), True
        X = np.atleast_2d(np.asarray(X, dtype=np.float64))
        return torch.from_numpy(np.ascontiguousarray(X)).to(self.device), False

    def _posterior(self, X, want_mean=True, want_var=False, want_dmean=False, want_dvar=False, noiseless=False, clip=True):
        if self._handle is None:
            raise RuntimeError("model has no data: call updateModel first")
        Xd, is_t = self._dev_in(X)
        N, d = Xd.shape
        assert d == self.input_dim
        m = self.output_dim
        with self._lock, torch.cuda.device(self.device):
            mean = torch.empty((m, N), dtype=torch.float64, device=self.device)
            var = torch.empty((m, N), dtype=torch.float64, device=self.device) if want_var else None
            dmean = torch.empty((m, N, d), dtype=torch.float64, device=self.device) if want_dmean else None
            dvar = torch.empty((m, N, d), dtype=torch.float64, device=self.device) if want_dvar else None
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(self._lib.bocf_posterior(self._handle, self._current_h, _ptr(Xd), N,
                                                (1 if clip else 2) if noiseless else 0,
                                                _ptr(mean), _ptr(var), _ptr(dmean), _ptr(dvar), st))
        outs = (mean if want_mean else None, var, dmean, dvar)
        if is_t:
            return outs
        return tuple(None if o is None else o.cpu().numpy() for o in outs)

    def expected_utility(self, X, composite, parameter, n_hyps, Z=None, grad=False):
        """sum over the first n_hyps hyper-samples of the expected composite utility at X under the NOISELESS posterior,
        NOT normalised -- the objective cbo._current_marginal_argmax maximises (cbo.py:121-235).  `composite` is a
        catalogued name or a CudaComposite (MC branch only: it has no closed form):
          Z is None : closed form psi(theta, mu, var) (cbo.py:170-198; LINEAR = the posterior-mean branch :126-168)
          Z (S, m)  : sum_s U(theta, mu + sqrt(var) Z_s) with the pathwise gradient (cbo.py:203-231).
        Returns (value (N,), gradient (N, d) or None) as numpy (CUDA tensors for tensor input)."""
        Xd, is_t = self._dev_in(X)
        N, d = Xd.shape
        theta = np.ascontiguousarray(np.asarray(parameter, dtype=np.float64).reshape(1, -1))
        ones = np.ones(1)
        zeros = np.zeros((int(n_hyps), 1))
        variant = "psi" if Z is None else "mean_utility"
        cid = composite_id(composite, self.output_dim)
        with self._lock, torch.cuda.device(self.device):
            Zt, S = None, 0
            if Z is not None:
                Z = np.ascontiguousarray(np.asarray(Z, dtype=np.float64))
                Zt = torch.from_numpy(np.ascontiguousarray(Z.T)).to(self.device)
                S = Z.shape[0]
            val = torch.empty((N,), dtype=torch.float64, device=self.device)
            g = torch.empty((N, d), dtype=torch.float64, device=self.device) if grad else None
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(self._lib.bocf_acq_eval(self._handle, _lib.VARIANTS[variant], cid, _ptr(Xd), N,
                                               _ptr(Zt), S, theta.ctypes.data_as(ctypes.c_void_p), 1, theta.shape[1],
                                               ones.ctypes.data_as(ctypes.c_void_p), zeros.ctypes.data_as(ctypes.c_void_p),
                                               int(n_hyps), 0, _ptr(val), _ptr(g), st))
            if is_t:
                return val, g
            return val.cpu().numpy(), (None if g is None else g.cpu().numpy())

    # ---- knowledge-gradient helpers (multi_outputGP.py:203-281,309-331 -> GPModel -> GPy/core/gp.py:493-627) --------
    def _cov_point(self, X, x2, grad=False):
        """(cov (m,N), dcov (m,N,d) or None): posterior covariance of the latent functions between the rows of X and the
        single point x2 under the current hyper-sample (bocf_posterior_cov_point)."""
        Xd, is_t = self._dev_in(X)
        N, d = Xd.shape
        x2d, _ = self._dev_in(np.asarray(x2, dtype=np.float64).reshape(1, -1) if not isinstance(x2, torch.Tensor) else x2.reshape(1, -1))
        m = self.output_dim
        with self._lock, torch.cuda.device(self.device):
            cov = torch.empty((m, N), dtype=torch.float64, device=self.device)
            dcov = torch.empty((m, N, d), dtype=torch.float64, device=self.device) if grad else None
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(self._lib.bocf_posterior_cov_point(self._handle, self._current_h, _ptr(Xd), N, _ptr(x2d), _ptr(cov),
                                                          _ptr(dcov), st))
        if is_t:
            return cov, dcov
        return cov.cpu().numpy(), (None if dcov is None else dcov.cpu().numpy())

    def posterior_covariance_between_points(self, X1, X2):
        """multi_outputGP.py:257-266 -> gp.py:577-585: (m, N1, N2); one device sweep per column of X2."""
        X2 = np.atleast_2d(np.asarray(X2, dtype=np.float64))
        return np.stack([self._cov_point(X1, x2)[0] for x2 in X2], axis=2)

    def partial_precomputation_for_covariance(self, X):
        """multi_outputGP.py:203-210 -> gp.py:493-501.  The reference caches W^-1 K(X_train, X); here the per-column
        vectors beta = W^-1 k(X_train, x2) are rebuilt inside the device call (two matrix-vector products on the
        resident factor), so this only records the points."""
        self._pp_cov_X = np.atleast_2d(np.asarray(X, dtype=np.float64)).copy()

    def posterior_covariance_between_points_partially_precomputed(self, X1, X2):
        """multi_outputGP.py:269-281 -> gp.py:588-599 (X2 must be the points of partial_precomputation_for_covariance)."""
        return self.posterior_covariance_between_points(X1, X2)

    def posterior_covariance_gradient(self, X, x2):
        """multi_outputGP.py:309-318 -> gp.py:601-609: d cov(X_i, x2) / d X_i, (m, N, d), x2 a single point."""
        return self._cov_point(X, np.asarray(x2, dtype=np.float64).reshape(-1), grad=True)[1]

    def partial_precomputation_for_covariance_gradient(self, x):
        """multi_outputGP.py:213-220 -> gp.py:504-512 (see partial_precomputation_for_covariance)."""
        self._pp_dcov_x = np.asarray(x, dtype=np.float64).reshape(-1).copy()

    def posterior_covariance_gradient_partially_precomputed(self, X, x2):
        """multi_outputGP.py:321-330 -> gp.py:612-627."""
        return self.posterior_covariance_gradient(X, x2)

    def partial_precomputation_for_variance_conditioned_on_next_point(self, next_point):
        """multi_outputGP.py:223-230 -> gp.py:515-530.  The reference refactorises K(X u {x_next}) + (noise + 1e-8) I; the
        same conditional variance follows from the resident factor by the rank-one Schur complement
            var(x | x_next) = var_nl(x) - cov(x, x_next)^2 / (var_nl(x_next) + noise + 1e-8),
        so only x_next and its own noiseless variance are kept."""
        xn = np.asarray(next_point, dtype=np.float64).reshape(1, -1)
        self._next_point = xn.copy()
        self._next_h = self._current_h
        _, v, _, _ = self._posterior(xn, want_var=True, noiseless=True, clip=False)
        noise = self._noise_of_current()                                      # (m,)
        self._next_s = v[:, 0] + noise + 1e-8                                 # Schur complement pivot per output

    def _noise_of_current(self):
        return np.asarray(self._hyp[3][self._current_h], dtype=np.float64)

    def posterior_variance_conditioned_on_next_point(self, X):
        """multi_outputGP.py:233-242 -> gp.py:533-544: (m, N); noiseless, NOT clipped (the reference does not clip here)."""
        cov, _ = self._cov_point(X, self._next_point[0])
        _, v, _, _ = self._posterior(X, want_var=True, noiseless=True, clip=False)
        return v - cov ** 2 / self._next_s[:, None]

    def posterior_variance_gradient_conditioned_on_next_point(self, X):
        """multi_outputGP.py:245-254 -> gp.py:547-575: (m, N, d)."""
        cov, dcov = self._cov_point(X, self._next_point[0], grad=True)
        dv = self._posterior(X, want_dvar=True)[3]
        return dv - (2.0 * cov / self._next_s[:, None])[:, :, None] * dcov

    def predict(self, X, full_cov=False):
        """multi_outputGP.py:138-149: (mean (m,N), variance incl. noise, clipped at 1e-10 (gpmodel.py:147))."""
        mean, var, _, _ = self._posterior(X, want_var=True)
        return mean, var

    def predict_noiseless(self, X, full_cov=False):
        mean, var, _, _ = self._posterior(X, want_var=True, noiseless=True)
        return mean, var

    def posterior_mean(self, X):
        return self._posterior(X)[0]

    def posterior_mean_at_evaluated_points(self):
        """multi_outputGP.py:176-180; stays on the device when called by the acquisitions."""
        return self._posterior(self.X)[0]

    def _posterior_mean_at_evaluated_points_dev(self):
        return self._posterior(self._X_dev)[0]

    def posterior_variance(self, X):
        return self._posterior(X, want_var=True)[1]

    def posterior_variance_noiseless(self, X):
        return self._posterior(X, want_var=True, noiseless=True)[1]

    def posterior_mean_gradient(self, X):
        return self._posterior(X, want_dmean=True)[2]

    def posterior_variance_gradient(self, X):
        return self._posterior(X, want_dvar=True)[3]

    # ---- marginal likelihood (SURVEY.md 8f rank 2) ---------------------------------------------------
    def log_likelihood_and_gradients(self):
        """log p(y) of every (hyper-sample, output) GP and its gradient w.r.t. variance, lengthscales and noise.

        Returns (lml (H,m), g_variance (H,m), g_lengthscale (H,m,d), g_noise (H,m)): what GP.log_likelihood() and the
        .gradient attributes hold after GP.parameters_changed (gp.py:247-266) for each of the reference's model
        instances.  One fused device pass (bocf_model_log_likelihood)."""
        if self._handle is None:
            raise RuntimeError("model has no data: call updateModel first")
        H, m, d = self.n_hyper_samples_loaded(), self.output_dim, self.input_dim
        lml = np.empty((H, m))
        gv = np.empty((H, m))
        gl = np.empty((H, m, d))
        gn = np.empty((H, m))
        with torch.cuda.device(self.device):
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(self._lib.bocf_model_log_likelihood(
                self._handle, lml.ctypes.data_as(ctypes.c_void_p), gv.ctypes.data_as(ctypes.c_void_p),
                gl.ctypes.data_as(ctypes.c_void_p), gn.ctypes.data_as(ctypes.c_void_p), st))
        return lml, gv, gl, gn

    def log_likelihood(self):
        return self.log_likelihood_and_gradients()[0]

    def fit_hyperparameters(self, max_iters=200, fit_noise=True, bounds=(1e-6, 1e6), verbose=False):
        """ML-II: maximise sum_j log p(y_j) over (variance, lengthscales[, noise]) of every output, all outputs in ONE
        L-BFGS-B run whose objective and gradient are a single device pass per iteration (Gram, Cholesky, L^-1, alpha,
        likelihood, gradients for all m outputs at once).  Optimises in log space (the positivity constraint of the
        reference's Logexp transform, gpmodel.py:84-100); keeps H = 1.  This is the deterministic part of
        GPModel.updateModel (gpmodel.py:117: model.optimize(max_iters=200)); the HMC sampling around it is out of scope.
        Returns the final (H = 1) log likelihoods (m,)."""
        import scipy.optimize
        if self.X is None:
            raise RuntimeError("model has no data: call updateModel first")
        kind, variance, lengthscale, noise = self._hyp
        m, d = self.output_dim, self.input_dim
        if lengthscale.shape[2] != d:
            lengthscale = np.ascontiguousarray(np.broadcast_to(lengthscale, lengthscale.shape[:2] + (d,)))
        v0, l0, n0 = variance[:1].copy(), lengthscale[:1].copy(), np.maximum(noise[:1].copy(), bounds[0])
        npar = (d + 2) if fit_noise else (d + 1)

        def unpack(theta):
            th = np.exp(theta.reshape(m, npar))
            var = th[:, 0][None, :]
            ls = th[:, 1:1 + d][None, :, :]
            nz = th[:, 1 + d][None, :] if fit_noise else n0
            return np.ascontiguousarray(var), np.ascontiguousarray(ls), np.ascontiguousarray(nz)

        def f_df(theta):
            var, ls, nz = unpack(theta)
            self._hyp = (kind, var, ls, nz)
            self._explicit_hyp = True
            try:
                self._upload_and_factorize()
            except _lib.NotPositiveDefiniteError:
                return 1e25, np.zeros_like(theta)
            lml, gv, gl, gn = self.log_likelihood_and_gradients()
            g = np.zeros((m, npar))
            g[:, 0] = gv[0] * var[0]                       # d/d log(theta) = theta * d/d theta
            g[:, 1:1 + d] = gl[0] * ls[0]
            if fit_noise:
                g[:, 1 + d] = gn[0] * nz[0]
            if verbose:
                print("fit_hyperparameters: log p(y) = %.6f" % lml.sum())
            return -float(lml.sum()), -g.reshape(-1)

        cols = [np.log(v0[0])[:, None], np.log(l0[0])]
        if fit_noise:
            cols.append(np.log(n0[0])[:, None])
        theta0 = np.concatenate(cols, axis=1).reshape(-1)
        lo, hi = np.log(bounds[0]), np.log(bounds[1])
        res = scipy.optimize.fmin_l_bfgs_b(f_df, theta0, bounds=[(lo, hi)] * theta0.size, maxiter=max_iters)
        f_df(res[0])                                       # leave the model factorised at the optimum
        return self.log_likelihood()[0]

    # ---- inspection (tests) ---------------------------------------------------------------------------
    def get_factor(self, h, j):
        """(L, Linv, alpha) of output j under hyper-sample h as numpy arrays."""
        n = self.X.shape[0]
        with torch.cuda.device(self.device):
            L = torch.empty((n, n), dtype=torch.float64, device=self.device)
            Li = torch.empty((n, n), dtype=torch.float64, device=self.device)
            al = torch.empty((n,), dtype=torch.float64, device=self.device)
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            _lib.check(self._lib.bocf_model_get_factor(self._handle, h, j, _ptr(L), _ptr(Li), _ptr(al), st))
        return L.cpu().numpy(), Li.cpu().numpy(), al.cpu().numpy()
