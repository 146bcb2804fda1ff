"""Composite Bayesian-optimisation loop with the reference's interface (cbo.py:19-546), for Python 3.

Host plumbing only: model update -> acquisition optimisation -> objective evaluation -> "current optimal value"
bookkeeping.  Every call into the model / acquisition lands in the CUDA path.  Restated without time.clock(),
np.asscalar, pathos and the plotting services; MultiObjective (multi_objective.py:12-82) and ExpectationUtility
(expectation_utility.py:3-9) are included because the loop needs them.
"""
import time

import numpy as np

from .optimization import GeneralOptimizer, ContextManager


class InvalidConfigError(Exception):
    pass


class ExpectationUtility(object):
    # expectation_utility.py:3-9
    def __init__(self, func, gradient):
        self.func = func
        self.gradient = gradient


class MultiObjective(object):
    """multi_objective.py:12-82 with as_list=False semantics (func(X) -> (m, N)) or a list of m callables."""

    def __init__(self, func, noise_var=None, objective_name=None, as_list=True, output_dim=None):
        self.func = func
        self.as_list = as_list
        self.output_dim = len(func) if as_list else output_dim
        self.noise_var = noise_var
        self.objective_name = ['no_name'] * self.output_dim if objective_name is None else objective_name

    def evaluate(self, X):
        f_eval = [None] * self.output_dim
        cost_eval = 0
        if self.as_list:
            for j in range(self.output_dim):
                f_eval[j] = np.reshape(self.func[j](X), (X.shape[0], 1))
        else:
            fX = self.func(X)
            for j in range(self.output_dim):
                f_eval[j] = np.reshape(fX[j, :], (X.shape[0], 1))
        return f_eval, cost_eval

    def evaluate_w_noise(self, X):
        f_noisy_eval, cost_eval = self.evaluate(X)
        if self.noise_var is not None:
            for j in range(self.output_dim):
                f_noisy_eval[j] += np.random.normal(scale=np.sqrt(self.noise_var[j]))
        return f_noisy_eval, cost_eval


class CBO(object):
    """cbo.py:19-546 (run_optimization, compute_next_evaluations, _current_max_value, _current_marginal_argmax)."""

    def __init__(self, model, space, objective, acquisition, evaluator, X_init, Y_init=None, cost=None,
                 normalize_Y=False, model_update_interval=1, expectation_utility=None):
        self.model = model
        self.space = space
        self.objective = objective
        self.acquisition = acquisition
        self.utility = acquisition.utility
        self.expectation_utility = expectation_utility
        self.evaluator = evaluator
        self.X = X_init
        self.Y = Y_init
        self.normalize_Y = normalize_Y
        self.model_update_interval = model_update_interval
        self.historical_optimal_values = []
        self.historical_time = []
        self.n_attributes = self.model.output_dim
        self.n_hyps_samples = min(10, self.model.number_of_hyps_samples())
        self.n_parameter_samples = 10
        self.full_parameter_support = self.utility.parameter_dist.use_full_support
        self.evaluation_optimizer = GeneralOptimizer(optimizer='lbfgs', space=space)
        self.context = None
        self.current_argmax = np.atleast_2d(X_init[0, :])
        self.suggested_points = []

    def _n_hyps(self):
        eff = getattr(self.acquisition, "_n_hyps_effective", None)
        return eff() if eff is not None else self.n_hyps_samples

    # ---- reporting path (cbo.py:61-83, 121-235) ---------------------------------------------------------------
    def _current_max_value(self):
        val = 0
        if self.full_parameter_support:
            support = self.utility.parameter_dist.support
            dist = self.utility.parameter_dist.prob_dist
            for i in range(len(support)):
                marginal_argmax = self._current_marginal_argmax(support[i])
                marginal_max_val = np.reshape(self.objective.evaluate(marginal_argmax)[0], (self.n_attributes,))
                val += self.utility.eval_func(support[i], marginal_max_val) * dist[i]
        else:
            samples = self.utility.parameter_dist.sample(self.n_parameter_samples)
            for i in range(len(samples)):
                marginal_argmax = self._current_marginal_argmax(samples[i])
                marginal_max_val = np.reshape(self.objective.evaluate(marginal_argmax)[0], (self.n_attributes,))
                val += self.utility.eval_func(samples[i], marginal_max_val)
            val /= len(samples)
        return float(np.squeeze(val))

    def _current_marginal_argmax(self, parameter):
        """argmax_x E_n[U(theta, f(x))] (cbo.py:121-235).  The three objectives the reference evaluates candidate by
        candidate in Python -- posterior-mean utility (linear U), closed-form psi, 50-sample MC utility -- are one
        device call per L-BFGS round each (multi_outputGP.expected_utility -> psi_acq_kernel / mc_acq_kernel<_,3|4>)."""
        model = self.model
        if not hasattr(model, "expected_utility"):
            raise TypeError("CBO needs a bocf_b200.multi_outputGP (CUDA) model: there is no CPU path "
                            "(CPU models are driven through oracle.cbo.CBO in the tests)")
        n_h = self._n_hyps()
        comp = self.utility.composite
        self.utility.composite_id(model.output_dim, model.device)     # a CudaComposite: compiled and checked once
        if self.utility.linear:                                           # cbo.py:126-168
            if comp != "linear":
                raise ValueError("Utility(linear=True) needs composite='linear'")
            Z = None
        elif self.expectation_utility is not None:                        # cbo.py:170-198
            self._check_expectation_utility(parameter)
            Z = None
        else:                                                             # cbo.py:203-231
            Z = np.random.normal(size=(50, self.n_attributes))

        def val_func(X):
            val, _ = model.expected_utility(np.atleast_2d(X), comp, parameter, n_h, Z=Z, grad=False)
            return -val.reshape(-1, 1)

        def val_func_with_gradient(X):
            val, g = model.expected_utility(np.atleast_2d(X), comp, parameter, n_h, Z=Z, grad=True)
            return -val.reshape(-1, 1), -g

        argmax = self.evaluation_optimizer.optimize(f=val_func, f_df=val_func_with_gradient, parallel=False)[0]
        model.set_hyperparameters(n_h - 1)          # the reference's h loop leaves the model on its last hyper-sample
        self.current_argmax = argmax
        return argmax

    def _check_expectation_utility(self, parameter):
        """The ExpectationUtility callables of the reference's interface cannot run in a kernel: the device evaluates
        the closed form catalogued for the composite.  Checked once against the callables the user passed."""
        if getattr(self, "_psi_checked", False):
            return
        from .utility import _host_psi
        pair = _host_psi(self.utility.composite)
        if pair is None:
            raise ValueError("no closed-form expectation is catalogued for composite %r: pass expectation_utility=None "
                             "(MC branch)" % (self.utility.composite,))
        rng = np.random.default_rng(0)
        m = self.n_attributes
        mu, v = rng.standard_normal(m), rng.uniform(0.1, 1.0, m)
        th = np.asarray(parameter, dtype=float)
        ok = np.allclose(self.expectation_utility.func(th, mu, v), pair[0](th, mu, v), rtol=1e-9, atol=1e-12) and \
            np.allclose(np.asarray(self.expectation_utility.gradient(th, mu, v), dtype=float).reshape(-1),
                        np.asarray(pair[1](th, mu, v), dtype=float).reshape(-1), rtol=1e-9, atol=1e-12)
        if not ok:
            raise ValueError("expectation_utility disagrees with the closed form of composite %r"
                             % (self.utility.composite,))
        self._psi_checked = True

    # ---- main loop (cbo.py:238-329) ---------------------------------------------------------------------------
    def run_optimization(self, max_iter=1, parallel=False, plot=False, results_file=None, max_time=np.inf, eps=1e-8,
                         context=None, verbosity=False):
        if self.objective is None:
            raise InvalidConfigError("Cannot run the optimization loop without the objective function")
        self.verbosity = verbosity
        self.results_file = results_file
        self.context = context
        self.eps = eps
        if (max_iter is None) and (max_time is None):
            self.max_iter, self.max_time = 0, np.inf
        elif (max_iter is None) and (max_time is not None):
            self.max_iter, self.max_time = np.inf, max_time
        elif (max_iter is not None) and (max_time is None):
            self.max_iter, self.max_time = max_iter, np.inf
        else:
            self.max_iter, self.max_time = max_iter, max_time

        if self.X is not None and self.Y is None:
            self.Y, cost_values = self.objective.evaluate(self.X)
        self.model.updateModel(self.X, self.Y)

        self.time_zero = time.perf_counter()
        self.cum_time = 0
        self.num_acquisitions = 0
        self.suggested_sample = self.X
        self.Y_new = self.Y
        while (self.max_time > self.cum_time) and (self.num_acquisitions < self.max_iter):
            tmp = self.suggested_sample
            self.suggested_sample = self.compute_next_evaluations()
            if np.all(self.suggested_sample == tmp):
                self.suggested_sample = self._perturb(self.suggested_sample)
            # cbo.py:299-302 calls update_Z_samples() without its argument inside try/except: the TypeError is
            # swallowed, so Z is never refreshed in the reference (SURVEY.md section 3A); kept that way.
            self.suggested_points.append(np.array(self.suggested_sample))
            self.X = np.vstack((self.X, self.suggested_sample))
            self.evaluate_objective()
            if (self.num_acquisitions % self.model_update_interval) == 0:
                self._update_model()
            current_max_val = self._current_max_value()
            self.historical_optimal_values.append(current_max_val)
            self.cum_time = time.perf_counter() - self.time_zero
            self.historical_time.append(self.cum_time)
            self.num_acquisitions += 1
            if verbosity:
                print("num acquisition: {}, time elapsed: {:.2f}s".format(self.num_acquisitions, self.cum_time))
        if results_file is not None:
            self.save_results(results_file)

    def evaluate_objective(self):
        # cbo.py:354-363
        self.Y_new, cost_new = self.objective.evaluate_w_noise(self.suggested_sample)
        for j in range(self.n_attributes):
            self.Y[j] = np.vstack((self.Y[j], self.Y_new[j]))

    def _perturb(self, x):
        # cbo.py:372-378
        perturbed_x = np.copy(x)
        while np.all(perturbed_x == x):
            perturbed_x = x + np.random.normal(size=x.shape, scale=1e-2)
            perturbed_x = self.space.round_optimum(perturbed_x)
        return perturbed_x

    def compute_next_evaluations(self, pending_zipped_X=None, ignored_zipped_X=None):
        # cbo.py:381-405
        if self.X is not None and self.Y is None:
            self.Y, cost_values = self.objective.evaluate(self.X)
        self.model.updateModel(self.X, self.Y)
        self.acquisition.optimizer.context_manager = ContextManager(self.space, self.context)
        return self.space.zip_inputs(self.evaluator.compute_batch(duplicate_manager=None,
                                                                   x_baseline=self.current_argmax))

    def _update_model(self):
        # cbo.py:409-419
        X_inmodel = self.space.unzip_inputs(self.X)
        Y_inmodel = list(self.Y)
        self.model.updateModel(X_inmodel, Y_inmodel)

    def save_results(self, filename):
        # cbo.py:541-546
        results = np.zeros((len(self.historical_optimal_values), 2))
        results[:, 0] = self.historical_optimal_values
        results[:, 1] = self.historical_time
        np.savetxt(filename, results)
