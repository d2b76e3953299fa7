"""``SurrogateModel`` with alabi's API (alabi/core.py:125-2787) on the GPU GP.

Kept method names / kwargs: ``init_samples``, ``init_gp``, ``active_train``,
``find_next_point``, ``surrogate_log_likelihood``,
``create_cached_surrogate_likelihood``, ``lnprob``, ``run_emcee``,
``run_dynesty``, ``save`` and the ``training_results`` bookkeeping.  What changes
is where the arithmetic runs:

* every ``george.GP`` becomes an ``alabi_b200.GP`` (K1-K3 on the device);
* the acquisition search evaluates one candidate batch on the device (K4) and
  only polishes the winner with scipy (the reference runs ``nopt`` scipy
  restarts of one-point predicts, alabi/core.py:1587-1667);
* ``run_emcee`` on the surrogate runs the whole stretch-move chain on the
  device (K5) instead of ``emcee`` calling ``lnprob`` per walker — and does not
  re-factorise K for every log-probability like alabi/core.py:1430 does;
* ``run_dynesty`` feeds batched surrogate predicts to a nested sampler.

Out of scope (SURVEY 2, not on the hot path): plotting, pymultinest /
ultranest drivers, ``active_train_parallel``, MPI pools.
"""
import os
import pickle
import time
import warnings
from functools import partial

import numpy as np
import scipy.optimize as op

from . import gp_utils, mcmc_utils
from . import kernels
from . import utility as ut
from .ensemble import EnsembleSampler, SurrogateLogProb
from .gp import GP

__all__ = ["SurrogateModel", "CachedSurrogateLikelihood"]

_KERNELS = {"ExpSquaredKernel": kernels.ExpSquaredKernel, "Matern32Kernel": kernels.Matern32Kernel,
            "Matern52Kernel": kernels.Matern52Kernel, "RationalQuadraticKernel": kernels.RationalQuadraticKernel}


class CachedSurrogateLikelihood:
    """Picklable callable: pre-computed GP + scalers -> mean or (mean, var) at
    one point ``(ndim,)`` or many ``(M, ndim)`` (alabi/core.py:28-122)."""

    def __init__(self, gp_iter, _y_cond, theta_scaler, y_scaler, ndim, return_var=False):
        self.gp_iter, self._y_cond = gp_iter, _y_cond
        self.theta_scaler, self.y_scaler = theta_scaler, y_scaler
        self.ndim, self.return_var = ndim, return_var

    def __call__(self, theta_xs):
        theta_xs = np.asarray(theta_xs)
        one = theta_xs.ndim == 1
        if one:
            theta_xs = theta_xs.reshape(1, -1)
        elif theta_xs.ndim != 2:
            raise ValueError(f"theta_xs must be 1D or 2D array, got {theta_xs.ndim}D")
        _xs = np.atleast_2d(self.theta_scaler.transform(theta_xs))
        if not self.return_var:
            _yp = self.gp_iter.predict(self._y_cond, _xs, return_var=False, return_cov=False)
            yp = self.y_scaler.inverse_transform(_yp.reshape(-1, 1)).flatten()
            return yp[0] if one else yp
        _yp, _vp = self.gp_iter.predict(self._y_cond, _xs, return_var=True, return_cov=False)
        yp = self.y_scaler.inverse_transform(_yp.reshape(-1, 1)).flatten()
        if getattr(self.y_scaler, "scale_", None) is not None:
            vp = _vp * self.y_scaler.scale_[0] ** 2
        else:
            eps = 1e-6
            tr = self.y_scaler.inverse_transform(np.array([[0.0], [eps]]))
            vp = _vp * ((tr[1] - tr[0]) / eps) ** 2
        return (yp[0], vp[0]) if one else (yp, vp)


class _SharedPoint:
    """One-entry cache in front of ``GP.predict_grad`` for the acquisition polish: scipy
    evaluates the utility and then its gradient at the same point, and the device call
    that yields d mu / d sigma^2 also yields mu and sigma^2."""

    def __init__(self, gp, y):
        self.gp, self._y = gp, y
        self._key, self._val = None, None

    def _eval(self, xs):
        xs = np.ascontiguousarray(np.asarray(xs, dtype=np.float64).reshape(1, -1))
        key = xs.tobytes()
        if key != self._key:
            self._val = self.gp.predict_grad(self._y, xs)
            self._key = key
        return self._val

    def predict(self, xs):
        if np.asarray(xs).size != self.gp.kernel.ndim:          # not a single point: plain batched predict
            return self.gp.predict(self._y, xs, return_var=True)
        r = self._eval(xs)
        return r[0], r[1]

    def predict_grad(self, y, xs):
        return self._eval(xs)


class SurrogateModel(object):
    def __init__(self, lnlike_fn=None, bounds=None, param_names=None, cache=True, savedir="results/",
                 model_name="surrogate_model", verbose=True, ncore=1, pool_method="forkserver",
                 ignore_warnings=True, random_state=None, device=None):
        if lnlike_fn is None:
            raise ValueError("Must supply lnlike_fn to train GP surrogate model.")
        if bounds is None:
            raise ValueError("Must supply prior bounds.")
        if random_state is None:
            random_state = int(time.time() * 1000000) % (2 ** 32)
        self.random_state = random_state
        self.lnlike_fn = lnlike_fn
        self.true_log_likelihood = lnlike_fn
        self.bounds = np.array(bounds)
        self.prior_sampler = partial(ut.prior_sampler, bounds=self.bounds, sampler="uniform", random_state=None)
        self.ndim = len(self.bounds)
        if param_names is not None:
            if len(param_names) != len(bounds):
                raise ValueError("Length of param_names must match length of bounds.")
            self.param_names = self.labels = param_names
        else:
            self.param_names = [r"$\theta_%s$" % i for i in range(self.ndim)]
            self.labels = [f"theta_{i}" for i in range(self.ndim)]
        self.cache, self.savedir, self.model_name = cache, savedir, model_name
        if not os.path.exists(self.savedir):
            os.makedirs(self.savedir)
        self.verbose = verbose
        if ignore_warnings:
            warnings.filterwarnings("ignore", category=UserWarning)
            warnings.filterwarnings("ignore", category=FutureWarning)
        self.pool_method = pool_method
        self.ncore = max(int(ncore), 1)        # likelihood evaluations only; GP work is on the GPU
        self.device = device
        self.emcee_run = self.dynesty_run = self.ultranest_run = False

    # -- persistence (alabi/core.py:327-404) ----------------------------------------
    def __getstate__(self):
        state = self.__dict__.copy()
        state["pool"] = None
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)

    def save(self):
        file = os.path.join(self.savedir, self.model_name)
        print(f"Caching model to {file}...")
        tmp = file + ".pkl.tmp"
        try:
            with open(tmp, "wb") as f:
                pickle.dump(self, f)
            os.rename(tmp, file + ".pkl")
        except Exception:
            if os.path.exists(tmp):
                os.remove(tmp)
            raise
        # human-readable report next to the pickle (alabi/core.py:394-404)
        from . import cache_utils
        if hasattr(self, "gp"):
            try:
                cache_utils.write_report_gp(self, file)
            except Exception as e:  # noqa: BLE001 - the reference reports and goes on
                print(f"Error writing GP report: {e}")
        if getattr(self, "emcee_run", False):
            cache_utils.write_report_emcee(self, file)
        if getattr(self, "dynesty_run", False):
            cache_utils.write_report_dynesty(self, file)

    # -- data / scalers ---------------------------------------------------------------
    def theta(self):
        return self.theta_scaler.inverse_transform(self._theta)

    def y(self):
        return self.y_scaler.inverse_transform(self._y.reshape(-1, 1)).flatten()

    def refit_scalers(self, theta, y, theta_scaler=None, y_scaler=None):
        if theta_scaler is not None:
            self.theta_scaler = theta_scaler
        if y_scaler is not None:
            self.y_scaler = y_scaler
        self.theta_scaler.fit(self.bounds.T)
        _theta = self.theta_scaler.transform(theta)
        _y = self.y_scaler.fit_transform(np.asarray(y).reshape(-1, 1)).flatten()
        for arr, nm in ((_theta, "theta_scaler"), (_y, "y_scaler")):
            if np.any(np.isnan(arr)):
                raise ValueError(f"Refitted {nm} produced NaN values!")
            if np.any(np.isinf(arr)):
                raise ValueError(f"Refitted {nm} produced Inf values!")
        return _theta, _y

    def init_train(self, nsample=None, sampler="uniform", fname="initial_training_sample.npz"):
        if nsample is None:
            nsample = 50 * self.ndim
        theta = self.prior_sampler(nsample=nsample, sampler=sampler, random_state=None)
        y = np.array([self.true_log_likelihood(tt) for tt in theta], dtype=float).reshape(-1, 1)
        for ii in range(len(y)):
            while not np.isfinite(y[ii]):
                new_theta = self.prior_sampler(nsample=1, sampler="uniform", random_state=None)
                y[ii] = np.asarray(self.true_log_likelihood(new_theta.flatten())).reshape(-1)[0]
                theta[ii] = new_theta
        if self.cache:
            np.savez(f"{self.savedir}/{fname}", theta=theta, y=y)
        return theta, y

    def load_train(self, cache_file):
        sims = np.load(cache_file)
        theta, y = sims["theta"], sims["y"]
        if self.ndim != theta.shape[1]:
            raise ValueError(f"Dimension of bounds (n={self.ndim}) does not match dimension of training theta "
                             f"(n={theta.shape[1]})")
        return theta, y

    def _load_or_train(self, n, sampler, file, default_name, what):
        if file is not None:
            cache_file = file if os.path.exists(file) else f"{self.savedir}/{file}"
            try:
                theta, y = self.load_train(cache_file)
                print(f"Loaded {len(theta)} {what} samples from {cache_file}.")
                return theta, y
            except Exception as e:  # noqa: BLE001
                print(f"Unable to reload {cache_file} due to error: {e}. Computing new samples...")
                return self.init_train(nsample=n, sampler=sampler, fname=file)
        return self.init_train(nsample=n, sampler=sampler, fname=default_name)

    def init_samples(self, ntrain=100, ntest=0, sampler="uniform", train_file=None, test_file=None):
        theta, y = self._load_or_train(ntrain, sampler, train_file, "initial_train_file_sample.npz", "train")
        if ntest > 0:
            self.theta_test, self.y_test = self._load_or_train(ntest, sampler, test_file,
                                                               "initial_test_sample.npz", "test")
            self.ntest = len(self.theta_test)
        else:
            self.theta_test, self.y_test, self.ntest = [], [], 0
        self.theta_train, self.y_train = theta, y
        self.ninit_train = self.ntrain = len(theta)
        self.nactive = 0

    # -- hyper-parameter vector plumbing (alabi/core.py:628-733) ----------------------------
    def set_hyperparam_prior_bounds(self):
        pnames = self.param_names_optimized if self.uniform_scales else self.param_names_full
        hp_bounds = [[None, None] for _ in pnames]
        if self.fit_mean:
            m, s = np.mean(self._y), np.std(self._y)
            hp_bounds[pnames.index("mean:value")] = [m - s, m + s]
        if self.fit_amp:
            v = np.var(self._y)
            hp_bounds[pnames.index(f"{self.kernel_amp_key}:log_constant")] = \
                [v * 10 ** self.gp_amp_rng[0], v * 10 ** self.gp_amp_rng[1]]
        if self.fit_white_noise:
            hp_bounds[pnames.index("white_noise:value")] = [self.white_noise - 3, self.white_noise + 3]
        if self._alpha_key() in pnames:
            hp_bounds[pnames.index(self._alpha_key())] = self.gp_alpha_rng
        if self.uniform_scales:
            hp_bounds[pnames.index(f"{self.kernel_scale_key}:metric:log_M")] = self.gp_scale_rng
        else:
            for ii in range(self.ndim):
                hp_bounds[pnames.index(f"{self.kernel_scale_key}:metric:log_M_{ii}_{ii}")] = self.gp_scale_rng
        self.hp_bounds = np.array(hp_bounds)
        self.gp_hyper_prior = partial(ut.lnprior_uniform, bounds=self.hp_bounds)

    def expand_hyperparameter_vector(self, optimized_params):
        if optimized_params is None:
            raise ValueError("optimized_params cannot be None")
        if not self.uniform_scales:
            return optimized_params
        full = np.ones(len(self.param_names_full))
        po, pf = self.param_names_optimized, self.param_names_full
        for on, name in ((self.fit_mean, "mean:value"),
                         (self.fit_amp, f"{getattr(self, 'kernel_amp_key', 'kernel')}:log_constant"),
                         (self.fit_white_noise, "white_noise:value")):
            if on:
                full[pf.index(name)] = optimized_params[po.index(name)]
        if self._alpha_key() in pf:
            full[pf.index(self._alpha_key())] = optimized_params[po.index(self._alpha_key())]
        for ii in range(self.ndim):
            full[pf.index(f"{self.kernel_scale_key}:metric:log_M_{ii}_{ii}")] = \
                optimized_params[po.index(f"{self.kernel_scale_key}:metric:log_M")]
        return np.array(full)

    def _alpha_key(self):
        """Name of the rational quadratic kernel's log_alpha in the george vector (absent for the other kernels)."""
        return f"{self.kernel_scale_key}:log_alpha"

    def set_hyperparameter_vector(self, tmp_gp, optimized_params):
        if optimized_params is None:
            raise ValueError("optimized_params cannot be None. Cannot set hyperparameters.")
        full = optimized_params
        if self.uniform_scales:
            # A vector that already has the full george length (what active_train hands to _fit_gp:
            # gp.get_parameter_vector()) is used as it is.  The reference re-expands it through the
            # positions of the OPTIMISED names (alabi/core.py:1780 -> 695-704), which swaps amplitude
            # and white noise on every refit; that accident is not reproduced.
            # ``reference_double_expansion = True`` (attribute, default off) reproduces it: the objective of
            # the reference's ML search then sees amplitude and white noise swapped, exactly as its code does
            # (pinned by tests/golden/hostlogic_golden.npz, generated from the reference's own init_gp).
            if getattr(self, "reference_double_expansion", False) or \
                    not (self.ndim > 1 and len(np.atleast_1d(optimized_params)) == len(self.param_names_full)):
                full = self.expand_hyperparameter_vector(optimized_params)
        tmp_gp.set_parameter_vector(full)
        return tmp_gp

    def get_hyperparameter_dict(self, gp):
        hp = gp.get_parameter_dict()
        if self.uniform_scales:
            hp[f"{self.kernel_scale_key}:metric:log_M"] = hp.pop(f"{self.kernel_scale_key}:metric:log_M_0_0")
            for ii in range(1, self.ndim):
                del hp[f"{self.kernel_scale_key}:metric:log_M_{ii}_{ii}"]
        return hp

    def get_hyperparameter_vector(self, gp):
        return np.fromiter(self.get_hyperparameter_dict(gp).values(), dtype=float)

    # -- GP initialisation (alabi/core.py:736-1094) ---------------------------------------
    def init_gp(self, kernel="ExpSquaredKernel", fit_amp=True, fit_mean=True, fit_white_noise=True,
                white_noise=-12, gp_scale_rng=[-2, 2], gp_amp_rng=[-1, 1], gp_alpha_rng=[-2, 2], uniform_scales=False,
                overwrite=False,
                theta_scaler=ut.no_scaler, y_scaler=ut.no_scaler, gp_opt_method="l-bfgs-b", gp_nopt=3,
                optimizer_kwargs={"maxiter": 100, "xatol": 1e-4, "fatol": 1e-3, "adaptive": True},
                hyperopt_method="cv", regularize=True, amp_0=1.0, mu_0=1.0, sigma_0=2.0, cv_folds=5,
                cv_scoring="mse", cv_n_candidates=100, cv_stage2_candidates=50, cv_stage2_width=0.5,
                cv_stage3_candidates=25, cv_stage3_width=0.2, cv_weighted_factor=1.0, multi_proc=True):
        if hasattr(self, "gp") and not overwrite:
            raise AssertionError("GP kernel already assigned. Use overwrite=True to re-assign the kernel.")
        self.fit_amp, self.fit_mean, self.fit_white_noise = fit_amp, fit_mean, fit_white_noise
        self.white_noise, self.uniform_scales = white_noise, uniform_scales
        self.gp_opt_method, self.gp_nopt = gp_opt_method, gp_nopt
        self.opt_gp_kwargs = {"hyperopt_method": hyperopt_method, "regularize": regularize, "amp_0": amp_0,
                              "mu_0": mu_0, "sigma_0": sigma_0, "optimizer_kwargs": optimizer_kwargs,
                              "cv_folds": cv_folds, "cv_scoring": cv_scoring, "cv_n_candidates": cv_n_candidates,
                              "cv_stage2_candidates": cv_stage2_candidates, "cv_stage2_width": cv_stage2_width,
                              "cv_stage3_candidates": cv_stage3_candidates, "cv_stage3_width": cv_stage3_width,
                              "cv_weighted_factor": cv_weighted_factor, "multi_proc": multi_proc}
        self.theta_scaler = theta_scaler
        self.theta_scaler.fit(self.bounds.T)
        self._bounds = self.theta_scaler.transform(self.bounds.T).T
        self._prior_sampler = partial(ut.prior_sampler, bounds=self._bounds, sampler="uniform", random_state=None)
        self.y_scaler = y_scaler
        self._theta, self._y = self.refit_scalers(self.theta_train, self.y_train)
        if self.ntest > 0:
            self._theta_test = self.theta_scaler.transform(self.theta_test)
            self._y_test = self.y_scaler.transform(np.asarray(self.y_test).reshape(-1, 1)).flatten()
        self._theta_train, self._y_train = self._theta, self._y
        self.training_results = {k: [] for k in (
            "iteration", "gp_hyperparameters", "gp_hyperparameter_opt_iteration", "gp_hyperparam_opt_time",
            "training_mse", "test_mse", "training_scaled_mse", "test_scaled_mse", "gp_kl_divergence",
            "gp_train_time", "obj_fn_opt_time", "acquisition_optimizer_niter")}
        self.gp_scale_rng, self.gp_amp_rng = gp_scale_rng, gp_amp_rng
        self.gp_alpha_rng = gp_alpha_rng      # bounds of ln(alpha) (RationalQuadraticKernel only)
        log_metric_bounds = [(min(gp_scale_rng), max(gp_scale_rng)) for _ in range(self.ndim)]
        if kernel not in _KERNELS:
            raise ValueError(f"Kernel '{kernel}' is not a valid option. Valid options: " + ", ".join(_KERNELS))
        self.gp = None
        for attempt in range(1, 11):       # retry with new random scale lengths (alabi/core.py:980-1048)
            log_l = np.random.uniform(min(gp_scale_rng), max(gp_scale_rng), self.ndim)
            if kernel == "RationalQuadraticKernel":
                # starts at alpha = 1; the reference's starting value for this kernel could not be checked
                self.kernel = _KERNELS[kernel](log_alpha=0.0, metric=np.exp(log_l), metric_bounds=log_metric_bounds,
                                               ndim=self.ndim)
            else:
                self.kernel = _KERNELS[kernel](metric=np.exp(log_l), metric_bounds=log_metric_bounds, ndim=self.ndim)
            self.kernel_name = kernel
            self.gp = gp_utils.configure_gp(self._theta, self._y, self.kernel, fit_amp=fit_amp, fit_mean=fit_mean,
                                            fit_white_noise=fit_white_noise, white_noise=white_noise,
                                            device=self.device)
            if self.gp is not None:
                if self.verbose:
                    print(f"Successfully initialized GP ({kernel}) on attempt {attempt}")
                break
            print("Warning: configure_gp returned None. Retrying with new initial scale length...")
        if self.gp is None:
            del self.gp
            raise RuntimeError(f"Failed to initialize GP after 10 attempts. Check your data, kernel choice, and "
                               f"scale bounds. Current settings: kernel={kernel}, gp_scale_rng={gp_scale_rng}")
        self.param_names_full = list(self.gp.get_parameter_names(include_frozen=False))
        self.param_names_optimized = []
        self.kernel_scale_key = [x for x in self.param_names_full if "metric:log_M" in x][0].split(":metric:log_M")[0]
        if fit_mean:
            self.param_names_optimized.append("mean:value")
        if fit_amp:
            self.kernel_amp_key = [x for x in self.param_names_full if "log_constant" in x][0].split(":log_constant")[0]
            self.param_names_optimized.append(f"{self.kernel_amp_key}:log_constant")
        if fit_white_noise:
            self.param_names_optimized.append("white_noise:value")
        if self._alpha_key() in self.param_names_full:
            self.param_names_optimized.append(self._alpha_key())
        if self.uniform_scales:
            self.param_names_optimized.append(f"{self.kernel_scale_key}:metric:log_M")
        else:
            self.param_names_optimized += [f"{self.kernel_scale_key}:metric:log_M_{ii}_{ii}" for ii in range(self.ndim)]
        self.hp_length_indices = [i for i, nm in enumerate(self.param_names_full) if "metric:log_m" in nm.lower()]
        self.hp_other_indices = [i for i, nm in enumerate(self.param_names_full) if "metric:log_m" not in nm.lower()]
        if self.uniform_scales:
            self.hp_length_index = [self.param_names_optimized.index(f"{self.kernel_scale_key}:metric:log_M")]
        self.initial_gp_hyperparameters = self.get_hyperparameter_vector(self.gp)
        self.gp, _ = self._opt_gp(**self.opt_gp_kwargs)
        if self.ntest > 0:
            _yt = self.gp.predict(self._y, self._theta_test, return_cov=False, return_var=False)
            yt = self.y_scaler.inverse_transform(_yt.reshape(-1, 1)).flatten()
            yt_true = self.y_scaler.inverse_transform(self._y_test.reshape(-1, 1)).flatten()
            return np.mean((yt_true - yt) ** 2)
        return None

    def _new_gp(self, _y):
        kernel = self.kernel * np.var(_y) if self.fit_amp else self.kernel
        return GP(kernel=kernel, fit_mean=self.fit_mean, mean=np.median(_y), white_noise=self.white_noise,
                  fit_white_noise=self.fit_white_noise, device=self.device)

    def _fit_gp(self, _theta=None, _y=None, hyperparameters=None):
        """New GP (amplitude var(y), mean median(y)) with the given hyper-vector,
        factorised on ``_theta`` (alabi/core.py:1097-1160)."""
        _theta = self._theta if _theta is None else _theta
        _y = self._y if _y is None else _y
        t0 = time.time()
        self.set_hyperparam_prior_bounds()
        if not np.all(np.isfinite(_theta)):
            raise ValueError("_theta contains NaN or Inf values")
        if not np.all(np.isfinite(_y)):
            raise ValueError(f"_y contains NaN or Inf values: {_y[~np.isfinite(_y)]}")
        y_var = np.var(_y)
        if not np.isfinite(y_var) or y_var == 0:
            raise ValueError(f"var(_y) is not finite or zero: {y_var}")
        gp = self._new_gp(_y)
        if hyperparameters is not None and not np.all(np.isfinite(np.atleast_1d(hyperparameters))):
            print(f"Warning: Hyperparameters contain NaN or Inf: {hyperparameters}\nReoptimizing from scratch...")
            gp, _ = self._opt_gp(**self.opt_gp_kwargs, _theta=_theta, _y=_y)
            if not np.all(np.isfinite(gp.get_parameter_vector())):
                raise ValueError("Reoptimized GP still has invalid parameters")
            return gp, time.time() - t0
        gp = self.set_hyperparameter_vector(gp, hyperparameters)
        gp.compute(_theta)
        return gp, time.time() - t0

    def _append_gp(self, _theta_prop, _y_prop):
        """O(N^2) alternative to ``_fit_gp`` for the active-learning step: when exactly
        one point was appended and the hyper-parameters are the current ones, the
        factor is extended by a bordered Cholesky update (``GP.append_point``) instead
        of being rebuilt (the reference refactorises, alabi/core.py:1780).  Returns
        None when the preconditions do not hold; ``incremental_fit = False`` disables it."""
        gp = getattr(self, "gp", None)
        if not getattr(self, "incremental_fit", True) or gp is None or not self.fit_mean:
            return None
        x_old = gp._x
        if not gp.computed or x_old is None or len(_theta_prop) != len(x_old) + 1:
            return None
        # theta() -> transform() round trips may move old points by an ulp
        tol = 8 * np.finfo(float).eps * max(1.0, float(np.max(np.abs(x_old))))
        if np.max(np.abs(np.asarray(_theta_prop)[:-1] - x_old)) > tol:
            return None
        t0 = time.time()
        try:
            gp.append_point(np.asarray(_theta_prop)[-1])
        except np.linalg.LinAlgError:
            return None
        return gp, time.time() - t0

    def _ml_objective(self, cur, _y, regularize=True, amp_0=1.0, mu_0=1.0, sigma_0=2.0):
        """(nll, grad_nll) of the maximum-likelihood search exactly as the reference composes them
        (alabi/core.py:1242-1278): negative log marginal likelihood of ``cur`` at the (expanded)
        hyper-vector plus the length-scale regulariser, non-finite -> 1e25; with
        ``uniform_scales`` the tied length scale receives the MEAN of the per-dimension
        gradients and the other entries are copied by their positions in the FULL vector
        (kept as the reference has it).  Every evaluation is one device factorisation."""
        kw = dict(amp_0=amp_0, mu_0=mu_0, sigma_0=sigma_0)

        def nll(p_opt):
            p = self.expand_hyperparameter_vector(p_opt) if self.uniform_scales else p_opt
            ll = -self.set_hyperparameter_vector(cur, p).log_likelihood(_y, quiet=True)
            if regularize:
                ll += gp_utils.regularization_term(p, self.hp_length_indices, **kw)
            return ll if np.isfinite(ll) else 1e25

        def grad_nll(p_opt):
            p = self.expand_hyperparameter_vector(p_opt) if self.uniform_scales else p_opt
            g = -self.set_hyperparameter_vector(cur, p).grad_log_likelihood(_y, quiet=True)
            if self.uniform_scales:
                gll = np.zeros(len(p_opt))
                gll[self.hp_length_index] = np.mean(g[self.hp_length_indices])
                gll[self.hp_other_indices] = g[self.hp_other_indices]
            else:
                gll = g
            if regularize:
                rg = gp_utils.regularization_gradient(p, self.hp_length_indices, **kw)
                if self.uniform_scales:
                    gll[self.hp_length_index] += np.mean(rg[self.hp_length_indices])
                else:
                    gll = gll + rg
            return gll
        return nll, grad_nll

    def _opt_gp(self, hyperopt_method="ml", regularize=True, amp_0=1.0, mu_0=1.0, sigma_0=2.0,
                optimizer_kwargs={"maxiter": 100, "xatol": 1e-4, "fatol": 1e-3, "adaptive": True}, cv_folds=5,
                cv_scoring="mse", cv_n_candidates=20, multi_proc=True, cv_stage2_candidates=None,
                cv_stage2_width=0.5, cv_stage3_candidates=None, cv_stage3_width=0.2,
                cv_weighted_mse_method="exponential", cv_weighted_factor=1.0, _theta=None, _y=None,
                theta_scaler=None, y_scaler=None):
        """Hyper-parameter optimisation: "ml" = gp_nopt L-BFGS-B restarts on the
        regularised negative log marginal likelihood (each evaluation is one
        device factorisation + gradient, K2); "cv" = k-fold random search
        (alabi/core.py:1163-1404)."""
        t0 = time.time()
        _theta = self._theta if _theta is None else _theta
        _y = self._y if _y is None else _y
        if hyperopt_method.lower() not in ("ml", "cv"):
            print(f"Invalid method '{hyperopt_method}'. Must be 'ml' or 'cv'. Defaulting to 'ml'.")
            hyperopt_method = "ml"
        use_gradient = self.gp_opt_method in ("newton-cg", "l-bfgs-b")
        self.set_hyperparam_prior_bounds()
        op_gp = None
        if hyperopt_method.lower() == "ml":
            cur = self.gp
            cur.compute(_theta)
            nll, grad_nll = self._ml_objective(cur, _y, regularize=regularize, amp_0=amp_0, mu_0=mu_0, sigma_0=sigma_0)

            def _optimize_fn(x0):
                return op.minimize(fun=nll, x0=x0, jac=grad_nll if use_gradient else None,
                                   method=self.gp_opt_method, bounds=self.hp_bounds, options=optimizer_kwargs)

            current_hp = self.get_hyperparameter_vector(cur)
            if self.gp_nopt <= 1:
                results = _optimize_fn(current_hp)
            else:
                p0 = ut.prior_sampler(bounds=self.hp_bounds, nsample=self.gp_nopt, sampler="lhs", random_state=None)
                p0[0] = current_hp
                from . import parallel as par
                if getattr(self, "shard_restarts", False) and par.world_size() > 1:
                    # restart r on rank r mod world, one all_gather of (fun, x) (SURVEY 8e)
                    results, _ = par.sharded_restarts(_optimize_fn, par.broadcast_object(p0))
                else:
                    results = min([_optimize_fn(p) for p in p0], key=lambda r: r.fun)
            op_gp = self.set_hyperparameter_vector(cur, results.x)
            try:
                op_gp.compute(_theta)
            except np.linalg.LinAlgError:
                # every restart ended on a hyper-vector whose covariance matrix does not
                # factorise (fun = 1e25): the reference raises here (alabi/core.py:1313-1314);
                # keeping the current hyper-parameters lets a long active-learning run go on
                print(f"Warning: optimised GP hyper-parameters {np.asarray(results.x)} are not factorisable "
                      f"(fun = {results.fun}); keeping the current ones")
                op_gp = self.set_hyperparameter_vector(cur, current_hp)
                op_gp.compute(_theta)
            if self.verbose:
                print(f"-logL {nll(current_hp):.4f} -> {nll(results.x):.4f} | {results.nit} iterations | "
                      f"Success: {results.success}")
        else:
            if self.verbose:
                print(f"\nOptimizing GP hyperparameters using {cv_folds}-fold cross-validation...")
            try:
                cands = ut.prior_sampler(bounds=self.hp_bounds, nsample=cv_n_candidates, sampler="lhs",
                                         random_state=None)
                if hasattr(self, "gp"):
                    cands[0] = self.get_hyperparameter_vector(self.gp)
                if self.uniform_scales:
                    cands = np.array([self.expand_hyperparameter_vector(c) for c in cands])
                op_gp = gp_utils.optimize_gp_kfold_cv(
                    self.gp, _theta, _y, cands, self.y_scaler, k_folds=cv_folds, scoring=cv_scoring, pool=None,
                    stage2_candidates=cv_stage2_candidates, stage2_width=cv_stage2_width,
                    stage3_candidates=cv_stage3_candidates, stage3_width=cv_stage3_width,
                    weighted_mse_method=cv_weighted_mse_method, weighted_mse_factor=cv_weighted_factor,
                    verbose=self.verbose and not multi_proc)
            except Exception as e:  # noqa: BLE001 - reference keeps the current GP when CV fails
                print(f"Warning: CV hyperparameter optimization failed: {e}\nKeeping the current GP...")
                op_gp = None
        if op_gp is None:
            if hasattr(self, "gp") and self.gp is not None:
                op_gp = self.gp
                op_gp.compute(_theta)
            else:
                op_gp = self._new_gp(_y)
                op_gp.compute(_theta)
        timing = time.time() - t0
        self.training_results["gp_hyperparam_opt_time"].append(timing)
        return op_gp, timing

    # -- surrogate evaluation (alabi/core.py:1406-1584) --------------------------------------
    def _conditioning(self, iter):
        """(theta, y, hyper-vector) the surrogate of iteration ``iter`` is built on."""
        tr = self.training_results
        if iter == 0 or len(tr["iteration"]) == 0:
            hp = tr["gp_hyperparameters"][0] if len(tr["gp_hyperparameters"]) else self.initial_gp_hyperparameters
            return self._theta[:self.ninit_train], self._y[:self.ninit_train], hp
        if iter == -1 or iter == len(tr["iteration"]):
            return self._theta, self._y, tr["gp_hyperparameters"][-1]
        if 0 < iter < len(tr["iteration"]):
            n = self.ninit_train + iter
            return self._theta[:n], self._y[:n], tr["gp_hyperparameters"][iter]
        raise ValueError(f"Iteration {iter} exceeds available training iterations ({tr['iteration'][-1]}).")

    def eval_gp_at_iteration(self, iter, return_var=False):
        """Predictor of the GP as it was at active-learning iteration ``iter``.
        The reference refactorises K on EVERY call (alabi/core.py:1430); here the
        latest iteration reuses the factor that ``active_train`` already holds."""
        _tc, _yc, hp = self._conditioning(iter)
        latest = len(_tc) == len(self._theta) and np.array_equal(np.asarray(hp), self.gp.get_parameter_vector()) \
            and self.gp.computed and self.gp._x is not None and len(self.gp._x) == len(_tc)
        if latest:
            gp_iter = self.gp
        else:
            gp_iter = self.set_hyperparameter_vector(self._new_gp(_yc), hp)
            gp_iter.compute(_tc)

        def gp_predict(x):
            x = np.atleast_2d(x)
            if x.shape[1] != self.ndim and x.size == self.ndim:
                x = x.reshape(1, -1)
            return gp_iter.predict(_yc, x, return_var=return_var, return_cov=False)
        return gp_predict

    def surrogate_log_likelihood(self, theta_xs, iter=-1, return_var=False):
        theta_xs = np.asarray(theta_xs)
        one = theta_xs.ndim == 1
        if one:
            theta_xs = theta_xs.reshape(1, -1)
        elif theta_xs.ndim != 2:
            raise ValueError(f"theta_xs must be 1D or 2D array, got {theta_xs.ndim}D")
        _xs = self.theta_scaler.transform(theta_xs)
        if hasattr(self, "training_results") and len(self.training_results["iteration"]) > 0:
            gp_ii = self.eval_gp_at_iteration(iter, return_var=return_var)
        else:
            gp_ii = lambda x: self.gp.predict(self._y, x, return_var=return_var, return_cov=False)
        if not return_var:
            yp = self.y_scaler.inverse_transform(gp_ii(_xs).reshape(-1, 1)).flatten()
            return yp[0] if one else yp
        _yp, _vp = gp_ii(_xs)
        yp = self.y_scaler.inverse_transform(_yp.reshape(-1, 1)).flatten()
        vp = self.y_scaler.inverse_transform(_vp.reshape(-1, 1)).flatten()
        return (yp[0], vp[0]) if one else (yp, vp)

    def surrogate_likelihood(self, theta_xs):
        return np.exp(self.surrogate_log_likelihood(theta_xs))

    def create_cached_surrogate_likelihood(self, iter=-1, return_var=False):
        if hasattr(self, "training_results") and len(self.training_results["iteration"]) > 0:
            _tc, _yc, _ = self._conditioning(iter)
            hp = self.training_results["gp_hyperparameters"][-1]      # reference always uses the last vector
        else:
            _tc, _yc, hp = self._theta, self._y, self.gp.get_parameter_vector()
        gp_iter = gp_utils.configure_gp(_tc, _yc, self.kernel, fit_amp=self.fit_amp, fit_mean=self.fit_mean,
                                        fit_white_noise=self.fit_white_noise, white_noise=self.white_noise,
                                        hyperparameters=hp, device=self.device)
        if gp_iter is None:
            raise RuntimeError("create_cached_surrogate_likelihood: covariance matrix is not positive definite")
        return CachedSurrogateLikelihood(gp_iter, _yc, self.theta_scaler, self.y_scaler, self.ndim,
                                         return_var=return_var)

    def _device_log_prob(self, iter=-1, bounds=None, prior_data=None):
        """SurrogateLogProb (GP mean + uniform or box-times-normal prior) for the device sampler."""
        _tc, _yc, hp = self._conditioning(iter) if len(self.training_results["iteration"]) > 0 else \
            (self._theta, self._y, self.gp.get_parameter_vector())
        gp = self.gp
        if not (gp.computed and gp._x is not None and len(gp._x) == len(_tc)
                and np.array_equal(np.asarray(hp), gp.get_parameter_vector())):
            gp = self.set_hyperparameter_vector(self._new_gp(_yc), hp)
            gp.compute(_tc)
        ts, to = ut.scaler_affine(self.theta_scaler, self.ndim)
        yk, ys, yo = ut.scaler_affine(self.y_scaler, self.ndim, inverse=True)
        return SurrogateLogProb(gp, _yc, self.bounds if bounds is None else bounds, ts, to, yk, ys, yo,
                                prior_data=prior_data)

    @staticmethod
    def _device_prior(prior_fn):
        """(bounds, prior_data) of a prior the device sampler evaluates itself: a
        ``functools.partial`` of ``ut.lnprior_uniform`` (bounds) or ``ut.lnprior_normal``
        (bounds, data) -- the two priors the reference ships (alabi/utility.py:218-275,
        370-378).  Any other callable is host Python and cannot run inside the kernel."""
        fn = getattr(prior_fn, "func", None)
        name = getattr(fn, "__name__", None)
        if not isinstance(prior_fn, partial) or name not in ("lnprior_uniform", "lnprior_normal"):
            raise NotImplementedError("alabi_b200.run_emcee evaluates the prior on the GPU: pass "
                                      "functools.partial(ut.lnprior_uniform, bounds=...) or "
                                      "functools.partial(ut.lnprior_normal, bounds=..., data=...)")
        names = ("bounds",) if name == "lnprior_uniform" else ("bounds", "data")
        kw = dict(zip(names, prior_fn.args))          # positional after x
        kw.update(prior_fn.keywords or {})
        if "bounds" not in kw or (name == "lnprior_normal" and "data" not in kw):
            raise ValueError(f"{name}: the partial must bind {names}")
        return np.asarray(kw["bounds"], dtype=np.float64), (kw.get("data") if name == "lnprior_normal" else None)

    # -- active learning (alabi/core.py:1587-1865) -----------------------------------------------
    def find_next_point(self, nopt=3, optimizer_kwargs={}, ncand=None):
        """Next training point: the utility is evaluated over a batch of uniform
        candidates on the device (K4, argmin over finite values); the winner and
        the next-best starts are then polished with ``nopt`` scipy runs of
        ``obj_opt_method`` on the one-point utility.  ``obj_opt_method="batch"``
        skips the polish."""
        t0 = time.time()
        predict_gp = lambda _xs: self.gp.predict(self._y, _xs, return_var=True)
        y_best = np.max(self._y)
        if self.algorithm == "jones":
            obj_fn = partial(self.utility, predict_gp=predict_gp, bounds=self._bounds, y_best=y_best)
        else:
            obj_fn = partial(self.utility, predict_gp=predict_gp, bounds=self._bounds)
        ncand = int(ncand or getattr(self, "ncand", None) or min(4096 * self.ndim, 65536))
        cand = self._prior_sampler(nsample=ncand)
        idx, val, util = self.gp.utility_argmin(self._y, cand, self._bounds, algorithm=self.algorithm,
                                                y_best=y_best, return_values=True)
        _thetaN = np.nan
        if idx >= 0:
            _thetaN, best = cand[idx].copy(), val
            if str(self.obj_opt_method).lower() != "batch" and nopt > 0:
                u = util.cpu().numpy()
                order = np.argsort(np.where(np.isfinite(u), u, np.inf))[:max(int(nopt), 1)]
                grad_obj_fn = None                      # alabi/core.py:1613-1618
                if getattr(self, "grad_utility", None) is not None:
                    self.gp._set_targets(self._y)
                    # the optimiser asks for the utility and its gradient at the same point: both
                    # are served by ONE device call (same kernels, same bits as separate calls)
                    grad_obj_fn = partial(self.grad_utility, gp=self.gp, bounds=self._bounds)
                    if str(self.obj_opt_method).lower() in ("l-bfgs-b", "bfgs", "cg", "newton-cg", "tnc", "slsqp", "trust-constr"):
                        shared = _SharedPoint(self.gp, self._y)     # methods that do use the gradient
                        obj_fn = partial(obj_fn.func, **{**obj_fn.keywords, "predict_gp": shared.predict})
                        grad_obj_fn = partial(self.grad_utility, gp=shared, bounds=self._bounds)
                tp, fp = ut.minimize_objective(obj_fn, bounds=self._bounds, nopt=len(order),
                                               method=self.obj_opt_method, options=optimizer_kwargs or None,
                                               grad_obj_fn=grad_obj_fn, starting_points=cand[order])
                if np.all(np.isfinite(tp)) and np.isfinite(fp) and fp < best:
                    _thetaN, best = np.asarray(tp), fp
        opt_timing = time.time() - t0
        if not np.all(np.isfinite(_thetaN)):
            print("Warning: Acquisition function optimization failed. Falling back to random sampling.")
            _thetaN = self._prior_sampler(nsample=1).flatten()
        thetaN = self.theta_scaler.inverse_transform(_thetaN.reshape(1, -1))
        yN = np.asarray(self.true_log_likelihood(thetaN.flatten()), dtype=float).reshape(-1)
        if not np.all(np.isfinite(yN)):
            print(f"New y value is NaN or Inf: {yN}. Check your likelihood function at theta={thetaN}")
            return None, None, opt_timing
        theta_prop = np.append(self.theta(), thetaN, axis=0)
        y_prop = np.append(self.y(), yN)
        _theta_prop, _y_prop = self.refit_scalers(theta_prop, y_prop)
        if not (np.all(np.isfinite(_theta_prop)) and np.all(np.isfinite(_y_prop))):
            return None, None, opt_timing
        return _theta_prop, _y_prop, opt_timing

    def active_train(self, niter=100, algorithm="bape", gp_opt_freq=20, save_progress=False,
                     obj_opt_method="l-bfgs-b", nopt=5, optimizer_kwargs={}, use_grad_opt=True, show_progress=True,
                     allow_opt_multiproc=True, max_attempts=10, ncand=None):
        self.algorithm = str(algorithm).lower()
        self.utility, self.grad_utility = ut.assign_utility(self.algorithm)
        if not use_grad_opt:
            self.grad_utility = None
        self.gp_opt_freq, self.obj_opt_method, self.ncand = gp_opt_freq, obj_opt_method, ncand
        tr = self.training_results
        first_iter = 0 if len(tr["iteration"]) == 0 else tr["iteration"][-1]
        if self.verbose:
            print(f"Running {niter} active learning iterations using {self.algorithm}...")
        it = range(1, niter + 1)
        if show_progress:
            import tqdm
            it = tqdm.tqdm(it)
        for ii in it:
            attempts, success = 0, False
            while not success:
                _theta_prop, _y_prop, opt_timing = self.find_next_point(nopt=nopt, optimizer_kwargs=optimizer_kwargs)
                if _theta_prop is None:
                    attempts += 1
                    if attempts >= max_attempts:
                        raise RuntimeError(f"Failed to find a valid training point after {max_attempts} attempts.")
                    continue
                fitted = self._append_gp(_theta_prop, _y_prop)
                if fitted is None:
                    fitted = self._fit_gp(_theta=_theta_prop, _y=_y_prop,
                                          hyperparameters=self.gp.get_parameter_vector())
                self.gp, fit_gp_timing = fitted
                success = True
            self._theta, self._y = _theta_prop, _y_prop
            if (ii + first_iter) % self.gp_opt_freq == 0:
                kw = self.opt_gp_kwargs.copy()
                kw["multi_proc"] = allow_opt_multiproc
                self.gp, _ = self._opt_gp(**kw)
                tr["gp_hyperparameter_opt_iteration"].append(ii + first_iter)
                if save_progress:
                    self.save()
            _yp = self.gp.predict(_y_prop, _theta_prop, return_cov=False, return_var=False)
            yp = self.y_scaler.inverse_transform(_yp.reshape(-1, 1)).flatten()
            training_mse = np.mean((self.y() - yp) ** 2)
            test_mse = np.nan
            if self.ntest > 0:
                _yt = self.gp.predict(self._y, self._theta_test, return_cov=False, return_var=False)
                yt = self.y_scaler.inverse_transform(_yt.reshape(-1, 1)).flatten()
                yt_true = self.y_scaler.inverse_transform(self._y_test.reshape(-1, 1)).flatten()
                test_mse = np.mean((yt_true - yt) ** 2)
            tr["iteration"].append(ii + first_iter)
            tr["gp_hyperparameters"].append(self.gp.get_parameter_vector())
            tr["training_mse"].append(training_mse)
            tr["test_mse"].append(test_mse)
            tr["training_scaled_mse"].append(training_mse / np.var(self.y()))
            tr["test_scaled_mse"].append(test_mse / np.var(self.y()))
            tr["gp_kl_divergence"].append(np.nan)
            tr["gp_train_time"].append(fit_gp_timing)
            tr["obj_fn_opt_time"].append(opt_timing)
            self.ntrain = len(self._theta)
            self.nactive = self.ntrain - self.ninit_train
        if self.cache:
            self.save()

    # -- samplers ------------------------------------------------------------------------------------
    def _lnlike_fn(self, _theta):
        """``lnlike_fn`` at a SCALED theta, returned in scaled y (alabi/core.py:407-422)."""
        theta = self.theta_scaler.inverse_transform(_theta).flatten()
        y = np.asarray(self.true_log_likelihood(theta)).reshape(-1, 1)
        return self.y_scaler.transform(y).flatten()

    def find_map(self, theta0=None, prior_fn=None, method="nelder-mead", nRestarts=15, options=None):
        """Not implemented in the reference either (alabi/core.py:2103-2105)."""
        raise NotImplementedError("Not implemented.")

    def lnprob(self, theta):
        """ln P = like_fn(theta) + prior_fn(theta) (alabi/core.py:2073-2100)."""
        if getattr(self, "like_fn_name", "surrogate") == "surrogate" and not hasattr(self, "gp"):
            raise NameError("GP has not been trained")
        if not hasattr(self, "prior_fn"):
            raise NameError("prior_fn has not been specified")
        if not hasattr(self, "like_fn"):
            self.like_fn = self.surrogate_log_likelihood
        theta = np.asarray(theta).reshape(1, -1)
        return self.like_fn(theta) + self.prior_fn(theta)

    def run_emcee(self, like_fn=None, prior_fn=None, nwalkers=None, nsteps=int(5e4), sampler_kwargs={},
                  run_kwargs={}, opt_init=False, multi_proc=True, prior_fn_comment=None, burn=None, thin=None,
                  samples_file=None, min_ess=int(1e4)):
        """Ensemble MCMC on the surrogate posterior.  With the default likelihood
        (the surrogate) and prior (uniform box) every step runs on the device
        (K5).  ``prior_fn`` may also be a ``functools.partial`` of ``ut.lnprior_uniform``
        or ``ut.lnprior_normal`` (box times independent normals): both are evaluated inside
        the kernel.  Other Python ``like_fn`` / ``prior_fn`` callables cannot run inside a
        CUDA kernel and are rejected."""
        if like_fn is not None and like_fn not in (self.surrogate_log_likelihood, "surrogate"):
            raise NotImplementedError("alabi_b200.run_emcee samples the GP surrogate on the GPU; a custom Python "
                                      "like_fn is outside the accelerated path")
        self.like_fn_name, self.like_fn = "surrogate", self.surrogate_log_likelihood
        if prior_fn is None:
            pbounds, pdata = self.bounds, None
            self.prior_fn = partial(ut.lnprior_uniform, bounds=self.bounds)
            self.prior_fn_comment = f"Default uniform prior. \nPrior function: ut.prior_fn_uniform\n\twith bounds {self.bounds}"
        else:
            pbounds, pdata = self._device_prior(prior_fn)
            self.prior_fn = prior_fn
            self.prior_fn_comment = prior_fn_comment if prior_fn_comment is not None else \
                f"User defined prior.Prior function: {prior_fn.func.__name__}"
        self.nwalkers = int(10 * self.ndim) if nwalkers is None else int(nwalkers)
        self.nsteps = int(nsteps)
        p0 = ut.prior_sampler(nsample=self.nwalkers, bounds=self.bounds, sampler="uniform", random_state=None)
        lp = self._device_log_prob(-1, bounds=pbounds, prior_data=pdata)
        if self.verbose:
            print(f"Running emcee-compatible GPU sampler with {self.nwalkers} walkers for {self.nsteps} steps...")
        all_chains, all_times, accumulated, run_number = [], [], 0, 1
        while True:
            t0 = time.time()
            self.emcee_sampler = EnsembleSampler(self.nwalkers, self.ndim, lp, **sampler_kwargs)
            self.emcee_sampler.run_mcmc(p0, self.nsteps, progress=True, **run_kwargs)
            all_times.append(time.time() - t0)
            iburn, ithin = mcmc_utils.estimate_burnin(self.emcee_sampler, verbose=self.verbose)
            samples_full = self.emcee_sampler.get_chain()
            cur_burn = burn if burn is not None else iburn
            cur_thin = thin if thin is not None else ithin
            cur = self.emcee_sampler.get_chain(discard=cur_burn, thin=cur_thin, flat=True)
            all_chains.append(cur)
            accumulated += cur.shape[0]
            if min_ess > 0 and self.verbose:
                print(f"Run {run_number} complete: {cur.shape[0]} samples (total {accumulated})")
            if accumulated >= min_ess:
                break
            run_number += 1
            if run_number > 10:
                print(f"WARNING: Reached maximum of 10 runs, stopping with {accumulated} samples")
                break
            p0 = self.emcee_sampler.get_last_sample().coords
        self.emcee_samples = np.vstack(all_chains) if len(all_chains) > 1 else all_chains[0]
        self.emcee_samples_full = samples_full
        self.iburn, self.ithin, self.burn, self.thin = iburn, ithin, cur_burn, cur_thin
        self.emcee_runtime = sum(all_times)
        self.emcee_samples_gp = self.emcee_samples
        self.acc_frac = np.mean(self.emcee_sampler.acceptance_fraction)
        self.autcorr_time = np.mean(self.emcee_sampler.get_autocorr_time(tol=0))
        if self.verbose:
            print(f"Total samples: {self.emcee_samples.shape[0]}")
            print("Mean acceptance fraction: {0:.3f}".format(self.acc_frac))
            print("Mean autocorrelation time: {0:.3f} steps".format(self.autcorr_time))
        self.emcee_run = True
        if self.cache:
            try:
                self.save()
            except Exception:  # noqa: BLE001
                pass
        cur_iter = 0 if len(self.training_results["iteration"]) == 0 else self.training_results["iteration"][-1]
        fname = f"{self.savedir}/{samples_file}" if samples_file is not None else \
            f"{self.savedir}/emcee_samples_final_{self.like_fn_name}_iter_{cur_iter}.npz"
        print(f"Saving final emcee samples to {fname} ...")
        np.savez(fname, samples=self.emcee_samples)

    def _builtin_nested_runner(self, ns, batch_like, lp, mode, skw, rkw, save_iter):
        """Closure running one built-in nested-sampling run (see run_dynesty)."""
        allowed_s = {"nlive", "walks", "slices", "nbatch", "rstate", "seed", "bound", "sample", "pool", "queue_size",
                     "use_pool"}
        allowed_r = {"dlogz", "dlogz_init", "maxiter", "maxcall", "wt_kwargs", "stop_kwargs", "nlive_init", "nlive_batch",
                     "maxbatch", "n_effective", "print_progress"}
        bad = (set(skw) - allowed_s) | (set(rkw) - allowed_r)
        if bad:
            raise TypeError(f"run_dynesty (built-in sampler): unsupported keyword(s) {sorted(bad)}; sampler_kwargs "
                            f"{sorted(allowed_s)}, run_kwargs {sorted(allowed_r)}")
        sample = str(skw.get("sample", "auto")).lower()
        if sample not in ("auto", "rwalk", "rslice"):
            raise NotImplementedError(f"sample={skw['sample']!r}: the built-in sampler proposes by constrained random "
                                      "walks (dynesty's 'rwalk', also for 'auto') or by random-direction slice "
                                      "sampling ('rslice')")
        sample = "rslice" if sample == "rslice" else "rwalk"
        if str(skw.get("bound", "multi")).lower() not in ("multi", "single", "none"):
            raise NotImplementedError(f"bound={skw['bound']!r} is not available in the built-in sampler")
        nlive = int(skw.get("nlive", 50 * self.ndim))
        walks = int(skw.get("walks", 25))
        slices = int(skw.get("slices", 5))
        seed = skw.get("seed", skw.get("rstate"))
        if seed is not None and not isinstance(seed, (int, np.integer)):
            seed = int(np.random.default_rng(seed).integers(2 ** 62))
        pfrac = float(dict(rkw.get("wt_kwargs", {"pfrac": 1.0})).get("pfrac", 1.0))
        maxiter = int(rkw.get("maxiter", int(5e4)))
        builtin = ns._builtin_transform(self.prior_transform)

        def run_one(run_number):
            rseed = None if seed is None else int(seed) + 7919 * (run_number - 1)
            if lp is not None and builtin is not None:
                kind, pbounds, pdata = builtin
                walker = ns.DeviceWalker(lp, pbounds, prior_data=pdata if kind == "normal" else None, seed=rseed)
            else:
                walker = ns.HostWalker(batch_like, self.prior_transform, self.ndim, rng=np.random.default_rng(rseed))
            ds = ns.BatchedNestedSampler(walker, self.ndim, nlive=nlive, walks=walks, nbatch=skw.get("nbatch"),
                                         rstate=None if rseed is None else rseed + 1, sample=sample, slices=slices)
            if save_iter is not None:
                path = os.path.join(self.savedir, f"dynesty_sampler_{self.like_fn_name}_run{run_number}.pkl")
                ds.checkpoint, ds.checkpoint_every = ns.save_checkpoint(path), int(save_iter)
            if mode == "dynamic":
                res = ds.run_dynamic(dlogz_init=rkw.get("dlogz_init", 0.5), nlive_init=rkw.get("nlive_init"),
                                     nlive_batch=rkw.get("nlive_batch"), maxiter=maxiter, maxcall=rkw.get("maxcall"),
                                     maxbatch=rkw.get("maxbatch"), n_effective=rkw.get("n_effective"), pfrac=pfrac,
                                     print_progress=bool(rkw.get("print_progress", False)))
            else:
                res = ds.run_nested(dlogz=rkw.get("dlogz", 0.01), maxiter=maxiter, maxcall=rkw.get("maxcall"),
                                    print_progress=bool(rkw.get("print_progress", False)))
            return ds, res
        return run_one

    def _dynesty_runner(self, ns, batch_like, mode, skw, rkw, save_iter):
        """Closure running one real-dynesty run with the reference's defaults (alabi/core.py:2600-2700);
        the likelihood is reached through a BatchPool, so a dynesty iteration of ``queue_size``
        proposals is one batched predict."""
        import dynesty
        like = ns.BatchLikelihood(batch_like)
        for key, val in {"bound": "multi", "nlive": 50 * self.ndim, "sample": "auto"}.items():
            skw.setdefault(key, val)
        qs = int(skw.pop("queue_size", 64))
        skw.pop("pool", None)
        skw.update(pool=ns.BatchPool(like, size=qs), queue_size=qs,
                   use_pool={"prior_transform": False, "loglikelihood": True, "propose_point": False, "update_bound": False})
        if mode == "dynamic":
            for key, val in {"wt_kwargs": {"pfrac": 1.0}, "stop_kwargs": {"pfrac": 1.0}, "maxiter": int(5e4), "dlogz_init": 0.5}.items():
                rkw.setdefault(key, val)
        else:
            rkw.setdefault("maxiter", int(5e4))
            rkw.pop("dlogz_init", None)
        cls = dynesty.DynamicNestedSampler if mode == "dynamic" else dynesty.NestedSampler

        def run_one(run_number):
            ds = cls(like, self.prior_transform, self.ndim, **skw)
            if save_iter is not None:
                last = 0
                while True:
                    ds.run_nested(maxiter=save_iter, **{k: v for k, v in rkw.items() if k != "maxiter"})
                    with open(os.path.join(self.savedir, f"dynesty_sampler_{self.like_fn_name}_run{run_number}.pkl"), "wb") as f:
                        pickle.dump(ds.results, f)
                    if ds.results.niter <= last:
                        break
                    last = ds.results.niter
            else:
                ds.run_nested(**rkw)
            return None, ds.results                      # the sampler holds the pool: keep the results only
        return run_one

    def run_dynesty(self, like_fn=None, prior_transform=None, mode="dynamic", sampler_kwargs={}, run_kwargs={},
                    multi_proc=False, save_iter=None, prior_transform_comment=None, samples_file=None,
                    min_ess=int(1e4)):
        """Nested sampling of the surrogate (or of a Python likelihood), alabi/core.py:2417-2787.

        * dynesty importable: exactly the reference's calls (``DynamicNestedSampler`` for
          ``mode="dynamic"``, ``NestedSampler`` for ``"static"``, the reference's default sampler /
          run kwargs), except that the surrogate likelihood is served through a ``pool``-shaped
          :class:`alabi_b200.nested.BatchPool`: the ``queue_size`` points dynesty proposes per
          iteration become ONE batched device predict (the reference re-factorises K for every
          single point, core.py:1430).
        * otherwise (this image: dynesty is not installable): the built-in
          :class:`alabi_b200.nested.BatchedNestedSampler` with the same two modes and result fields
          (``samples, logwt, logz, logzerr, niter``).  With the surrogate likelihood and one of the
          reference's prior transforms (``ut.prior_transform_uniform`` / ``_normal``, or None) every
          batch of constrained random walks is one kernel launch (``ab_nested_walk``, or
          ``ab_nested_rslice`` for random-direction slice sampling); a custom Python ``like_fn`` /
          ``prior_transform`` runs the same algorithms with host-side chains.
          ``sampler_kwargs``: nlive (50 ndim), walks (25), slices (5), nbatch, rstate / seed, bound,
          sample ("auto" = "rwalk", or "rslice"); ``run_kwargs``: dlogz, dlogz_init (0.5), maxiter (5e4), maxcall,
          wt_kwargs {"pfrac": 1.0}, nlive_init, nlive_batch, maxbatch, n_effective, print_progress;
          anything else raises.  ``save_iter`` pickles the dead points every that many iterations;
          ``multi_proc`` has no meaning here (the batch is the parallelism)."""
        from . import nested as ns
        if mode not in ("dynamic", "static"):
            raise ValueError(f"mode {mode} is not a valid option. Choose 'dynamic' or 'static'.")
        surrogate = like_fn is None or (isinstance(like_fn, str) and like_fn.lower() in ("surrogate", "gp", "surrogate_log_likelihood")) \
            or like_fn == self.surrogate_log_likelihood
        lp = None
        if surrogate:
            self.like_fn_name = "surrogate"
            lp = self._device_log_prob(-1)
            gp, yc = lp.gp, lp.y
            ts, to = lp.theta_scale, lp.theta_offset

            def batch_like(theta):
                ys = gp.predict(yc, np.atleast_2d(theta) * ts + to, return_cov=False)
                return self.y_scaler.inverse_transform(ys.reshape(-1, 1)).flatten()
            self.like_fn = self.surrogate_log_likelihood
        elif isinstance(like_fn, str):
            if like_fn.lower() not in ("true", "true_log_likelihood"):
                raise ValueError(f"Unknown string identifier for like_fn: '{like_fn}'. Valid options: 'surrogate', 'true', "
                                 "'gp', 'surrogate_log_likelihood', 'true_log_likelihood'")
            self.like_fn_name, self.like_fn = "true", self.true_log_likelihood
            batch_like = lambda theta: np.array([float(np.asarray(self.true_log_likelihood(t)).reshape(-1)[0])
                                                 for t in np.atleast_2d(theta)])
        elif callable(like_fn):
            self.like_fn_name = "true" if like_fn == self.true_log_likelihood else "custom"
            self.like_fn = like_fn
            batch_like = lambda theta: np.array([float(np.asarray(like_fn(t)).reshape(-1)[0]) for t in np.atleast_2d(theta)])
        else:
            raise TypeError(f"like_fn must be None, a string, or a callable function. Received type: {type(like_fn)}")
        if prior_transform is None:
            self.prior_transform = partial(ut.prior_transform_uniform, bounds=self.bounds)
            self.prior_transform_comment = ("Default uniform prior transform. \nPrior function: ut.prior_transform_uniform\n"
                                            f"\twith bounds {self.bounds}")
        else:
            self.prior_transform = prior_transform
            self.prior_transform_comment = prior_transform_comment if prior_transform_comment is not None else \
                f"User defined prior transform.Prior function: {getattr(prior_transform, '__name__', 'unrecorded')}"
        t0 = time.time()
        skw = dict(sampler_kwargs)
        rkw = dict(run_kwargs)
        try:
            import dynesty                                # noqa: F401
            have_dynesty = not skw.pop("builtin", False)
        except ImportError:
            have_dynesty = False
            skw.pop("builtin", None)

        if have_dynesty:
            run_one = self._dynesty_runner(ns, batch_like, mode, skw, rkw, save_iter)
        else:
            run_one = self._builtin_nested_runner(ns, batch_like, lp, mode, skw, rkw, save_iter)
        all_samples, all_logz, accumulated, run_number = [], [], 0, 1
        while True:
            ds, res = run_one(run_number)
            w = np.exp(res.logwt - res.logz[-1])
            eq = ns.resample_equal(res.samples, w)
            all_samples.append(eq)
            all_logz.append(res.logz[-1])
            accumulated += eq.shape[0]
            if self.verbose:
                print(f"Run {run_number} complete: {eq.shape[0]} samples, logZ = {res.logz[-1]:.3f}")
            if accumulated >= min_ess or run_number >= 10:
                if accumulated < min_ess:
                    print(f"WARNING: Reached maximum of 10 runs, stopping with {accumulated} samples")
                break
            run_number += 1
        self.dynesty_samples = np.vstack(all_samples) if len(all_samples) > 1 else all_samples[0]
        self.dynesty_logz = max(all_logz)
        self.dynesty_sampler, self.dynesty_results = ds, res
        self.dynesty_logz_err = res.logzerr[-1]
        if self.like_fn_name == "true":
            self.dynesty_samples_true = self.dynesty_samples
        elif self.like_fn_name == "surrogate":
            self.dynesty_samples_surrogate = self.dynesty_samples
        self.dynesty_run = True
        self.dynesty_runtime = time.time() - t0
        if self.cache:
            try:
                self.save()
            except Exception:  # noqa: BLE001
                pass
        cur_iter = 0 if len(self.training_results["iteration"]) == 0 else self.training_results["iteration"][-1]
        fname = f"{self.savedir}/{samples_file}" if samples_file is not None else \
            f"{self.savedir}/dynesty_samples_final_{self.like_fn_name}_iter_{cur_iter}.npz"
        print(f"Saved dynesty samples to {fname}")
        np.savez(fname, samples=self.dynesty_samples)
