"""GPU Gaussian process with the george.GP protocol alabi consumes (SURVEY 8b).

Mirrors ``george.GP(kernel, fit_mean, mean, white_noise, fit_white_noise)``
(alabi/gp_utils.py:233, alabi/core.py:1141) and its ``compute / recompute /
predict / log_likelihood / grad_log_likelihood / set|get_parameter_vector /
get_parameter_names / get_parameter_dict`` methods, the ``_x / _y / _alpha``
attributes and ``solver.get_inverse()`` (alabi/utility.py:577-610).  All
arithmetic runs in libalabi_b200.so through ``alabi_b200._lib`` (ctypes);
torch only carries device buffers.  No CPU fallback exists.
"""
import copy
import ctypes

import numpy as np

from . import _lib
from .kernels import Kernel, Product

__all__ = ["GP", "LinAlgError"]

LinAlgError = np.linalg.LinAlgError
TINY = 1.25e-12


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise _lib.AlabiB200Error("alabi_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


class _Handle:
    """Owns one ``ab_gp*``; freed with the object."""

    def __init__(self, device=None):
        torch = _torch()
        self.lib = _lib.load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.stream = torch.cuda.current_stream(self.device)
        h = ctypes.c_void_p()
        _lib.check(self.lib.ab_gp_create(ctypes.byref(h), self.device, ctypes.c_void_p(self.stream.cuda_stream)),
                   "ab_gp_create")
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.ab_gp_destroy(self.h)
                self.h = None
        except Exception:
            pass


class _Solver:
    """``gp.solver`` facade (george BasicSolver attributes alabi touches)."""

    def __init__(self, gp):
        self._gp = gp

    @property
    def log_determinant(self):
        gp = self._gp
        out = ctypes.c_double()
        _lib.check(gp._hd.lib.ab_gp_log_determinant(gp._hd.h, ctypes.byref(out)), "ab_gp_log_determinant")
        return out.value

    @property
    def computed(self):
        return self._gp.computed

    def get_inverse(self):
        """Dense K^-1 as a NumPy array (alabi/utility.py:610)."""
        gp = self._gp
        torch = _torch()
        n = len(gp._x)
        out = torch.empty((n, n), dtype=torch.float64, device=f"cuda:{gp._hd.device}")
        _lib.check(gp._hd.lib.ab_gp_get_inverse(gp._hd.h, _lib.ptr(out)), "ab_gp_get_inverse")
        return out.cpu().numpy()

    def apply_inverse(self, y):
        return self.get_inverse() @ np.asarray(y, dtype=np.float64)


class GP:
    cv_workspace_limit_bytes = 16 << 30      # device scratch ceiling of one cv_batch call

    def __init__(self, kernel=None, fit_kernel=True, mean=None, fit_mean=None, white_noise=None,
                 fit_white_noise=None, solver=None, device=None, **kwargs):
        if kernel is None or not isinstance(kernel, Kernel):
            raise ValueError("alabi_b200.GP needs an alabi_b200.kernels kernel")
        # own copy: `kernel * var(y)` keeps a reference to the caller's kernel object, and several
        # GPs built from one SurrogateModel.kernel must not see each other's hyper-parameters
        self.kernel = copy.deepcopy(kernel)
        self.mean_value = 0.0 if mean is None else float(mean)
        self.white_noise_value = np.log(TINY) if white_noise is None else float(white_noise)
        self.fit_mean = bool(fit_mean) if fit_mean is not None else False
        self.fit_white_noise = bool(fit_white_noise) if fit_white_noise is not None else False
        self.fit_kernel = bool(fit_kernel)
        self._device = device
        self._hd = None
        self._x = None
        self._yerr2 = 0.0
        self._y = None
        self._alpha_np = None
        self._y_dev = None
        self.computed = False
        self._inputs_pushed = False
        self._kernel_pushed = False
        self._targets_pushed = False
        self._factor_key = None          # hyper-parameters the device factor was computed for
        self.solver = _Solver(self)

    # -- pickling / copying: drop device state, rebuild lazily -----------------------
    def __getstate__(self):
        st = self.__dict__.copy()
        for k in ("_hd", "_y_dev", "solver"):
            st[k] = None
        st.update(computed=False, _inputs_pushed=False, _kernel_pushed=False, _targets_pushed=False, _factor_key=None)
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self.solver = _Solver(self)

    def __copy__(self):
        new = GP.__new__(GP)
        st = self.__getstate__()
        st["kernel"] = copy.deepcopy(self.kernel)      # a copy never shares hyper-parameters
        new.__setstate__(st)
        return new

    # -- george "mean" / "white_noise" views -----------------------------------------
    @property
    def mean(self):
        return self.mean_value

    @property
    def white_noise(self):
        return self.white_noise_value

    def __len__(self):
        return len(self.get_parameter_vector())

    # -- parameter protocol ----------------------------------------------------------
    def get_parameter_names(self, include_frozen=False):
        names = []
        if self.fit_mean or include_frozen:
            names.append("mean:value")
        if self.fit_white_noise or include_frozen:
            names.append("white_noise:value")
        if self.fit_kernel or include_frozen:
            names += ["kernel:" + n for n in self.kernel.get_parameter_names()]
        return tuple(names)

    def get_parameter_vector(self, include_frozen=False):
        v = []
        if self.fit_mean or include_frozen:
            v.append(self.mean_value)
        if self.fit_white_noise or include_frozen:
            v.append(self.white_noise_value)
        if self.fit_kernel or include_frozen:
            v += list(self.kernel.get_parameter_vector())
        return np.array(v, dtype=np.float64)

    def set_parameter_vector(self, vector, include_frozen=False):
        v = np.atleast_1d(np.asarray(vector, dtype=np.float64))
        cur = self.get_parameter_vector(include_frozen)
        if len(v) != len(cur):
            raise ValueError("dimension mismatch")
        n = 0
        if self.fit_mean or include_frozen:
            self.mean_value = float(v[n]); n += 1
        if self.fit_white_noise or include_frozen:
            self.white_noise_value = float(v[n]); n += 1
        if self.fit_kernel or include_frozen:
            self.kernel.set_parameter_vector(v[n:])
        # george marks the model dirty on every set; here the factor is kept only when the values
        # now in force are exactly the ones it was computed for (compared against what was pushed
        # to the device, never against a live object another GP could have modified)
        if not (self.computed and self._factor_key is not None and self._spec_key() == self._factor_key):
            self._mark_dirty()

    def _spec_key(self):
        kid, amp, log_M = self.kernel.spec()
        return (int(kid), float(amp), np.asarray(log_M, dtype=np.float64).tobytes(), _log_alpha(self.kernel),
                float(self.mean_value), float(self.white_noise_value), float(self._yerr2))

    def get_parameter_dict(self, include_frozen=False):
        return dict(zip(self.get_parameter_names(include_frozen), self.get_parameter_vector(include_frozen)))

    def get_parameter(self, name):
        return self.get_parameter_dict(include_frozen=True)[name]

    def set_parameter(self, name, value):
        names = list(self.get_parameter_names(include_frozen=True))
        v = self.get_parameter_vector(include_frozen=True)
        v[names.index(name)] = value
        self.set_parameter_vector(v, include_frozen=True)

    def get_parameter_bounds(self, include_frozen=False):
        b = []
        if self.fit_mean or include_frozen:
            b.append((None, None))
        if self.fit_white_noise or include_frozen:
            b.append((None, None))
        if self.fit_kernel or include_frozen:
            b += list(self.kernel.get_parameter_bounds())
        return b

    def _mark_dirty(self):
        self.computed = False
        self._kernel_pushed = False
        self._targets_pushed = False
        self._alpha_np = None
        self._factor_key = None

    @property
    def dirty(self):
        return not self.computed

    # -- device plumbing -------------------------------------------------------------------
    def _handle(self):
        if self._hd is None:
            self._hd = _Handle(self._device)
            self._inputs_pushed = self._kernel_pushed = self._targets_pushed = False
        return self._hd

    def _dev(self, a):
        torch = _torch()
        hd = self._handle()
        if isinstance(a, torch.Tensor):
            return a.to(device=f"cuda:{hd.device}", dtype=torch.float64).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(f"cuda:{hd.device}")

    def _push(self):
        hd = self._handle()
        if not self._inputs_pushed:
            xd = self._dev(self._x)
            _lib.check(hd.lib.ab_gp_set_inputs(hd.h, _lib.ptr(xd), self._x.shape[0], self._x.shape[1]),
                       "ab_gp_set_inputs")
            hd.stream.synchronize()           # xd may be freed after this call
            self._inputs_pushed = True
            self._kernel_pushed = False
        if not self._kernel_pushed:
            _set_kernel(hd, self.kernel, self.mean_value, self.white_noise_value, float(self._yerr2))
            self._kernel_pushed = True
            self._targets_pushed = False

    def parse_samples(self, t):
        t = np.atleast_1d(np.asarray(t, dtype=np.float64))
        if t.ndim == 1:
            t = np.atleast_2d(t).T
        if t.ndim != 2 or t.shape[1] != self.kernel.ndim:
            raise ValueError("Dimension mismatch")
        return np.ascontiguousarray(t)

    # -- george API ----------------------------------------------------------------------------
    def compute(self, x, yerr=0.0, **kwargs):
        """Build K = amp k(x, x) + (yerr^2 + exp(white_noise)) I and factorise it
        (K1 + K2).  Raises ``numpy.linalg.LinAlgError`` if K is not SPD."""
        x = self.parse_samples(x)
        if self._x is None or x.shape != self._x.shape or not np.array_equal(x, self._x):
            self._x = x
            self._inputs_pushed = False
        self._yerr2 = float(yerr) ** 2
        self._mark_dirty()
        self._push()
        hd = self._hd
        rc = _lib.check(hd.lib.ab_gp_factor(hd.h), "ab_gp_factor")
        if rc > 0:
            raise LinAlgError(f"{rc}-th leading minor of the covariance matrix is not positive definite")
        self.computed = True
        self._factor_key = self._spec_key()
        return self

    def append_point(self, x_new):
        """Append ONE training point to a computed model in O(N^2) (bordered Cholesky
        update, ``ab_gp_append_point``) — the same factor, up to rounding, as
        ``compute(vstack(x, x_new))``, which is what the reference does after every
        active-learning step (alabi/core.py:1780).  Targets are reset: pass the new
        ``y`` to the next ``predict`` / ``log_likelihood`` call."""
        if not self.computed or self._x is None:
            raise RuntimeError("You need to compute the model first")
        x_new = np.ascontiguousarray(np.asarray(x_new, dtype=np.float64).reshape(-1))
        if x_new.shape[0] != self.kernel.ndim:
            raise ValueError("Dimension mismatch")
        hd = self._hd
        xd = self._dev(x_new)
        rc = _lib.check(hd.lib.ab_gp_append_point(hd.h, _lib.ptr(xd)), "ab_gp_append_point")
        hd.stream.synchronize()
        self._x = np.vstack([self._x, x_new[None, :]])
        self._targets_pushed = False
        self._alpha_np = None
        self._y = None
        if rc > 0:
            self.computed = False
            raise LinAlgError(f"{rc}-th leading minor of the covariance matrix is not positive definite")
        return self

    def recompute(self, quiet=False, **kwargs):
        if not self.computed:
            if self._x is None:
                raise RuntimeError("You need to compute the model first")
            try:
                self.compute(self._x, np.sqrt(self._yerr2), **kwargs)
            except (ValueError, LinAlgError):
                if quiet:
                    return False
                raise
        return True

    def _set_targets(self, y):
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
        if len(y) != len(self._x):
            raise ValueError("Dimension mismatch")
        if self._targets_pushed and self._y is not None and np.array_equal(y, self._y):
            return
        hd = self._hd
        self._y = y
        self._y_dev = self._dev(y)
        _lib.check(hd.lib.ab_gp_set_targets(hd.h, _lib.ptr(self._y_dev)), "ab_gp_set_targets")
        self._targets_pushed = True
        self._alpha_np = None

    @property
    def _alpha(self):
        """alpha = K^-1 (y - mean) as NumPy (alabi/utility.py:581)."""
        if self._alpha_np is None and self._targets_pushed:
            torch = _torch()
            hd = self._hd
            out = torch.empty(len(self._x), dtype=torch.float64, device=f"cuda:{hd.device}")
            _lib.check(hd.lib.ab_gp_get_alpha(hd.h, _lib.ptr(out)), "ab_gp_get_alpha")
            self._alpha_np = out.cpu().numpy()
        return self._alpha_np

    def log_likelihood(self, y, quiet=False):
        if not self.recompute(quiet=quiet):
            return -np.inf
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
        if len(y) != len(self._x):
            raise ValueError("Dimension mismatch")
        hd = self._hd
        self._y = y
        self._y_dev = self._dev(y)
        out = ctypes.c_double()
        _lib.check(hd.lib.ab_gp_log_likelihood(hd.h, _lib.ptr(self._y_dev), ctypes.byref(out)), "ab_gp_log_likelihood")
        self._targets_pushed = True
        self._alpha_np = None
        ll = out.value
        return ll if np.isfinite(ll) else -np.inf

    lnlikelihood = log_likelihood

    def nll(self, vector, y, quiet=True):
        self.set_parameter_vector(vector)
        return -self.log_likelihood(y, quiet=quiet)

    def grad_log_likelihood(self, y, quiet=False):
        npar = len(self.get_parameter_vector())
        if not self.recompute(quiet=quiet):
            return np.zeros(npar)
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
        hd = self._hd
        d = self._x.shape[1]
        nx = 1 if self.kernel.kernel_id == RQ_KERNEL_ID else 0   # the log_alpha entry
        out = (ctypes.c_double * (d + 3 + nx))()
        if self._targets_pushed and self._y is not None and np.array_equal(y, self._y):
            yp = None                    # alpha of the preceding log_likelihood / predict is still valid
        else:
            self._y = y
            self._y_dev = self._dev(y)
            yp = _lib.ptr(self._y_dev)
            self._alpha_np = None
        _lib.check(hd.lib.ab_gp_grad_log_likelihood(hd.h, yp, out), "ab_gp_grad_log_likelihood")
        self._targets_pushed = True
        full = np.array(out[:], dtype=np.float64)
        g = []
        if self.fit_mean:
            g.append(full[0])
        if self.fit_white_noise:
            g.append(full[1])
        if self.fit_kernel:
            if isinstance(self.kernel, Product):
                g.append(full[2])
            if nx:
                g.append(full[3])
            gm = full[3 + nx:3 + nx + d]
            g += [gm.sum()] if getattr(self.kernel if not isinstance(self.kernel, Product) else self.kernel.k2,
                                       "isotropic", False) else list(gm)
        return np.array(g, dtype=np.float64)

    grad_lnlikelihood = grad_log_likelihood

    def grad_nll(self, vector, y, quiet=True):
        self.set_parameter_vector(vector)
        return -self.grad_log_likelihood(y, quiet=quiet)

    def predict(self, y, t, return_cov=True, return_var=False, cache=True, kernel=None):
        """Predictive mean at ``t`` and, as in george, the full predictive covariance
        (``return_cov=True``, the default: ``(mu, cov)``, cov = K(t, t) - K(t, x) K^-1 K(x, t)
        without white noise) or the variance (``return_var=True``, which takes precedence:
        ``(mu, var)``).  ``t`` may be a NumPy array (host buffers, copies included) or a CUDA
        torch tensor (device buffers in, torch tensors out).  ``mu`` has the same bits in every
        mode, ``diag(cov)`` the bits of ``var``."""
        self.recompute()
        self._set_targets(y)
        hd = self._hd
        want_var = bool(return_var)
        want_cov = bool(return_cov) and not want_var
        try:
            import torch
            is_dev = isinstance(t, torch.Tensor) and t.is_cuda
        except ImportError:
            is_dev = False
        if want_cov:
            torch = _torch()
            tq = (t.reshape(-1, self.kernel.ndim).to(dtype=torch.float64).contiguous() if is_dev
                  else self._dev(self.parse_samples(t)))
            mu, cov = self._predict_cov_dev(tq)
            if is_dev:
                return mu, cov
            return mu.cpu().numpy(), cov.cpu().numpy()
        if is_dev:
            tq = t.reshape(-1, self.kernel.ndim).to(dtype=torch.float64).contiguous()
            m = tq.shape[0]
            mu = torch.empty(m, dtype=torch.float64, device=tq.device)
            var = torch.empty(m, dtype=torch.float64, device=tq.device) if want_var else None
            if m > 0:
                _lib.check(hd.lib.ab_gp_predict(hd.h, _lib.ptr(tq), m, _lib.ptr(mu), _lib.ptr(var)), "ab_gp_predict")
            return (mu, var) if want_var else mu
        xs = self.parse_samples(t)
        m = xs.shape[0]
        if m == 0:
            e = np.empty(0, dtype=np.float64)
            return (e, e.copy()) if want_var else e
        mu = np.empty(m, dtype=np.float64)
        var = np.empty(m, dtype=np.float64) if want_var else None
        _lib.check(hd.lib.ab_gp_predict_host(hd.h, _lib.ptr(xs), m, _lib.ptr(mu), _lib.ptr(var)), "ab_gp_predict_host")
        return (mu, var) if want_var else mu

    def _predict_cov_dev(self, tq):
        """(mu, cov) as device tensors for the device query block ``tq`` (m x d); targets set."""
        torch = _torch()
        hd = self._hd
        m = tq.shape[0]
        mu = torch.empty(m, dtype=torch.float64, device=tq.device)
        cov = torch.empty((m, m), dtype=torch.float64, device=tq.device)
        if m > 0:
            _check_alloc(hd.lib.ab_gp_predict_cov(hd.h, _lib.ptr(tq), m, _lib.ptr(mu), _lib.ptr(cov), m),
                         "ab_gp_predict_cov", 16 * hd.lib.ab_gp_padded_size(hd.h) * ((m + 255) // 256 * 256))
        return mu, cov

    # -- draws (george GP.sample_conditional / GP.sample) ----------------------------------------------
    def sample_conditional(self, y, t, size=1, seed=None, jitter=None):
        """Draws from the GP posterior at ``t`` (george's ``sample_conditional``): returns
        ``(size, M)``, or ``(M,)`` when ``size == 1``.  The covariance stays on the device
        (``ab_gp_predict_cov`` then ``ab_mvn_sample``).  ``seed=None`` takes a seed from NumPy's
        global stream, so ``np.random.seed`` makes runs reproducible; with the same seed the
        first k draws of ``size=n`` equal the draws of ``size=k``.  ``jitter``: see ``sample``."""
        torch = _torch()
        self.recompute()
        self._set_targets(y)
        is_dev = isinstance(t, torch.Tensor) and t.is_cuda
        tq = (t.reshape(-1, self.kernel.ndim).to(dtype=torch.float64).contiguous() if is_dev
              else self._dev(self.parse_samples(t)))
        mu, cov = self._predict_cov_dev(tq)
        out = _mvn_draw(self._hd, cov, mu, size, seed, jitter, self.kernel.spec()[1])
        return _draw_result(out, size, is_dev)

    def sample(self, t=None, size=1, seed=None, jitter=None):
        """Draws from the GP prior (george's ``sample``): at ``t``, N(mean, amp k(t, t));
        with ``t=None`` at the training inputs from the full covariance K of ``compute``, white
        noise and yerr^2 included (one more factorisation of the N x N matrix).  Returns
        ``(size, M)``, or ``(M,)`` when ``size == 1``.

        george draws through NumPy's SVD, which accepts a semi-definite covariance; a Cholesky
        does not.  ``jitter=None`` therefore tries delta = 0, 1e-12, 1e-10, 1e-8 and 1e-6 times the
        kernel amplitude on the diagonal, warns (RuntimeWarning) when delta > 0 was needed and
        raises ``LinAlgError`` after the last step; a float uses exactly that jitter."""
        torch = _torch()
        amp = self.kernel.spec()[1]
        if t is None:
            if self._x is None:
                raise RuntimeError("You need to compute the model first")
            self.recompute()
            hd = self._hd
            n = self._x.shape[0]
            dev = f"cuda:{hd.device}"
            cov = torch.empty((n, n), dtype=torch.float64, device=dev)
            _lib.check(hd.lib.ab_gp_build_cov(hd.h, _lib.ptr(cov), 1), "ab_gp_build_cov")
            mean = torch.full((n,), float(self.mean_value), dtype=torch.float64, device=dev)
            return _draw_result(_mvn_draw(hd, cov, mean, size, seed, jitter, amp), size, False)
        is_dev = isinstance(t, torch.Tensor) and t.is_cuda
        if self._x is not None:
            self._push()
            hd = self._hd
        else:
            hd = _scratch_handle(self.kernel, self.parse_samples(t)[:1])
        tq = (t.reshape(-1, self.kernel.ndim).to(dtype=torch.float64).contiguous() if is_dev
              else torch.from_numpy(self.parse_samples(t)).to(f"cuda:{hd.device}"))
        m = tq.shape[0]
        cov = torch.empty((m, m), dtype=torch.float64, device=tq.device)
        if m > 0:
            _lib.check(hd.lib.ab_gp_cross_cov(hd.h, _lib.ptr(tq), m, _lib.ptr(tq), m, _lib.ptr(cov)), "ab_gp_cross_cov")
        mean = torch.full((m,), float(self.mean_value), dtype=torch.float64, device=tq.device)
        return _draw_result(_mvn_draw(hd, cov, mean, size, seed, jitter, amp), size, is_dev)

    def predict_grad(self, y, t):
        """(mu, var, d mu / dx, d var / dx) at the query points ``t`` (M x d); the
        gradients are M x d, w.r.t. the query coordinates (``ab_gp_predict_grad``).
        Analytic replacement for ``grad_gp_mean_prediction`` /
        ``grad_gp_var_prediction`` (alabi/utility.py:558-621)."""
        torch = _torch()
        self.recompute()
        self._set_targets(y)
        hd = self._hd
        tq = self._dev(self.parse_samples(t))
        m, d = tq.shape
        dev = tq.device
        # one device block for the four results, one copy back (the polish calls this per point)
        out = torch.empty(m * (2 + 2 * d), dtype=torch.float64, device=dev)
        mu, var = out[:m], out[m:2 * m]
        dmu, dvar = out[2 * m:2 * m + m * d], out[2 * m + m * d:]
        if m > 0:
            _lib.check(hd.lib.ab_gp_predict_grad(hd.h, _lib.ptr(tq), m, _lib.ptr(mu), _lib.ptr(var), _lib.ptr(dmu),
                                                 _lib.ptr(dvar)), "ab_gp_predict_grad")
        host = out.cpu().numpy()
        return (host[:m], host[m:2 * m], host[2 * m:2 * m + m * d].reshape(m, d), host[2 * m + m * d:].reshape(m, d))

    # -- batched acquisition (K4) -------------------------------------------------------------------
    def utility_argmin(self, y, candidates, bounds, algorithm="bape", y_best=0.0, zeta=0.01, return_values=False):
        """Evaluate an acquisition utility over a candidate batch and return
        (index of the smallest finite value, that value[, all values])."""
        torch = _torch()
        self.recompute()
        self._set_targets(y)
        hd = self._hd
        uid = {"bape": 0, "agp": 1, "jones": 2}[str(algorithm).lower()]
        cq = candidates if (isinstance(candidates, torch.Tensor) and candidates.is_cuda) else self._dev(self.parse_samples(candidates))
        cq = cq.reshape(-1, self.kernel.ndim).contiguous()
        m = cq.shape[0]
        b = np.ascontiguousarray(np.asarray(bounds, dtype=np.float64).reshape(-1))
        util = torch.empty(m, dtype=torch.float64, device=cq.device) if return_values else None
        if m == 0:                                   # empty candidate set: no finite utility
            return (-1, float("inf"), util) if return_values else (-1, float("inf"))
        idx, val = ctypes.c_int64(), ctypes.c_double()
        _lib.check(hd.lib.ab_gp_utility_argmin(hd.h, uid, _lib.ptr(cq), m, b.ctypes.data_as(_lib.c_double_p),
                                               float(y_best), float(zeta), _lib.ptr(util), ctypes.byref(idx),
                                               ctypes.byref(val)), "ab_gp_utility_argmin")
        return (idx.value, val.value, util) if return_values else (idx.value, val.value)

    # -- state export / import (multi-GPU broadcast of L and alpha) -------------------------------------
    def export_state(self):
        torch = _torch()
        hd = self._hd
        npad = hd.lib.ab_gp_padded_size(hd.h)
        L = torch.empty((npad, npad), dtype=torch.float64, device=f"cuda:{hd.device}")
        alpha = torch.empty(len(self._x), dtype=torch.float64, device=f"cuda:{hd.device}")
        _lib.check(hd.lib.ab_gp_get_factor(hd.h, _lib.ptr(L)), "ab_gp_get_factor")
        _lib.check(hd.lib.ab_gp_get_alpha(hd.h, _lib.ptr(alpha)), "ab_gp_get_alpha")
        return L, alpha

    def export_block_inverses(self):
        """Inverses of the diagonal blocks of L, (npad/128) x 128 x 128 (broadcast with L so
        that every replica derives L^-1 and variances with identical bits)."""
        torch = _torch()
        hd = self._hd
        npad = hd.lib.ab_gp_padded_size(hd.h)
        D = torch.empty((npad // 128, 128, 128), dtype=torch.float64, device=f"cuda:{hd.device}")
        _lib.check(hd.lib.ab_gp_get_block_inverses(hd.h, _lib.ptr(D)), "ab_gp_get_block_inverses")
        return D

    def import_state(self, x, y, L, alpha, yerr=0.0, Dinv=None):
        """Adopt a factor computed on another GPU (after a broadcast)."""
        self._x = self.parse_samples(x)
        self._yerr2 = float(yerr) ** 2
        self._inputs_pushed = False
        self._mark_dirty()
        self._push()
        hd = self._hd
        _lib.check(hd.lib.ab_gp_import_state_full(hd.h, _lib.ptr(L), _lib.ptr(Dinv), _lib.ptr(alpha)),
                   "ab_gp_import_state_full")
        hd.stream.synchronize()
        self._y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
        self.computed = True
        self._factor_key = self._spec_key()
        self._targets_pushed = True
        return self

    def get_matrix(self, x1, x2=None):
        return self.kernel.get_value(x1, x2)

    # -- batched k-fold cross-validation jobs (SURVEY 8f-1) ----------------------------------------------
    def cv_batch(self, x, y, candidates, folds, job_cand=None):
        """Factorise / score many (candidate, fold) jobs in one batched device call
        (``ab_gp_cv_batch``).  ``candidates`` (ncand, P) are hyper-vectors in this GP's
        ``get_parameter_vector()`` layout; ``folds`` is a list of (train_idx, val_idx) pairs, job b
        using candidate ``job_cand[b]`` (default: ``len(folds) // ncand`` consecutive folds per
        candidate).  Returns (preds, loglik, status): the predictive mean at each job's
        validation rows (list of arrays), the log-likelihood of its training rows and the
        Cholesky status (0 = ok, else the first non-positive pivot).  The GP's own state
        (hyper-parameters, factor) is not touched."""
        torch = _torch()
        hd = self._handle()
        x = self.parse_samples(x)
        y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
        cands = np.atleast_2d(np.asarray(candidates, dtype=np.float64))
        n, d = x.shape
        ncand, njobs = len(cands), len(folds)
        if job_cand is None:
            per = njobs // ncand
            if per * ncand != njobs:
                raise ValueError("folds must hold the same number of folds for every candidate (or pass job_cand)")
            job_cand = np.repeat(np.arange(ncand), per)
        job_cand = np.ascontiguousarray(job_cand, dtype=np.int32)
        # candidate vectors -> [mean, white_noise, amp, (log_alpha,) log_M...] through a scratch copy of this GP
        probe = self.__copy__()
        nx = 1 if self.kernel.kernel_id == RQ_KERNEL_ID else 0
        params = np.empty((ncand, 3 + nx + d))
        for c, v in enumerate(cands):
            probe.set_parameter_vector(v)
            kid, amp, log_M = probe.kernel.spec()
            params[c, 0], params[c, 1], params[c, 2] = probe.mean_value, probe.white_noise_value, amp
            if nx:
                params[c, 3] = probe.kernel.log_alpha
            params[c, 3 + nx:] = log_M
        ntr = np.array([len(f[0]) for f in folds], dtype=np.int32)
        nva = np.array([len(f[1]) for f in folds], dtype=np.int32)
        ld_tr, ld_va = int(ntr.max()), max(int(nva.max()), 1)
        tr = np.zeros((njobs, ld_tr), dtype=np.int32)
        va = np.zeros((njobs, ld_va), dtype=np.int32)
        for b, (a_, v_) in enumerate(folds):
            tr[b, :len(a_)] = a_
            va[b, :len(v_)] = v_
        dev = f"cuda:{hd.device}"
        xd, yd = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
        trd, vad = torch.from_numpy(tr).to(dev), torch.from_numpy(va).to(dev)
        pred = torch.empty((njobs, ld_va), dtype=torch.float64, device=dev)
        loglik = np.empty(njobs, dtype=np.float64)
        status = np.empty(njobs, dtype=np.int32)
        ci = ctypes.POINTER(ctypes.c_int)
        # scratch from torch's caching allocator (a cudaMalloc / cudaFree of gigabytes per stage costs
        # more than the factorisations): everything in one launch when it fits, else a capped block
        need = int(hd.lib.ab_gp_cv_workspace_bytes(ld_tr, d, ld_va, ncand, njobs))
        one = int(hd.lib.ab_gp_cv_workspace_bytes(ld_tr, d, ld_va, ncand, 1))
        free_b = torch.cuda.mem_get_info(hd.device)[0] + torch.cuda.memory_reserved(hd.device) - torch.cuda.memory_allocated(hd.device)
        cap = max(one, min(need, self.cv_workspace_limit_bytes, int(0.6 * free_b)))
        work = torch.empty(cap, dtype=torch.uint8, device=dev)
        _lib.check(hd.lib.ab_gp_cv_batch(hd.h, _lib.ptr(xd), _lib.ptr(yd), n, d, int(kid), ncand,
                                         params.ctypes.data_as(_lib.c_double_p), njobs, job_cand.ctypes.data_as(ci),
                                         ntr.ctypes.data_as(ci), nva.ctypes.data_as(ci), _lib.ptr(trd), ld_tr, _lib.ptr(vad),
                                         ld_va, _lib.ptr(pred), loglik.ctypes.data_as(_lib.c_double_p),
                                         status.ctypes.data_as(ci), _lib.ptr(work), cap), "ab_gp_cv_batch")
        ph = pred.cpu().numpy()
        return [ph[b, :nva[b]] for b in range(njobs)], loglik, status


RQ_KERNEL_ID = 3       # AB_KERNEL_RATQUAD: the kernel with a parameter of its own


def _log_alpha(kernel):
    return float(kernel.log_alpha) if kernel.kernel_id == RQ_KERNEL_ID else None


def _set_kernel(hd, kernel, mean, white_noise, yerr2):
    """Push ``kernel``'s hyper-parameters to the handle (ab_gp_set_kernel, or ab_gp_set_kernel_rq for
    the rational quadratic kernel)."""
    kid, amp, log_M = kernel.spec()
    lm = log_M.ctypes.data_as(_lib.c_double_p)
    if kid == RQ_KERNEL_ID:
        _lib.check(hd.lib.ab_gp_set_kernel_rq(hd.h, amp, float(kernel.log_alpha), lm, mean, white_noise, yerr2),
                   "ab_gp_set_kernel_rq")
    else:
        _lib.check(hd.lib.ab_gp_set_kernel(hd.h, kid, amp, lm, mean, white_noise, yerr2), "ab_gp_set_kernel")


JITTER_LADDER = (0.0, 1e-12, 1e-10, 1e-8, 1e-6)      # times the kernel amplitude


def _check_alloc(rc, what, nbytes):
    """_lib.check, with a failed device allocation (cudaErrorMemoryAllocation) as MemoryError."""
    if rc == -102:
        raise MemoryError(f"{what}: cannot allocate about {nbytes / 1e9:.2f} GB of device workspace "
                          f"({_lib.last_error()})")
    return _lib.check(rc, what)


def _mvn_draw(hd, cov, mean, size, seed, jitter, amp):
    """``size`` draws of N(mean, cov + delta I) as a (size, m) device tensor (ab_mvn_sample),
    delta from the jitter ladder or exactly ``jitter``."""
    import warnings
    torch = _torch()
    size = int(size)
    if size < 1:
        raise ValueError("size must be >= 1")
    m = cov.shape[0]
    out = torch.empty((size, m), dtype=torch.float64, device=cov.device)
    if m == 0:
        return out
    if seed is None:
        seed = int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    ladder = [float(d) * float(amp) for d in JITTER_LADDER] if jitter is None else [float(jitter)]
    info = ctypes.c_int(0)
    for delta in ladder:
        rc = _check_alloc(hd.lib.ab_mvn_sample(hd.h, _lib.ptr(cov), m, m, _lib.ptr(mean), delta, size, seed,
                                               _lib.ptr(out), ctypes.byref(info)),
                          "ab_mvn_sample", 8 * ((m + 127) // 128 * 128) * (2 * ((size + 127) // 128 * 128) + m))
        if rc == 0:
            if delta > 0.0 and jitter is None:
                warnings.warn(f"covariance is not positive definite; drew with jitter {delta:g} on its diagonal",
                              RuntimeWarning, stacklevel=3)
            return out
    raise LinAlgError(f"{info.value}-th leading minor of the covariance matrix is not positive definite "
                      f"(jitter {ladder[-1]:g})")


def _draw_result(out, size, is_dev):
    r = out[0] if int(size) == 1 else out
    return r if is_dev else r.cpu().numpy()


_SCRATCH_HANDLES = {}


def _scratch_handle(kernel, x):
    """The per-device scratch handle of _kernel_value with inputs ``x`` and ``kernel`` pushed."""
    torch = _torch()
    cur = torch.cuda.current_device()
    hd = _SCRATCH_HANDLES.get(cur)
    if hd is None or hd.stream != torch.cuda.current_stream(cur):
        hd = _SCRATCH_HANDLES[cur] = _Handle(cur)
    a = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(f"cuda:{hd.device}")
    _lib.check(hd.lib.ab_gp_set_inputs(hd.h, _lib.ptr(a), a.shape[0], a.shape[1]), "ab_gp_set_inputs")
    _set_kernel(hd, kernel, 0.0, -50.0, 0.0)
    hd.stream.synchronize()                  # `a` may be freed after this call
    return hd


def _kernel_value(kernel, x1, x2=None, diag=False):
    """kernel.get_value(x1[, x2]) on the GPU via a scratch handle."""
    torch = _torch()
    x1 = np.atleast_2d(np.asarray(x1, dtype=np.float64))
    if x1.shape[1] != kernel.ndim and x1.shape[0] == kernel.ndim and x1.shape[1] == 1:
        x1 = x1.T
    x2 = x1 if x2 is None else np.atleast_2d(np.asarray(x2, dtype=np.float64))
    kid, amp, log_M = kernel.spec()
    if diag:
        return np.full(len(x1), amp)
    # one scratch handle per device, reused: numerical_kernel_gradient calls this 2 d times per point
    cur = torch.cuda.current_device()
    hd = _SCRATCH_HANDLES.get(cur)
    if hd is None or hd.stream != torch.cuda.current_stream(cur):
        hd = _SCRATCH_HANDLES[cur] = _Handle(cur)
    dev = f"cuda:{hd.device}"
    a = torch.from_numpy(np.ascontiguousarray(x1)).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(x2)).to(dev)
    _lib.check(hd.lib.ab_gp_set_inputs(hd.h, _lib.ptr(a), a.shape[0], a.shape[1]), "ab_gp_set_inputs")
    _set_kernel(hd, kernel, 0.0, -50.0, 0.0)
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float64, device=dev)
    _lib.check(hd.lib.ab_gp_cross_cov(hd.h, _lib.ptr(a), a.shape[0], _lib.ptr(b), b.shape[0], _lib.ptr(out)),
               "ab_gp_cross_cov")
    return out.cpu().numpy()
