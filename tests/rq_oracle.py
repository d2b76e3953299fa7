"""CPU reference for george's RationalQuadraticKernel, built on oracle/gp.py.

TEST INFRASTRUCTURE ONLY.  george is not installed; its kernel is restated from its
documentation (recalled, like the other george facts in ``oracle/gp.py``):

    k(r^2) = (1 + r^2 / (2 alpha))^(-alpha),  alpha = exp(log_alpha),  r^2 = sum_k dx_k^2 / M_k

george names the kernel's own parameter before the metric (recalled, not checked):
``log_alpha``, then ``metric:log_M_i_i``.  Inside the amplitude product the full GP vector is
``[mean:value, white_noise:value, kernel:k1:log_constant, kernel:k2:log_alpha,
kernel:k2:metric:log_M_0_0, ...]``.  scikit-learn's ``RationalQuadratic(length_scale=l,
alpha=alpha)`` is the same function with M = l^2 (an independent check, tests/test_rq_kernel_host.py).

Every function takes the kernel id (or george name) of ``oracle.gp`` plus an optional
``log_alpha``; kinds 0-2 are delegated to ``oracle.gp`` unchanged.
"""
import numpy as np

from oracle import gp as ogp

RQ = 3
KERNEL_IDS = dict(ogp.KERNEL_IDS, RationalQuadraticKernel=RQ)


def _kind(kind):
    return KERNEL_IDS.get(kind, kind)


def rq_g(x):
    """g(x) = log1p(x) - x / (1 + x) >= 0 without the cancellation of the two terms at small x:
    the series x^2/2 - 2x^3/3 + 3x^4/4 - ... (through x^15) below x = 1/16, the direct form above
    (the same split as the device, csrc/common.cuh ab_rq_g)."""
    x = np.asarray(x, dtype=np.float64)
    p = np.zeros_like(x)
    for n in range(15, 1, -1):
        p = p * x + (-1.0) ** n * (n - 1) / n
    series = p * x * x
    with np.errstate(invalid="ignore"):
        direct = np.log1p(x) - x / (1.0 + x)
    return np.where(x < 0.0625, series, direct)


def radial(kind, r2, log_alpha=None):
    """k(r^2)."""
    if _kind(kind) != RQ:
        return ogp.radial(kind, r2)
    a = np.exp(log_alpha)
    return np.exp(-a * np.log1p(r2 / (2.0 * a)))


def radial_grad(kind, r2, log_alpha=None):
    """dk/d(r^2)."""
    if _kind(kind) != RQ:
        return ogp.radial_grad(kind, r2)
    a = np.exp(log_alpha)
    x = r2 / (2.0 * a)
    return -0.5 * np.exp(-a * np.log1p(x)) / (1.0 + x)


def radial_dlog_alpha(r2, log_alpha):
    """dk/dlog(alpha) = -alpha k g(x), x = r^2 / (2 alpha)."""
    a = np.exp(log_alpha)
    x = r2 / (2.0 * a)
    return -a * np.exp(-a * np.log1p(x)) * rq_g(x)


def kernel_value(kind, x1, x2, log_M, log_const=None, log_alpha=None):
    """amp * k(x1, x2); amp = exp(log_const) (ConstantKernel product) or 1."""
    k = radial(kind, ogp.scaled_sqdist(x1, x2, log_M), log_alpha)
    if log_const is not None:
        k = np.exp(log_const) * k
    return k


class OracleGP(ogp.OracleGP):
    """``oracle.gp.OracleGP`` that also knows the rational quadratic kernel (``log_alpha`` given)."""

    def __init__(self, kind, ndim, log_M, log_const=None, mean=0.0, fit_mean=False, white_noise=-12.0,
                 fit_white_noise=False, log_alpha=None):
        super().__init__(_kind(kind), ndim, log_M, log_const=log_const, mean=mean, fit_mean=fit_mean,
                         white_noise=white_noise, fit_white_noise=fit_white_noise)
        self.log_alpha = None if log_alpha is None else float(log_alpha)
        if (self.kind == RQ) != (self.log_alpha is not None):
            raise ValueError("log_alpha is given exactly for the rational quadratic kernel")

    def get_parameter_names(self, include_frozen=False):
        names = list(super().get_parameter_names(include_frozen))
        if self.log_alpha is not None:
            pre = "kernel:k2:" if self.log_const is not None else "kernel:"
            names.insert(len(names) - self.ndim, pre + "log_alpha")
        return tuple(names)

    def get_parameter_vector(self):
        v = list(super().get_parameter_vector())
        if self.log_alpha is not None:
            v.insert(len(v) - self.ndim, self.log_alpha)
        return np.array(v, dtype=np.float64)

    def set_parameter_vector(self, v):
        v = np.asarray(v, dtype=np.float64)
        if self.log_alpha is None:
            return super().set_parameter_vector(v)
        if len(v) != len(self.get_parameter_vector()):
            raise ValueError("dimension mismatch")
        n = 0
        if self.fit_mean:
            self.mean = float(v[n]); n += 1
        if self.fit_white_noise:
            self.white_noise = float(v[n]); n += 1
        if self.log_const is not None:
            self.log_const = float(v[n]); n += 1
        self.log_alpha = float(v[n])
        self.log_M = v[n + 1:n + 1 + self.ndim].copy()
        self.computed = False
        self._alpha = None

    def get_matrix(self, x1, x2=None):
        x2 = x1 if x2 is None else x2
        return kernel_value(self.kind, x1, x2, self.log_M, self.log_const, self.log_alpha)

    def grad_log_likelihood(self, y, quiet=False):
        """The N x N x P construction of george, with the d/dlog(alpha) column in george's order."""
        if self.kind != RQ:
            return super().grad_log_likelihood(y, quiet=quiet)
        npar = len(self.get_parameter_vector())
        if not self.recompute(quiet=quiet):
            return np.zeros(npar)
        alpha = self._compute_alpha(y)
        A = np.outer(alpha, alpha) - self.get_inverse()
        out = []
        if self.fit_mean:
            out.append(np.sum(alpha))
        if self.fit_white_noise:
            out.append(0.5 * np.exp(self.white_noise) * np.trace(A))
        x = self._x
        r2 = ogp.scaled_sqdist(x, x, self.log_M)
        amp = 1.0 if self.log_const is None else np.exp(self.log_const)
        if self.log_const is not None:
            out.append(0.5 * np.sum(A * (amp * radial(RQ, r2, self.log_alpha))))
        out.append(0.5 * np.sum(A * (amp * radial_dlog_alpha(r2, self.log_alpha))))
        dk = amp * radial_grad(RQ, r2, self.log_alpha)
        inv_M = np.exp(-self.log_M)
        for k in range(self.ndim):
            d2 = (x[:, None, k] - x[None, :, k]) ** 2 * inv_M[k]
            out.append(0.5 * np.sum(A * dk * (-d2)))
        return np.array(out, dtype=np.float64)

    def predict_grad(self, y, t, h=None):
        """d mu / dx and d sigma^2 / dx as ``oracle.gp.OracleGP.predict_grad`` (analytic only)."""
        if self.kind != RQ or h is not None:
            return super().predict_grad(y, t, h)
        self.recompute()
        alpha = self._compute_alpha(y)
        xs = np.atleast_2d(np.asarray(t, dtype=np.float64))
        amp = 1.0 if self.log_const is None else np.exp(self.log_const)
        inv_M = np.exp(-self.log_M)
        dmu, dvar = np.zeros_like(xs), np.zeros_like(xs)
        for q in range(len(xs)):
            diff = xs[q][None, :] - self._x
            r2 = np.sum(diff * diff * inv_M[None, :], axis=1)
            gk = (amp * radial_grad(RQ, r2, self.log_alpha))[:, None] * 2.0 * diff * inv_M[None, :]
            ks = self.get_matrix(xs[q][None, :], self._x).ravel()
            dmu[q] = gk.T @ alpha
            dvar[q] = -2.0 * gk.T @ self.apply_inverse(ks)
        return dmu, dvar


def make_gp(kind, x, y, log_M, amp=None, mean=None, white_noise=-12.0, fit_mean=True, fit_white_noise=True,
            compute=True, log_alpha=None):
    """``oracle.gp.make_gp`` with an optional ``log_alpha`` (rational quadratic kernel)."""
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    ndim = x.shape[1]
    log_const = None if amp is None else np.log(float(amp) / ndim)
    gp = OracleGP(_kind(kind), ndim, log_M, log_const=log_const, mean=np.median(y) if mean is None else mean,
                  fit_mean=fit_mean, white_noise=white_noise, fit_white_noise=fit_white_noise, log_alpha=log_alpha)
    if compute:
        gp.compute(x)
    return gp
