"""george.kernels look-alikes for the four kernels of the surrogate hot path.

Mirrors the constructor and parameter protocol alabi uses
(``kernels.ExpSquaredKernel(metric=vec, metric_bounds=[...], ndim=d)`` at
alabi/core.py:998-1014, ``kernel * float`` at alabi/gp_utils.py:230-231 and
alabi/core.py:1136-1139, ``kernel.get_parameter_names()`` at
alabi/gp_utils.py:333,1251, ``kernel.get_value(x1, x2)`` at
alabi/utility.py:549-550,607).  The objects only carry hyper-parameters; all
arithmetic happens in the CUDA library (K1 / cross-covariance kernels).
"""
import numpy as np

__all__ = ["ExpSquaredKernel", "Matern32Kernel", "Matern52Kernel", "RationalQuadraticKernel", "ConstantKernel",
           "Product"]


class Kernel:
    is_kernel = True
    ndim = 1

    # george: float * kernel builds ConstantKernel(log(c / ndim)) * kernel
    def __mul__(self, b):
        if not hasattr(b, "is_kernel"):
            return Product(ConstantKernel(log_constant=np.log(float(b) / self.ndim), ndim=self.ndim), self)
        return Product(self, b)

    def __rmul__(self, b):
        if not hasattr(b, "is_kernel"):
            return Product(ConstantKernel(log_constant=np.log(float(b) / self.ndim), ndim=self.ndim), self)
        return Product(b, self)

    def __len__(self):
        return len(self.get_parameter_vector())

    def get_parameter_dict(self, include_frozen=False):
        return dict(zip(self.get_parameter_names(), self.get_parameter_vector()))

    def get_parameter(self, name):
        return self.get_parameter_dict()[name]

    def set_parameter(self, name, value):
        names = list(self.get_parameter_names())
        v = self.get_parameter_vector()
        v[names.index(name)] = value
        self.set_parameter_vector(v)

    # -- value: evaluated on the GPU through a scratch GP handle ----------------
    def get_value(self, x1, x2=None, diag=False):
        from .gp import _kernel_value
        return _kernel_value(self, x1, x2, diag)

    def spec(self):
        """(kernel_id, amp, log_M vector) — what the C ABI takes."""
        raise NotImplementedError


class ConstantKernel(Kernel):
    kernel_id = None

    def __init__(self, log_constant=0.0, ndim=1, axes=None):
        self.log_constant = float(log_constant)
        self.ndim = int(ndim)

    def get_parameter_names(self, include_frozen=False):
        return ("log_constant",)

    def get_parameter_vector(self, include_frozen=False):
        return np.array([self.log_constant])

    def set_parameter_vector(self, v, include_frozen=False):
        self.log_constant = float(np.atleast_1d(v)[0])

    def get_parameter_bounds(self, include_frozen=False):
        return [(None, None)]


class _Stationary(Kernel):
    kernel_id = None

    def __init__(self, metric=None, metric_bounds=None, ndim=1, axes=None, lower=True, block=None, bounds=None):
        if block is not None or axes is not None:
            raise NotImplementedError("alabi_b200 kernels support the full-axis metric only")
        self.ndim = int(ndim)
        m = np.atleast_1d(np.asarray(metric, dtype=np.float64))
        if m.ndim != 1:
            raise NotImplementedError("general (dense) metrics are outside the alabi hot path")
        if len(m) == 1:
            self.isotropic = True
        elif len(m) == self.ndim:
            self.isotropic = False
        else:
            raise ValueError("dimension mismatch between metric and ndim")
        if np.any(m <= 0):
            raise ValueError("metric must be positive")
        self.log_M = np.log(m)
        self.metric_bounds = metric_bounds

    def get_parameter_names(self, include_frozen=False):
        return tuple(f"metric:log_M_{i}_{i}" for i in range(len(self.log_M)))

    def get_parameter_vector(self, include_frozen=False):
        return self.log_M.copy()

    def set_parameter_vector(self, v, include_frozen=False):
        v = np.atleast_1d(np.asarray(v, dtype=np.float64))
        if len(v) != len(self.log_M):
            raise ValueError("dimension mismatch")
        self.log_M = v.copy()

    def get_parameter_bounds(self, include_frozen=False):
        if self.metric_bounds is None:
            return [(None, None)] * len(self.log_M)
        return list(self.metric_bounds)

    def spec(self):
        lm = np.full(self.ndim, self.log_M[0]) if self.isotropic else self.log_M
        return self.kernel_id, 1.0, np.ascontiguousarray(lm, dtype=np.float64)


class ExpSquaredKernel(_Stationary):
    """k(r^2) = exp(-r^2 / 2),  r^2 = sum_i (x_i - x'_i)^2 / M_i."""
    kernel_id = 0


class Matern32Kernel(_Stationary):
    """k(r^2) = (1 + sqrt(3 r^2)) exp(-sqrt(3 r^2))."""
    kernel_id = 1


class Matern52Kernel(_Stationary):
    """k(r^2) = (1 + sqrt(5 r^2) + 5 r^2 / 3) exp(-sqrt(5 r^2))."""
    kernel_id = 2


class RationalQuadraticKernel(_Stationary):
    """k(r^2) = (1 + r^2 / (2 alpha))^(-alpha),  alpha = exp(log_alpha).

    The kernel's own parameter comes before the metric, as in george:
    names ``("log_alpha", "metric:log_M_0_0", ...)``, vector ``[log_alpha, log_M...]``.
    ``spec()`` keeps the (kernel_id, amp, log_M) form of the other kernels; the device
    reads ``log_alpha`` separately (``ab_gp_set_kernel_rq``)."""
    kernel_id = 3

    def __init__(self, log_alpha, metric, metric_bounds=None, ndim=1, axes=None, lower=True, block=None, bounds=None):
        super().__init__(metric=metric, metric_bounds=metric_bounds, ndim=ndim, axes=axes, lower=lower, block=block)
        self.log_alpha = float(log_alpha)

    def get_parameter_names(self, include_frozen=False):
        return ("log_alpha",) + super().get_parameter_names()

    def get_parameter_vector(self, include_frozen=False):
        return np.concatenate([[self.log_alpha], self.log_M])

    def set_parameter_vector(self, v, include_frozen=False):
        v = np.atleast_1d(np.asarray(v, dtype=np.float64))
        if len(v) != 1 + len(self.log_M):
            raise ValueError("dimension mismatch")
        self.log_alpha = float(v[0])
        self.log_M = v[1:].copy()

    def get_parameter_bounds(self, include_frozen=False):
        return [(None, None)] + super().get_parameter_bounds()


class Product(Kernel):
    """ConstantKernel * stationary kernel (the only product alabi builds)."""

    def __init__(self, k1, k2):
        if isinstance(k2, ConstantKernel) and not isinstance(k1, ConstantKernel):
            k1, k2 = k2, k1
        if not isinstance(k1, ConstantKernel) or not isinstance(k2, _Stationary):
            raise NotImplementedError("only ConstantKernel * {ExpSquared, Matern32, Matern52, RationalQuadratic}Kernel "
                                      "is supported")
        self.k1, self.k2 = k1, k2
        self.ndim = k2.ndim

    @property
    def kernel_id(self):
        return self.k2.kernel_id

    @property
    def log_alpha(self):
        """log_alpha of a RationalQuadraticKernel factor (AttributeError for the other kernels)."""
        return self.k2.log_alpha

    def get_parameter_names(self, include_frozen=False):
        return tuple("k1:" + n for n in self.k1.get_parameter_names()) + \
               tuple("k2:" + n for n in self.k2.get_parameter_names())

    def get_parameter_vector(self, include_frozen=False):
        return np.concatenate([self.k1.get_parameter_vector(), self.k2.get_parameter_vector()])

    def set_parameter_vector(self, v, include_frozen=False):
        v = np.atleast_1d(np.asarray(v, dtype=np.float64))
        self.k1.set_parameter_vector(v[:1])
        self.k2.set_parameter_vector(v[1:])

    def get_parameter_bounds(self, include_frozen=False):
        return self.k1.get_parameter_bounds() + self.k2.get_parameter_bounds()

    def spec(self):
        kid, _, lm = self.k2.spec()
        with np.errstate(over="ignore"):      # an optimiser may stray to exp(...) = inf: K is then not factorisable
            amp = float(np.exp(self.k1.log_constant))
        return kid, amp, lm
