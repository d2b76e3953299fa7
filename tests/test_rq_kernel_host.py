"""RationalQuadraticKernel on the CPU: the reference (tests/rq_oracle.py) against scikit-learn's
RationalQuadratic and against finite differences, the kernel object's george protocol, and the
SurrogateModel host logic around the kernel's own hyper-parameter (log_alpha)."""
import copy
import os
import pickle
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import rq_oracle as rq  # noqa: E402

sk = pytest.importorskip("sklearn.gaussian_process")
from sklearn.gaussian_process.kernels import ConstantKernel, RationalQuadratic, WhiteKernel  # noqa: E402


def _data(n, d, seed):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-2, 2, size=(n, d))
    y = np.sin(X.sum(axis=1)) - 0.3 * np.sum(X ** 2, axis=1) + 0.01 * rng.normal(size=n)
    return rng, X, y


@pytest.mark.parametrize("log_alpha", [-2.0, 0.0, 3.0])
@pytest.mark.parametrize("n,d,iso", [(60, 1, True), (200, 3, True), (250, 4, False)])
def test_reference_matches_sklearn(n, d, iso, log_alpha):
    """Kernel matrix, log-likelihood and its gradient (incl. d/dlog alpha) against sklearn.  sklearn's
    RationalQuadratic is isotropic: the anisotropic case pre-scales X by 1/sqrt(M) and uses l = 1."""
    rng, X, y = _data(n, d, 100 * n + d)
    log_M = np.full(d, 2.0 * np.log(1.3)) if iso else rng.uniform(-0.6, 1.0, size=d)
    amp, wn, mean = 1.7 * np.var(y), np.exp(-7.0), float(np.median(y))
    o = rq.OracleGP("RationalQuadraticKernel", d, log_M, log_const=np.log(amp), mean=mean, fit_mean=True,
                    white_noise=np.log(wn), fit_white_noise=True, log_alpha=log_alpha)
    o.compute(X)
    Xs = X if iso else X * np.exp(-0.5 * log_M)
    ell = np.exp(0.5 * log_M[0]) if iso else 1.0
    kern = ConstantKernel(amp) * RationalQuadratic(length_scale=ell, alpha=np.exp(log_alpha)) + WhiteKernel(wn)
    gpr = sk.GaussianProcessRegressor(kernel=kern, alpha=0.0, optimizer=None, normalize_y=False)
    gpr.fit(Xs, y - mean)
    K = o.get_matrix(X)
    K[np.diag_indices(n)] += wn
    np.testing.assert_allclose(K, kern(Xs), rtol=1e-12, atol=1e-14)
    ll_s, g_s = gpr.log_marginal_likelihood(kern.theta, eval_gradient=True)
    assert abs(o.log_likelihood(y) - ll_s) <= 1e-9 * abs(ll_s)
    g_o = o.grad_log_likelihood(y)         # [mean, white_noise, log_constant, log_alpha, log_M...]
    # sklearn theta (hyper-parameters sorted by name): [log constant, log alpha, log l, log noise]
    assert [h.name for h in kern.hyperparameters] == ["k1__k1__constant_value", "k1__k2__alpha", "k1__k2__length_scale",
                                                      "k2__noise_level"]
    scale = np.max(np.abs(g_s))
    assert abs(g_o[1] - g_s[3]) <= 1e-8 * scale
    assert abs(g_o[2] - g_s[0]) <= 1e-8 * scale
    assert abs(g_o[3] - g_s[1]) <= 1e-8 * scale
    if iso:                                # d/dlog M = 1/2 d/dlog l, summed over the tied dimensions
        assert abs(0.5 * g_s[2] - g_o[4:].sum()) <= 1e-8 * scale


@pytest.mark.parametrize("log_alpha", [-2.0, 0.0, 3.0, 12.0])
def test_reference_gradient_matches_finite_differences(log_alpha):
    """Every gradient entry against a central difference of the log-likelihood; at log_alpha = 12 every
    pair of points has x = r^2 / (2 alpha) < 1e-4, where the direct form of g(x) would cancel."""
    rng, X, y = _data(120, 3, 7)
    o = rq.make_gp("RationalQuadraticKernel", X, y, rng.uniform(-0.3, 0.8, size=3), amp=np.var(y),
                   white_noise=-6.0, log_alpha=log_alpha)
    g = o.grad_log_likelihood(y)
    p0 = o.get_parameter_vector()
    assert o.get_parameter_names()[3] == "kernel:k2:log_alpha" and p0[3] == log_alpha
    for i in range(len(p0)):
        h = 1e-5 * max(1.0, abs(p0[i]))
        lp = []
        for s in (1, -1):
            p = p0.copy()
            p[i] += s * h
            o.set_parameter_vector(p)
            lp.append(o.log_likelihood(y))
        fd = (lp[0] - lp[1]) / (2 * h)
        assert abs(fd - g[i]) <= 1e-6 * max(abs(g[i]), 1e-3 * np.max(np.abs(g))), (i, fd, g[i])
    o.set_parameter_vector(p0)
    # the alpha derivative is not lost to cancellation: it stays negative-definite-signed (g(x) > 0)
    r2 = np.array([0.0, 1e-30, 1e-12, 1e-3, 0.5, 3.0])
    dk = rq.radial_dlog_alpha(r2, log_alpha)
    assert dk[0] == 0.0 and np.all(dk[1:] < 0.0)


def test_g_is_accurate_on_both_sides_of_the_series_switch():
    """g(x) = log1p(x) - x / (1 + x): the 15-term series below x = 1/16 and the direct form above both
    agree with a 40-term series (converged to rounding for x <= 1/8)."""
    x = np.array([1e-150, 1e-9, 1e-4, 0.01, 0.06, 0.0625 * (1 - 1e-12), 0.0625, 0.08, 0.125])
    p = np.zeros_like(x)
    for n in range(40, 1, -1):
        p = p * x + (-1.0) ** n * (n - 1) / n
    np.testing.assert_allclose(rq.rq_g(x), p * x * x, rtol=3e-14)
    assert rq.rq_g(np.array(1e-150)) > 0.0


def test_kernel_object_protocol():
    from alabi_b200 import kernels as K
    k = K.RationalQuadraticKernel(log_alpha=0.7, metric=[1.5, 2.0, 0.5], metric_bounds=[(-2, 2)] * 3, ndim=3)
    assert k.get_parameter_names() == ("log_alpha", "metric:log_M_0_0", "metric:log_M_1_1", "metric:log_M_2_2")
    np.testing.assert_array_equal(k.get_parameter_vector(), [0.7, np.log(1.5), np.log(2.0), np.log(0.5)])
    assert k.get_parameter_bounds() == [(None, None), (-2, 2), (-2, 2), (-2, 2)]
    assert len(k) == 4
    kid, amp, lm = k.spec()
    assert (kid, amp) == (3, 1.0) and np.array_equal(lm, np.log([1.5, 2.0, 0.5]))
    p = k * 3.0
    assert isinstance(p, K.Product) and p.kernel_id == 3 and p.log_alpha == 0.7
    assert p.get_parameter_names() == ("k1:log_constant", "k2:log_alpha", "k2:metric:log_M_0_0",
                                       "k2:metric:log_M_1_1", "k2:metric:log_M_2_2")
    kid, amp, lm = p.spec()
    assert kid == 3 and amp == pytest.approx(1.0) and len(lm) == 3
    v = p.get_parameter_vector()
    v[1] = -1.25
    p.set_parameter_vector(v)
    assert p.log_alpha == -1.25 and k.log_alpha == -1.25
    p.set_parameter("k2:log_alpha", 2.0)
    assert p.get_parameter("k2:log_alpha") == 2.0
    for c in (pickle.loads(pickle.dumps(p)), copy.deepcopy(p)):
        assert c.log_alpha == 2.0 and np.array_equal(c.get_parameter_vector(), p.get_parameter_vector())
        assert c.get_parameter_names() == p.get_parameter_names()
    iso = K.RationalQuadraticKernel(0.0, metric=2.0, ndim=4)
    assert iso.get_parameter_names() == ("log_alpha", "metric:log_M_0_0") and len(iso.spec()[2]) == 4
    with pytest.raises(ValueError):
        k.set_parameter_vector([0.0, 1.0, 1.0])
    # the device GP's parameter protocol and the dirty check see log_alpha
    from alabi_b200.gp import GP
    g = GP(kernel=K.RationalQuadraticKernel(0.3, metric=[1.0, 1.0], ndim=2) * 2.0, fit_mean=True, mean=0.0,
           white_noise=-8.0, fit_white_noise=True)
    assert g.get_parameter_names() == ("mean:value", "white_noise:value", "kernel:k1:log_constant", "kernel:k2:log_alpha",
                                       "kernel:k2:metric:log_M_0_0", "kernel:k2:metric:log_M_1_1")
    key = g._spec_key()
    g.set_parameter("kernel:k2:log_alpha", 0.4)
    assert g._spec_key() != key


def _rq_stand_in():
    """alabi_b200.gp.GP on the CPU, backed by the RQ reference (like tests/test_host_logic.py's stand-in)."""
    from alabi_b200 import kernels as K

    class RQBackedGP(rq.OracleGP):
        def __init__(self, kernel=None, fit_mean=False, mean=0.0, white_noise=-12.0, fit_white_noise=False, device=None,
                     **kw):
            base, log_const = (kernel.k2, float(kernel.k1.log_constant)) if isinstance(kernel, K.Product) else (kernel, None)
            lm = np.full(base.ndim, base.log_M[0]) if base.isotropic else np.array(base.log_M, dtype=float)
            super().__init__(base.kernel_id, base.ndim, lm, log_const=log_const, mean=mean, fit_mean=fit_mean,
                             white_noise=white_noise, fit_white_noise=fit_white_noise, log_alpha=base.log_alpha)
            self.kernel = kernel
    return RQBackedGP


@pytest.mark.parametrize("uniform_scales", [False, True])
def test_init_gp_host_logic(uniform_scales, tmp_path, monkeypatch):
    """SurrogateModel.init_gp(kernel="RationalQuadraticKernel"): names, the log_alpha prior bound
    (gp_alpha_rng), the optimised names and expand_hyperparameter_vector with uniform_scales."""
    from sklearn import preprocessing
    from alabi_b200 import core, gp_utils
    stand_in = _rq_stand_in()
    monkeypatch.setattr(core, "GP", stand_in)
    monkeypatch.setattr(gp_utils, "GP", stand_in)
    d = 3
    bounds = np.array([(-2.0, 2.0)] * d)
    rng, theta, y = _data(40, d, 3)
    sm = core.SurrogateModel(lnlike_fn=lambda t: 0.0, bounds=bounds, savedir=str(tmp_path), cache=False, verbose=False)
    sm.theta_train, sm.y_train, sm.theta_test, sm.y_test = theta, y, [], []
    sm.ntrain, sm.ntest = len(theta), 0
    np.random.seed(5)
    sm.init_gp(kernel="RationalQuadraticKernel", uniform_scales=uniform_scales, white_noise=-8, gp_alpha_rng=[-1.5, 2.5],
               theta_scaler=preprocessing.MinMaxScaler(), y_scaler=preprocessing.StandardScaler(), gp_nopt=1,
               hyperopt_method="ml", optimizer_kwargs={"maxiter": 20})
    assert sm.param_names_full == ["mean:value", "white_noise:value", "kernel:k1:log_constant", "kernel:k2:log_alpha"] + \
        [f"kernel:k2:metric:log_M_{i}_{i}" for i in range(d)]
    opt = ["mean:value", "kernel:k1:log_constant", "white_noise:value", "kernel:k2:log_alpha"]
    opt += ["kernel:k2:metric:log_M"] if uniform_scales else [f"kernel:k2:metric:log_M_{i}_{i}" for i in range(d)]
    assert sm.param_names_optimized == opt
    pnames = opt if uniform_scales else sm.param_names_full
    hb = np.array(sm.hp_bounds, dtype=float)
    assert not np.any(np.isnan(hb))
    np.testing.assert_array_equal(hb[pnames.index("kernel:k2:log_alpha")], [-1.5, 2.5])
    assert sm.initial_gp_hyperparameters[pnames.index("kernel:k2:log_alpha")] == 0.0     # alpha = 1 at the start
    if uniform_scales:
        p = np.array([0.1, 0.2, -7.0, 1.75, 0.3])
        full = sm.expand_hyperparameter_vector(p)
        np.testing.assert_array_equal(full, [0.1, -7.0, 0.2, 1.75, 0.3, 0.3, 0.3])
    # the fit left a finite model with log_alpha inside what the optimiser was allowed
    la = sm.gp.get_parameter_dict()["kernel:k2:log_alpha"]
    assert -1.5 <= la <= 2.5 and np.isfinite(sm.gp.log_likelihood(sm._y))


def test_unknown_and_known_kernel_names():
    from alabi_b200 import core
    assert "RationalQuadraticKernel" in core._KERNELS
