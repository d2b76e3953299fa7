"""GPU tests of the full predictive covariance (GP.predict(return_cov=True), ab_gp_predict_cov) and of
the multivariate-normal draws (GP.sample_conditional, GP.sample, ab_mvn_sample), for all four kernels.

Covariance: against the CPU oracle (oracle.gp / tests/rq_oracle.py, cov = K(t,t) - Kxs K^-1 Kxs^T) within
the sigma^2 bound of test_gpu_benchmark_configs.py, |dSigma_ab| <= (16 sqrt(kappa) + N / 8) eps amp, and
bit for bit against the device's own variance and mean paths.  Draws: exact replay of the normals
(Philox4x32-10 from oracle/philox.py plus NumPy Box-Muller, ``replay_normals`` below), Monte-Carlo
moments, determinism, shapes and the failure paths."""
import ctypes
import os
import pickle
import sys

import numpy as np
import pytest

from oracle import philox as oph

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import rq_oracle as rq  # noqa: E402

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
KINDS = ["ExpSquaredKernel", "Matern32Kernel", "Matern52Kernel", "RationalQuadraticKernel"]
STREAM_MVN = 3                       # AB_STREAM_MVN of include/alabi_b200.h


def replay_normals(seed, m, size):
    """CPU replay of the normals of ab_mvn_sample: Z[i][s] (m x size), counter (i, s // 2, 0, STREAM_MVN),
    key = seed, u1 = 1 - u53(x, y), u2 = u53(z, w), Z[i][2p] = r cos(2 pi u2), Z[i][2p + 1] = r sin(2 pi u2)."""
    npair = (size + 1) // 2
    i = np.repeat(np.arange(m, dtype=np.uint64), npair)
    p = np.tile(np.arange(npair, dtype=np.uint64), m)
    x, y, z, w = oph.philox4x32(i, p, 0, STREAM_MVN, seed & 0xFFFFFFFF, seed >> 32)
    u1 = 1.0 - oph.u53(x, y)
    u2 = oph.u53(z, w)
    r = np.sqrt(-2.0 * np.log(u1))
    out = np.empty((m, 2 * npair))
    out[:, 0::2] = (r * np.cos(2.0 * np.pi * u2)).reshape(m, npair)
    out[:, 1::2] = (r * np.sin(2.0 * np.pi * u2)).reshape(m, npair)
    return out[:, :size], r.reshape(m, npair)


def make_pair(kind, n, d, seed=0, white_noise=-6.0, lo=-1.0, hi=1.0):
    import alabi_b200 as ab
    rng = np.random.default_rng(seed)
    X = rng.uniform(lo, hi, size=(n, d))
    y = np.sin(X.sum(axis=1)) + 0.3 * np.cos(2.0 * X[:, 0]) + 0.05 * rng.normal(size=n)
    log_M = rng.uniform(-0.5, 0.8, size=d)
    la = 0.5 if kind == "RationalQuadraticKernel" else None
    o = rq.make_gp(kind, X, y, log_M, amp=np.var(y), white_noise=white_noise, log_alpha=la)
    if la is None:
        k = getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d)
    else:
        k = ab.kernels.RationalQuadraticKernel(la, metric=np.exp(log_M), ndim=d)
    g = ab.GP(kernel=k * np.var(y), fit_mean=True, mean=np.median(y), white_noise=white_noise, fit_white_noise=True)
    g.compute(X)
    return o, g, X, y, rng


def kappa_of(o, X):
    K = o.get_matrix(X) + np.exp(o.white_noise) * np.eye(len(X))
    ev = np.linalg.eigvalsh(K)
    return ev[-1] / ev[0]


def check_cov_bits(g, y, t, mu, cov):
    """The bit-identity properties of one (mu, cov) = g.predict(y, t)."""
    m = len(t)
    mu_v, var_v = g.predict(y, t, return_var=True)
    np.testing.assert_array_equal(np.diag(cov), var_v)
    np.testing.assert_array_equal(mu, mu_v)
    np.testing.assert_array_equal(mu, g.predict(y, t, return_cov=False))
    np.testing.assert_array_equal(cov, cov.T)
    if m >= 2:
        rng = np.random.default_rng(m)
        idx = rng.permutation(m)[:max(1, (2 * m) // 3)]
        mu_s, cov_s = g.predict(y, t[idx])
        np.testing.assert_array_equal(cov_s, cov[np.ix_(idx, idx)])
        np.testing.assert_array_equal(mu_s, mu[idx])


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [150, 257, 1000])
def test_cov_against_oracle_and_bits(kind, n):
    import torch
    d = 5
    o, g, X, y, rng = make_pair(kind, n, d, seed=n + len(kind))
    amp = np.exp(o.log_const)
    bound = (16.0 * np.sqrt(kappa_of(o, X)) + n / 8.0) * EPS * amp
    t_all = rng.uniform(-1.1, 1.1, size=(300, d))
    t_all[5] = X[3]                                        # a query on a training point
    for m in [1, 7, 8, 9, 127, 128, 129, 300]:
        t = t_all[:m]
        mu, cov = g.predict(y, t)                          # george's default: return_cov=True
        assert mu.shape == (m,) and cov.shape == (m, m) and isinstance(cov, np.ndarray)
        mu_o, cov_o = o.predict(y, t, return_cov=True)
        err = np.max(np.abs(cov - cov_o))
        assert err <= bound, (kind, n, m, err / (EPS * amp), bound / (EPS * amp))
        assert np.max(np.abs(mu - mu_o)) <= 1e-9 * np.max(np.abs(mu_o)), (kind, n, m)
        check_cov_bits(g, y, t, mu, cov)
        # device tensors in -> device tensors out, same bits
        td = torch.from_numpy(t).cuda()
        mu_d, cov_d = g.predict(y, td, return_cov=True)
        assert mu_d.is_cuda and cov_d.is_cuda
        np.testing.assert_array_equal(mu_d.cpu().numpy(), mu)
        np.testing.assert_array_equal(cov_d.cpu().numpy(), cov)
    # return_var keeps precedence (george); an empty query set gives empty results
    mu, var = g.predict(y, t_all[:4], return_cov=True, return_var=True)
    assert var.shape == (4,)
    mu0, cov0 = g.predict(y, np.empty((0, d)))
    assert mu0.shape == (0,) and cov0.shape == (0, 0)


def test_cov_c4_size_subset():
    """N = 8192, d = 10, M = 2048: a 256-query subset against the oracle (valid by the sub-batch property,
    which is checked bit for bit on the same subset).  kappa is bounded by N (amp + noise) / noise."""
    kind, n, d, m = "ExpSquaredKernel", 8192, 10, 2048
    o, g, X, y, rng = make_pair(kind, n, d, seed=4, white_noise=-8.0)
    amp = np.exp(o.log_const)
    noise = np.exp(o.white_noise)
    kappa = n * (amp + noise) / noise
    bound = (16.0 * np.sqrt(kappa) + n / 8.0) * EPS * amp
    t = rng.uniform(-1.1, 1.1, size=(m, d))
    mu, cov = g.predict(y, t)
    idx = np.sort(rng.choice(m, 256, replace=False))
    mu_s, cov_s = g.predict(y, t[idx])
    np.testing.assert_array_equal(cov_s, cov[np.ix_(idx, idx)])
    np.testing.assert_array_equal(mu_s, mu[idx])
    mu_o, cov_o = o.predict(y, t[idx], return_cov=True)
    err = np.max(np.abs(cov_s - cov_o))
    assert err <= bound, (err / (EPS * amp), bound / (EPS * amp))
    np.testing.assert_array_equal(np.diag(cov), g.predict(y, t, return_var=True)[1])
    np.testing.assert_array_equal(cov, cov.T)


def _lib_handle(g):
    return g._hd.lib, g._hd.h


def test_normals_replay_and_conditional_draws():
    import torch
    from alabi_b200 import _lib
    o, g, X, y, rng = make_pair("Matern52Kernel", 400, 3, seed=11, white_noise=-6.0)
    lib, h = _lib_handle(g)
    # identity covariance, no mean: the draws ARE the normals (L = I, every product exact)
    m, size, seed = 37, 301, 0x1234_5678_9ABC_DEF0
    eye = torch.eye(m, dtype=torch.float64, device="cuda")
    out = torch.empty((size, m), dtype=torch.float64, device="cuda")
    info = ctypes.c_int(-7)
    rc = lib.ab_mvn_sample(h, _lib.ptr(eye), m, m, None, 0.0, size, seed, _lib.ptr(out), ctypes.byref(info))
    assert rc == 0 and info.value == 0
    z_dev = out.cpu().numpy().T
    z_ref, rad = replay_normals(seed, m, size)
    scale = np.repeat(rad, 2, axis=1)[:, :size]             # |z| <= r: error relative to the radius
    assert np.max(np.abs(z_dev - z_ref) / scale) < 1e-14
    # conditional draws = mu + chol(Sigma_dev) z on a well-conditioned set (d = 10, queries spread
    # over a box twice the training box: neighbouring queries are a few length scales apart)
    o, g, X, y, rng = make_pair("Matern52Kernel", 400, 10, seed=12, white_noise=-6.0)
    m, size, seed = 200, 64, 99
    t = rng.uniform(-2.0, 2.0, size=(m, 10))
    mu, cov = g.predict(y, t)
    draws = g.sample_conditional(y, t, size=size, seed=seed, jitter=0.0)
    assert draws.shape == (size, m)
    z, _ = replay_normals(seed, m, size)
    L = np.linalg.cholesky(cov)
    ref = mu[None, :] + (L @ z).T
    # Cholesky perturbation: |dL| / |L| <~ kappa(Sigma) m eps (two factorisations in different orders)
    ev = np.linalg.eigvalsh(cov)
    kap = ev[-1] / ev[0]
    tol = 8.0 * m * kap * EPS * np.sqrt(np.max(np.diag(cov))) * np.max(np.abs(z)) + 1e-12 * np.max(np.abs(mu))
    assert np.max(np.abs(draws - ref)) <= tol, (np.max(np.abs(draws - ref)), tol, kap)


def _moments_ok(draws, mu, cov, what):
    s = draws.shape[0]
    mean = draws.mean(axis=0)
    sd = np.sqrt(np.diag(cov))
    assert np.all(np.abs(mean - mu) <= 5.0 * sd / np.sqrt(s)), (what, (mean - mu) / (sd / np.sqrt(s)))
    c = np.cov(draws, rowvar=False)
    se = np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / s)
    assert np.all(np.abs(c - cov) <= 5.0 * se), (what, np.max(np.abs(c - cov) / se))


def test_draw_moments():
    o, g, X, y, rng = make_pair("ExpSquaredKernel", 12, 4, seed=5, white_noise=-6.0)
    t = rng.uniform(-2.0, 2.0, size=(12, 4))
    S = 200_000
    mu, cov = g.predict(y, t)
    _moments_ok(g.sample_conditional(y, t, size=S, seed=1), mu, cov, "sample_conditional")
    prior = o.get_matrix(t)
    _moments_ok(g.sample(t, size=S, seed=2), np.full(12, g.mean_value), prior, "sample(t)")
    K = o.get_matrix(X) + np.exp(o.white_noise) * np.eye(len(X))
    _moments_ok(g.sample(size=S, seed=3), np.full(12, g.mean_value), K, "sample()")


def test_draw_determinism_prefix_and_shapes():
    import torch
    o, g, X, y, rng = make_pair("RationalQuadraticKernel", 300, 4, seed=8)
    t = rng.uniform(-1.0, 1.0, size=(50, 4))
    a = g.sample_conditional(y, t, size=10, seed=42)
    b = g.sample_conditional(y, t, size=10, seed=42)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(a[:3], g.sample_conditional(y, t, size=3, seed=42))
    np.testing.assert_array_equal(a[0], g.sample_conditional(y, t, seed=42))
    assert not np.array_equal(a, g.sample_conditional(y, t, size=10, seed=43))
    np.random.seed(123)
    c = g.sample_conditional(y, t, size=4)
    np.random.seed(123)
    np.testing.assert_array_equal(c, g.sample_conditional(y, t, size=4))
    # george's shapes: (size, M), or (M,) for size == 1
    assert g.sample_conditional(y, t).shape == (50,)
    assert g.sample(t, size=5, seed=1).shape == (5, 50)
    assert g.sample(t, seed=1).shape == (50,)
    assert g.sample(size=2, seed=1).shape == (2, 300)
    assert g.sample(seed=1).shape == (300,)
    # device queries -> device draws with the same bits
    dd = g.sample_conditional(y, torch.from_numpy(t).cuda(), size=10, seed=42)
    assert dd.is_cuda
    np.testing.assert_array_equal(dd.cpu().numpy(), a)
    # a GP that was never computed draws from its prior at t
    import alabi_b200 as ab
    fresh = ab.GP(kernel=ab.kernels.Matern32Kernel(metric=[0.5, 0.5, 0.5, 0.5], ndim=4) * 2.0)
    np.testing.assert_array_equal(fresh.sample(t, size=3, seed=9), fresh.sample(t, size=3, seed=9))


def test_failure_paths():
    import torch
    from alabi_b200 import _lib
    o, g, X, y, rng = make_pair("Matern32Kernel", 200, 3, seed=21)
    lib, h = _lib_handle(g)
    m = 40
    bad = torch.eye(m, dtype=torch.float64, device="cuda")
    bad[17, 17] = -1.0                                      # indefinite: first non-positive pivot 18
    out = torch.full((5, m), 123.0, dtype=torch.float64, device="cuda")
    info = ctypes.c_int(0)
    rc = lib.ab_mvn_sample(h, _lib.ptr(bad), m, m, None, 0.0, 5, 1, _lib.ptr(out), ctypes.byref(info))
    assert rc == 18 and info.value == 18
    assert torch.all(out == 123.0)
    # bad arguments
    good = torch.eye(m, dtype=torch.float64, device="cuda")
    P = _lib.ptr
    assert lib.ab_mvn_sample(h, P(good), m, m - 1, None, 0.0, 5, 1, P(out), ctypes.byref(info)) == -1
    assert lib.ab_mvn_sample(h, P(good), m, m, None, 0.0, 0, 1, P(out), ctypes.byref(info)) == -1
    assert lib.ab_mvn_sample(h, P(good), m, m, None, -1e-3, 5, 1, P(out), ctypes.byref(info)) == -1
    assert lib.ab_mvn_sample(h, P(good), m, m, None, float("nan"), 5, 1, P(out), ctypes.byref(info)) == -1
    assert lib.ab_mvn_sample(h, None, m, m, None, 0.0, 5, 1, P(out), ctypes.byref(info)) == -1
    assert lib.ab_mvn_sample(h, P(good), m, m, None, 0.0, 5, 1, None, ctypes.byref(info)) == -1
    tq = torch.from_numpy(rng.uniform(-1, 1, size=(m, 3))).cuda()
    mu = torch.empty(m, dtype=torch.float64, device="cuda")
    cov = torch.empty((m, m), dtype=torch.float64, device="cuda")
    assert lib.ab_gp_predict_cov(h, P(tq), m, P(mu), P(cov), m - 1) == -1
    assert lib.ab_gp_predict_cov(h, P(tq), m, None, P(cov), m) == -1
    # a padded leading dimension: the same bits in the leading m x m block, the padding untouched
    mu_r, cov_r = g.predict(y, tq)                          # also sets the targets of the handle
    wide = torch.full((m, m + 3), -5.0, dtype=torch.float64, device="cuda")
    assert lib.ab_gp_predict_cov(h, P(tq), m, P(mu), P(wide), m + 3) == 0
    np.testing.assert_array_equal(wide[:, :m].cpu().numpy(), cov_r.cpu().numpy())
    assert torch.all(wide[:, m:] == -5.0)
    # duplicated queries: Sigma is singular; the jitter ladder draws with a warning, jitter=0 raises
    t = np.vstack([np.repeat(rng.uniform(-1, 1, size=(1, 3)), 16, axis=0), rng.uniform(-1, 1, size=(8, 3))])
    with pytest.warns(RuntimeWarning, match="jitter"):
        dr = g.sample_conditional(y, t, size=4, seed=3)
    assert dr.shape == (4, 24) and np.all(np.isfinite(dr))
    with pytest.raises(np.linalg.LinAlgError):
        g.sample_conditional(y, t, size=4, seed=3, jitter=0.0)
    with pytest.raises(ValueError):
        g.sample_conditional(y, t, size=0)


def test_pickle_and_copy_after_return_cov():
    import copy
    o, g, X, y, rng = make_pair("ExpSquaredKernel", 500, 3, seed=31)
    t = rng.uniform(-1, 1, size=(150, 3))
    mu, cov = g.predict(y, t)
    for g2 in (pickle.loads(pickle.dumps(g)), copy.copy(g)):
        mu2, cov2 = g2.predict(y, t)
        np.testing.assert_array_equal(mu2, mu)
        np.testing.assert_array_equal(cov2, cov)
        np.testing.assert_array_equal(g2.sample_conditional(y, t, size=3, seed=5, jitter=1e-8),
                                      g.sample_conditional(y, t, size=3, seed=5, jitter=1e-8))
