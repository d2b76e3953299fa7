"""GPU parity: K1 covariance, K2 Cholesky / logL / gradient, K3 predict, K4
utilities against the CPU oracle on identical seeded inputs (through the
C ABI via alabi_b200.GP).  Tolerances follow north_star: 1e-9 relative in FP64
on well-conditioned problems."""
import numpy as np
import pytest

from oracle import gp as ogp, utility as ou, benchmarks as ob

pytestmark = pytest.mark.gpu

KINDS = ["ExpSquaredKernel", "Matern32Kernel", "Matern52Kernel"]


def make_pair(kind, n, d, seed=0, white_noise=-6.0, fit_amp=True, log_M=None):
    import alabi_b200 as ab
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1, 1, size=(n, d))
    y = np.sin(X.sum(axis=1)) + 0.3 * np.cos(2.0 * X[:, 0]) + 0.05 * rng.normal(size=n)
    if log_M is None:
        log_M = rng.uniform(-0.5, 0.8, size=d)
    amp = np.var(y) if fit_amp else None
    o = ogp.make_gp(kind, X, y, log_M, amp=amp, white_noise=white_noise, compute=True)
    k = getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d)
    if fit_amp:
        k = k * np.var(y)
    g = ab.GP(kernel=k, fit_mean=True, mean=np.median(y), white_noise=white_noise, fit_white_noise=True)
    g.compute(X)
    return o, g, X, y, rng


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,d", [(50, 2), (150, 2), (333, 5), (1000, 3), (1300, 10)])
def test_names_vector_loglike_grad(kind, n, d):
    o, g, X, y, rng = make_pair(kind, n, d, seed=n + d)
    assert g.get_parameter_names() == o.get_parameter_names()
    np.testing.assert_allclose(g.get_parameter_vector(), o.get_parameter_vector(), rtol=1e-14, atol=1e-15)
    ll_o, ll_g = o.log_likelihood(y), g.log_likelihood(y)
    assert abs(ll_g - ll_o) <= 1e-9 * abs(ll_o), (ll_g, ll_o)
    assert abs(g.solver.log_determinant - o.log_determinant) <= 1e-10 * abs(o.log_determinant) + 1e-9
    go, gg = o.grad_log_likelihood(y), g.grad_log_likelihood(y)
    scale = np.maximum(np.abs(go), 1e-6 * np.max(np.abs(go)))
    assert np.max(np.abs(gg - go) / scale) < 1e-7, (gg, go)
    # a new hyper-vector marks the model dirty and is refactorised
    p = o.get_parameter_vector() + rng.normal(0, 0.1, size=len(o.get_parameter_vector()))
    o.set_parameter_vector(p)
    g.set_parameter_vector(p)
    ll_o, ll_g = o.log_likelihood(y), g.log_likelihood(y)
    assert abs(ll_g - ll_o) <= 1e-9 * abs(ll_o)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,d,m", [(50, 2, 1), (150, 2, 7), (700, 4, 1000), (1100, 10, 5000)])
def test_predict_mean_var(kind, n, d, m):
    o, g, X, y, rng = make_pair(kind, n, d, seed=7 * n + d)
    t = rng.uniform(-1.1, 1.1, size=(m, d))
    mu_o, var_o = o.predict(y, t, return_var=True)
    mu_g = g.predict(y, t, return_cov=False)
    mu_g2, var_g = g.predict(y, t, return_var=True)
    # mean-only and mean+var paths share one fixed summation order
    np.testing.assert_array_equal(mu_g, mu_g2)
    assert rel(mu_g, mu_o) < 1e-9
    amp = np.exp(o.log_const)
    assert np.max(np.abs(var_g - var_o)) < 1e-9 * amp, np.max(np.abs(var_g - var_o)) / amp
    # alpha, K^-1 and kernel values as alabi/utility.py reads them
    assert rel(g._alpha, o._alpha) < 1e-8
    if n <= 700:
        Ki = g.solver.get_inverse()
        np.testing.assert_allclose(Ki, o.get_inverse(), rtol=0, atol=1e-9 * np.max(np.abs(Ki)))
        np.testing.assert_allclose(g.kernel.get_value(t[:5], X), o.get_matrix(t[:5], X), rtol=1e-12, atol=1e-300)


def test_device_tensor_io_and_no_amp():
    import torch
    o, g, X, y, rng = make_pair("Matern32Kernel", 400, 3, seed=5, fit_amp=False)
    assert g.get_parameter_names()[2] == "kernel:metric:log_M_0_0"
    t = rng.uniform(-1, 1, size=(300, 3))
    mu, var = g.predict(y, torch.from_numpy(t).cuda(), return_var=True)
    mu_o, var_o = o.predict(y, t, return_var=True)
    assert rel(mu.cpu().numpy(), mu_o) < 1e-9 and np.max(np.abs(var.cpu().numpy() - var_o)) < 1e-9


def test_not_positive_definite_paths():
    import alabi_b200 as ab
    rng = np.random.default_rng(1)
    X = rng.uniform(-1, 1, size=(200, 2))
    X[1] = X[0]
    y = rng.normal(size=200)
    k = ab.kernels.ExpSquaredKernel(metric=[1.0, 1.0], ndim=2) * 2.0     # amp = 1.0 exactly
    g = ab.GP(kernel=k, mean=0.0, white_noise=-80.0)
    with pytest.raises(np.linalg.LinAlgError):
        g.compute(X)
    assert g.log_likelihood(y, quiet=True) == -np.inf
    assert np.all(g.grad_log_likelihood(y, quiet=True) == 0.0)


@pytest.mark.parametrize("algo", ["bape", "agp", "jones"])
def test_utility_argmin_matches_oracle(algo):
    o, g, X, y, rng = make_pair("ExpSquaredKernel", 300, 2, seed=11)
    bounds = np.array([(-1.0, 1.0), (-1.0, 1.0)])
    cand = rng.uniform(-1.2, 1.2, size=(20000, 2))
    mu_o, var_o = o.predict(y, cand, return_var=True)
    u_o = ou.utility(algo, mu_o, var_o, ou.in_bounds(cand, bounds), y_best=y.max())
    idx, val, u_g = g.utility_argmin(y, cand, bounds, algorithm=algo, y_best=y.max(), return_values=True)
    u_g = u_g.cpu().numpy()
    fin = np.isfinite(u_o)
    assert np.array_equal(np.isfinite(u_g), fin)
    assert np.array_equal(np.isposinf(u_g), np.isposinf(u_o))
    np.testing.assert_allclose(u_g[fin], u_o[fin], rtol=1e-7, atol=1e-9)
    want = int(np.argmin(np.where(fin, u_o, np.inf)))
    assert idx == want and val == u_g[idx]


def test_pickle_copy_roundtrip():
    import copy
    import pickle
    o, g, X, y, rng = make_pair("Matern52Kernel", 260, 2, seed=3)
    t = rng.uniform(-1, 1, size=(50, 2))
    ref = g.predict(y, t, return_cov=False)
    for h in (pickle.loads(pickle.dumps(g)), copy.copy(g), copy.deepcopy(g)):
        np.testing.assert_array_equal(h.predict(y, t, return_cov=False), ref)


@pytest.mark.parametrize("n", [2048, 4096])
def test_large_factor_matches_lapack(n):
    """The dataflow factor at sizes with many tile columns against LAPACK: the
    log-likelihood and L, and alpha against the oracle's cho_solve.  Each tile is
    summed in one long-K pass, a different rounding order from LAPACK's."""
    import alabi_b200 as ab
    c = ob.make_config("c4", n_override=n)
    X, y = c["X"] / 3.0, c["y"]
    d = X.shape[1]
    log_M = np.zeros(d) + 1.0
    o = ogp.make_gp("ExpSquaredKernel", X, y, log_M, amp=np.var(y), white_noise=-6.0)
    g = ab.GP(kernel=ab.kernels.ExpSquaredKernel(metric=np.exp(log_M), ndim=d) * np.var(y),
              fit_mean=True, mean=np.median(y), white_noise=-6.0, fit_white_noise=True)
    g.compute(X)
    ll = g.log_likelihood(y)
    L, alpha = g.export_state()
    L, alpha = L.cpu().numpy(), alpha.cpu().numpy()
    ll_o = o.log_likelihood(y)
    assert abs(ll - ll_o) <= 1e-9 * abs(ll_o)
    Lo = o._factor[0].T
    assert np.max(np.abs(np.tril(L)[:n, :n] - Lo)) < 1e-9 * np.max(np.abs(Lo))
    o._compute_alpha(y)
    err = np.max(np.abs(alpha - o._alpha)) / np.max(np.abs(o._alpha))
    assert err <= 1e-9, err


@pytest.mark.parametrize("kind,n0,nadd,d", [("ExpSquaredKernel", 60, 5, 2), ("Matern32Kernel", 126, 5, 3),
                                            ("Matern52Kernel", 383, 4, 2), ("ExpSquaredKernel", 1000, 3, 5)])
def test_append_point_equals_refactorisation(kind, n0, nadd, d):
    """Bordered Cholesky update (ab_gp_append_point) against a fresh factorisation of
    the extended training set and against the oracle, including the steps that cross
    a 128-row padding boundary."""
    o, g, X, y, rng = make_pair(kind, n0 + nadd, d, seed=11)
    import alabi_b200 as ab
    log_M = o.log_M
    mk = lambda: ab.GP(kernel=getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d) * (np.exp(o.log_const) * d),
                       fit_mean=True, mean=o.mean, white_noise=o.white_noise, fit_white_noise=True)
    ga = mk()
    ga.compute(X[:n0])
    t = rng.uniform(X.min(), X.max(), size=(300, d))
    for k in range(nadd):
        ga.append_point(X[n0 + k])
        m = n0 + k + 1
        gf = mk()
        gf.compute(X[:m])
        oo = ogp.OracleGP(kind, d, log_M, log_const=o.log_const, mean=o.mean, fit_mean=True,
                          white_noise=o.white_noise, fit_white_noise=True).compute(X[:m])
        ll_a, ll_f, ll_o = ga.log_likelihood(y[:m]), gf.log_likelihood(y[:m]), oo.log_likelihood(y[:m])
        assert abs(ll_a - ll_f) <= 1e-10 * abs(ll_f)
        assert abs(ll_a - ll_o) <= 1e-9 * abs(ll_o)
        mu_a, var_a = ga.predict(y[:m], t, return_var=True)
        mu_f, var_f = gf.predict(y[:m], t, return_var=True)
        assert rel(mu_a, mu_f) < 1e-10
        assert np.max(np.abs(var_a - var_f)) < 1e-10 * np.exp(o.log_const)
        ga_g, gf_g = ga.grad_log_likelihood(y[:m]), gf.grad_log_likelihood(y[:m])
        assert np.max(np.abs(ga_g - gf_g)) <= 1e-8 * np.max(np.abs(gf_g))
    La, _ = ga.export_state()
    Lf, _ = gf.export_state()
    m = n0 + nadd
    assert np.max(np.abs(np.tril(La.cpu().numpy())[:m, :m] - np.tril(Lf.cpu().numpy())[:m, :m])) < 1e-10 * float(Lf.abs().max())


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n,d,m", [(60, 1, 3), (300, 2, 40), (700, 5, 300), (1100, 10, 1500)])
def test_predict_grad(kind, n, d, m):
    """ab_gp_predict_grad: analytic d mu / dx, d sigma^2 / dx against the oracle's analytic
    form (1e-8) and against the reference's finite-difference construction (1e-4)."""
    if d == 1 and kind != "ExpSquaredKernel":
        pytest.skip("1-D covered once")
    o, g, X, y, rng = make_pair(kind, n, d, seed=5 * n + d)
    t = rng.uniform(-1.1, 1.1, size=(m, d))
    mu_g, var_g, dmu_g, dvar_g = g.predict_grad(y, t)
    mu_o, var_o = o.predict(y, t, return_var=True)
    amp = np.exp(o.log_const)
    assert rel(mu_g, mu_o) < 1e-9
    assert np.max(np.abs(var_g - var_o)) < 1e-9 * amp
    sub = slice(0, min(m, 60))
    dmu_o, dvar_o = o.predict_grad(y, t[sub])
    assert np.max(np.abs(dmu_g[sub] - dmu_o)) <= 1e-8 * np.max(np.abs(dmu_o))
    assert np.max(np.abs(dvar_g[sub] - dvar_o)) <= 1e-8 * max(np.max(np.abs(dvar_o)), 1e-6 * amp)
    dmu_f, dvar_f = o.predict_grad(y, t[:5], h=1e-6)
    assert np.max(np.abs(dmu_g[:5] - dmu_f)) <= 1e-4 * np.max(np.abs(dmu_f))
    assert np.max(np.abs(dvar_g[:5] - dvar_f)) <= 1e-4 * max(np.max(np.abs(dvar_f)), 1e-6 * amp)


def test_grad_utilities_match_reference_expressions():
    """grad_agp_utility / grad_bape_utility (alabi/utility.py:704-850) on the device
    gradients, against the same expressions on the oracle's gradients, and against a
    finite difference of the utility itself where the reference's expression is its
    true derivative (bape)."""
    from alabi_b200 import utility as ut
    o, g, X, y, rng = make_pair("ExpSquaredKernel", 250, 2, seed=77)
    b = np.array([(-1.2, 1.2)] * 2)
    g._set_targets(y)
    g._y = y
    for th in rng.uniform(-1, 1, size=(4, 2)):
        dmu_o, dvar_o = o.predict_grad(y, th[None, :])
        _, var_o = o.predict(y, th[None, :], return_var=True)
        ga = ut.grad_agp_utility(th, g, b)
        np.testing.assert_allclose(ga, -(dmu_o[0] + 0.5 * dvar_o[0]), rtol=1e-7, atol=1e-10)
        gb = ut.grad_bape_utility(th, g, b)
        e = np.exp(var_o[0])
        np.testing.assert_allclose(gb, -2.0 * dmu_o[0] - (1.0 + e / (e - 1.0)) * dvar_o[0], rtol=1e-6, atol=1e-9)
        pg = lambda xs: g.predict(y, xs, return_var=True)
        h = 1e-5
        fd = np.array([(ut.bape_utility(th + h * np.eye(2)[k], pg, b) - ut.bape_utility(th - h * np.eye(2)[k], pg, b)) / (2 * h)
                       for k in range(2)])
        np.testing.assert_allclose(gb, fd, rtol=2e-4, atol=1e-6)
    assert np.all(np.isinf(ut.grad_agp_utility(np.array([5.0, 0.0]), g, b)))


def test_small_and_large_batches_give_identical_bits():
    """Few query tiles take the split-over-row-blocks variance kernel, large batches the
    one-CTA-per-tile kernel: same operations in the same order, so a query gets the same
    mean and variance bits whatever batch it arrives in (one-point acquisition calls vs
    candidate sweeps)."""
    o, g, X, y, rng = make_pair("Matern52Kernel", 700, 3, seed=41)
    t = rng.uniform(-1, 1, size=(12000, 3))
    mu_big, var_big = g.predict(y, t, return_var=True)
    for m in (1, 7, 130, 1000):
        mu_s, var_s = g.predict(y, t[:m], return_var=True)
        np.testing.assert_array_equal(mu_s, mu_big[:m])
        np.testing.assert_array_equal(var_s, var_big[:m])
    mu_o, var_o = o.predict(y, t[:50], return_var=True)
    assert rel(mu_big[:50], mu_o) < 1e-9 and np.max(np.abs(var_big[:50] - var_o)) < 1e-9 * np.exp(o.log_const)


@pytest.mark.parametrize("kind,n,d", [("ExpSquaredKernel", 50, 2), ("Matern32Kernel", 150, 2), ("Matern52Kernel", 333, 5),
                                      ("ExpSquaredKernel", 1000, 3), ("Matern32Kernel", 1300, 10), ("Matern52Kernel", 2100, 12)])
def test_few_query_path_reproduces_batched_bits(kind, n, d):
    """m <= 8 queries run on kernels that spread one query over the GPU (few_cross / few_gemv /
    few_finish): same mean and variance BITS as the batched kernels (path switched off, and the
    same queries inside a large batch), for mean-only and mean+variance calls, and parity with
    the oracle to 1e-9."""
    o, g, X, y, rng = make_pair(kind, n, d, seed=n + 3)
    t = rng.uniform(-1.05, 1.05, size=(3000, d))
    t[3] = X[7]                                         # a training point (variance ~ 0)
    mu_big, var_big = g.predict(y, t, return_var=True)
    hd = g._hd
    for m in (1, 2, 3, 4, 5, 8):
        hd.lib.ab_gp_set_few_query_path(hd.h, 1)
        mu_f, var_f = g.predict(y, t[:m], return_var=True)
        mu_only = g.predict(y, t[:m], return_cov=False)
        hd.lib.ab_gp_set_few_query_path(hd.h, 0)
        mu_b, var_b = g.predict(y, t[:m], return_var=True)
        hd.lib.ab_gp_set_few_query_path(hd.h, 1)
        np.testing.assert_array_equal(mu_f, mu_b)
        np.testing.assert_array_equal(var_f, var_b)
        np.testing.assert_array_equal(mu_f, mu_big[:m])
        np.testing.assert_array_equal(var_f, var_big[:m])
        np.testing.assert_array_equal(mu_only, mu_f)
    # gradients w.r.t. the query point (the default L-BFGS polish calls them one point at a time)
    big = g.predict_grad(y, t[:300])
    for m in (1, 3, 8):
        hd.lib.ab_gp_set_few_query_path(hd.h, 1)
        few = g.predict_grad(y, t[:m])
        hd.lib.ab_gp_set_few_query_path(hd.h, 0)
        bat = g.predict_grad(y, t[:m])
        hd.lib.ab_gp_set_few_query_path(hd.h, 1)
        for a, b_, c in zip(few, bat, big):
            np.testing.assert_array_equal(a, b_)
            np.testing.assert_array_equal(a, c[:m])
    # single queries taken from anywhere in the batch
    for i in (11, 257, 2999):
        mu1, var1 = g.predict(y, t[i:i + 1], return_var=True)
        assert mu1[0] == mu_big[i] and var1[0] == var_big[i]
    mu_o, var_o = o.predict(y, t[:8], return_var=True)
    mu_f, var_f = g.predict(y, t[:8], return_var=True)
    assert rel(mu_f, mu_o) < 1e-9 and np.max(np.abs(var_f - var_o)) < 1e-9 * np.exp(o.log_const)
    # utilities over a handful of candidates take the same path
    b = np.array([(-1.0, 1.0)] * d)
    idx, val = g.utility_argmin(y, t[:6], b, algorithm="bape")
    inside = ou.in_bounds(t[:6], b)
    want = ou.utility("bape", mu_big[:6], var_big[:6], inside, 0.0)
    assert idx == ou.first_argmin(want)


def test_large_host_batch_overlapped_copies_identical():
    """Host-buffer predicts larger than one variance panel are processed panel by panel with
    the device -> host copies overlapped; the numbers must be the ones the device-tensor
    path returns for the same queries."""
    import torch
    o, g, X, y, rng = make_pair("Matern32Kernel", 300, 2, seed=9)
    m = 16 * 148 * 128 + 12345                      # more than the largest panel (16 waves)
    t = rng.uniform(-1, 1, size=(m, 2))
    mu_h, var_h = g.predict(y, t, return_var=True)
    mu_d, var_d = g.predict(y, torch.from_numpy(t).cuda(), return_var=True)
    np.testing.assert_array_equal(mu_h, mu_d.cpu().numpy())
    np.testing.assert_array_equal(var_h, var_d.cpu().numpy())
    mu_o, var_o = o.predict(y, t[-40:], return_var=True)
    assert rel(mu_h[-40:], mu_o) < 1e-9 and np.max(np.abs(var_h[-40:] - var_o)) < 1e-9 * np.exp(o.log_const)


@pytest.mark.parametrize("kind,nstart,reg", [("ExpSquaredKernel", 1, False), ("Matern52Kernel", 3, True)])
def test_optimize_gp_ml_restarts(kind, nstart, reg):
    """gp_utils.optimize_gp (alabi/gp_utils.py:251-447) drives the device objective and
    gradient; the same driver on the oracle GP from the same starts reaches the same
    regularised optimum."""
    from alabi_b200 import gp_utils, utility as ut
    o, g, X, y, rng = make_pair(kind, 220, 2, seed=5)
    P = len(g.get_parameter_vector())
    hp_bounds = [(-10.0, 10.0)] * P
    # hyper-prior box wider than the optimiser's: L-BFGS-B's first projected step lands ON its
    # bounds, where a strict prior of the same box returns -inf
    prior = lambda p: ut.lnprior_uniform(p, [(-20.0, 20.0)] * P)
    lidx = [i for i, nm in enumerate(g.get_parameter_names()) if "log_M" in nm]
    base = np.array(g.get_parameter_vector())
    p0 = base if nstart == 1 else np.vstack([base] + [base + rng.normal(0, 0.3, size=P) for _ in range(nstart - 1)])
    # (the reference's regularisation "gradient" is not the derivative of its term -- SURVEY a15 --
    # so a single regularised L-BFGS-B run may stop where it started; restarts pick by log-likelihood)
    obj = lambda gp_, p: gp_utils._nll(p, gp_, y, prior) + (gp_utils.regularization_term(p, lidx) if reg else 0.0)
    f0 = obj(g, base)
    gp_utils.optimize_gp(g, X, y, prior, p0, bounds=hp_bounds, lengthscale_indices=lidx, regularize=reg)
    gp_utils.optimize_gp(o, X, y, prior, p0, bounds=hp_bounds, lengthscale_indices=lidx, regularize=reg)
    pg, po = np.array(g.get_parameter_vector()), np.array(o.get_parameter_vector())
    fg, fo = obj(g, pg), obj(o, po)
    assert fg < f0 - 1e-3 and np.all(np.abs(pg) <= 10.0)
    # same optimum.  With the reference's inconsistent regulariser "gradient" (SURVEY a15) L-BFGS-B
    # stops where its line search gives up, and two FP64 paths whose gradients differ in the last
    # digits may give up a few 1e-5 (relative objective) apart: that much is allowed there
    tol = 1e-6 if not reg else 2e-4
    assert abs(fg - fo) <= tol * max(1.0, abs(fo)), (fg, fo)
    np.testing.assert_allclose(pg, po, rtol=0, atol=2e-3 if not reg else 0.1)
    # device objective at the oracle's optimum equals the oracle's value there (1e-9)
    assert abs(obj(g, po) - fo) <= 1e-9 * max(1.0, abs(fo))
    assert g.computed and abs(g.log_likelihood(y) - o.log_likelihood(y)) <= 1e-5 * abs(o.log_likelihood(y))


def test_shared_point_cache_serves_utility_and_gradient():
    """find_next_point's one-entry cache: the utility and its gradient at one point come from one
    predict_grad call, with the bits of separate predict / predict_grad calls."""
    from alabi_b200 import utility as ut
    from alabi_b200.core import _SharedPoint
    o, g, X, y, rng = make_pair("Matern32Kernel", 260, 3, seed=12)
    b = np.array([(-1.0, 1.0)] * 3)
    sp = _SharedPoint(g, y)
    calls = {"n": 0}
    real = g.predict_grad

    def counting(yy, xs):
        calls["n"] += 1
        return real(yy, xs)
    g.predict_grad = counting
    g._set_targets(y)
    for x in rng.uniform(-0.9, 0.9, size=(5, 3)):
        u_direct = ut.bape_utility(x, lambda q: g.predict(y, q, return_var=True), b)
        n0 = calls["n"]
        u = ut.bape_utility(x, sp.predict, b)
        gr = ut.grad_bape_utility(x, sp, b)
        assert calls["n"] == n0 + 1                       # one device call for both
        gr_direct = ut.grad_bape_utility(x, g, b)
        assert u == u_direct
        np.testing.assert_array_equal(gr, gr_direct)
    mu, var = sp.predict(X[:10])                          # batches pass straight through
    assert mu.shape == (10,) and var.shape == (10,)


@pytest.mark.parametrize("kind,n,d", [("ExpSquaredKernel", 150, 2), ("Matern32Kernel", 1000, 3), ("Matern52Kernel", 333, 5)])
def test_cv_batch_matches_oracle_folds(kind, n, d):
    """k-fold CV as one batched device job (ab_gp_cv_batch): per (candidate, fold) the predictions at
    the held-out rows, the log-likelihood and the fold MSE equal the oracle doing the SAME folds;
    a candidate whose covariance matrix is not positive definite fails like the reference's worker;
    the batched scores equal the one-by-one device path."""
    import time
    from sklearn.model_selection import KFold
    from alabi_b200 import gp_utils, utility as ut
    o, g, X, y, rng = make_pair(kind, n, d, seed=n + 3 * d, white_noise=-8.0)
    base = g.get_parameter_vector()
    ncand, k = 6, 5
    cands = base + rng.normal(0, 0.3, size=(ncand, len(base)))
    cands[0] = base
    folds, job_cand = [], []
    for c in range(ncand):
        for tr, va in KFold(n_splits=k, shuffle=True, random_state=c).split(X):
            folds.append((tr, va))
            job_cand.append(c)
    preds, lls, status = g.cv_batch(X, y, cands, folds, job_cand=job_cand)
    np.testing.assert_array_equal(g.get_parameter_vector(), base)           # the GP itself is untouched
    assert np.all(status == 0)
    for b, (tr, va) in enumerate(folds):
        oc = ogp.make_gp(kind, X[tr], y[tr], np.zeros(d), amp=1.0, compute=False)
        oc.set_parameter_vector(cands[job_cand[b]])
        oc.compute(X[tr])
        ll_o = oc.log_likelihood(y[tr])
        mu_o = oc.predict(y[tr], X[va])
        assert abs(lls[b] - ll_o) <= 1e-9 * abs(ll_o), (b, lls[b], ll_o)
        np.testing.assert_allclose(preds[b], mu_o, rtol=1e-8, atol=1e-8 * np.max(np.abs(mu_o)))
        assert abs(np.mean((y[va] - preds[b]) ** 2) - np.mean((y[va] - mu_o) ** 2)) <= 1e-7 * np.mean((y[va] - mu_o) ** 2) + 1e-14
    # a candidate that cannot be factorised: white noise -80 on duplicated points
    Xd, yd = X.copy(), y.copy()
    Xd[1] = Xd[0]
    bad = base.copy()
    bad[1] = -80.0
    folds2 = [(np.arange(n - 20), np.arange(n - 20, n))] * 2
    p2, l2, s2 = g.cv_batch(Xd, yd, np.array([base, bad]), folds2, job_cand=[0, 1])
    assert s2[0] == 0 and np.isfinite(l2[0]) and s2[1] > 0 and l2[1] == -np.inf and np.all(np.isnan(p2[1]))
    # the stage evaluation used by optimize_gp_kfold_cv: batched == one-by-one
    t0 = time.time()
    sb = gp_utils._evaluate_candidates(g, X, y, ut.no_scaler, cands, k, "mse", "exponential", 1.0, batched=True, random_state=7)
    tb = time.time() - t0
    t0 = time.time()
    ss = gp_utils._evaluate_candidates(g, X, y, ut.no_scaler, cands, k, "mse", "exponential", 1.0, batched=False, random_state=7)
    ts = time.time() - t0
    np.testing.assert_allclose(sb, ss, rtol=1e-7, atol=1e-14)
    print(f"cv stage of {ncand} x {k} jobs at n = {n}: batched {tb * 1e3:.1f} ms, one by one {ts * 1e3:.1f} ms")
