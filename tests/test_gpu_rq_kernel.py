"""GPU parity of the rational quadratic kernel (george's RationalQuadraticKernel, kernel id 3) on every
device path: covariance, log-likelihood and gradient (incl. d/dlog alpha), prediction and its gradient,
the few-query kernels, append_point, batched CV, the sampler and the nested walks, against the CPU
reference in tests/rq_oracle.py on seeded inputs.  Tolerances are those of test_gpu_gp.py."""
import os
import pickle
import sys

import numpy as np
import pytest

from oracle import emcee as oem, nested as onest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import rq_oracle as rq  # noqa: E402

pytestmark = pytest.mark.gpu

RQ = "RationalQuadraticKernel"


def rq_kernel(log_alpha, log_M, d):
    import alabi_b200 as ab
    metric = np.exp(log_M[0]) if d == 1 else np.exp(log_M)      # d = 1: the isotropic (scalar) metric
    return ab.kernels.RationalQuadraticKernel(log_alpha, metric=metric, ndim=d)


def make_pair(n, d, log_alpha, seed=0, white_noise=-8.0, lo=-1.0, hi=1.0, log_M=None):
    import alabi_b200 as ab
    rng = np.random.default_rng(seed)
    X = rng.uniform(lo, hi, size=(n, d))
    y = np.sin(X.sum(axis=1)) + 0.3 * np.cos(2.0 * X[:, 0]) + 0.05 * rng.normal(size=n)
    if log_M is None:
        log_M = np.full(d, 0.3) if d == 1 else rng.uniform(-0.5, 0.8, size=d)
    o = rq.make_gp(RQ, X, y, log_M, amp=np.var(y), white_noise=white_noise, log_alpha=log_alpha)
    g = ab.GP(kernel=rq_kernel(log_alpha, log_M, d) * np.var(y), fit_mean=True, mean=np.median(y),
              white_noise=white_noise, fit_white_noise=True)
    g.compute(X)
    return o, g, X, y, rng


def rel_to_scale(a, b):
    """Largest difference relative to the largest |b|.  The predictive mean of these targets crosses zero
    (min |mu| / max |mu| is 1e-5 .. 3e-3 on every input set here), and near a zero each entry carries the
    absolute error of the solve, not a relative one: at N = 150, d = 1, log_alpha = -2 (cond(K) = 1.3e5)
    the LAPACK reference itself is 4e-13 from an extended-precision solve, 2e-10 of the smallest |mu|."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


@pytest.mark.parametrize("n,d,log_alpha", [(150, 1, -2.0), (150, 3, 0.0), (150, 20, 3.0), (1000, 3, 3.0),
                                           (1000, 10, -2.0), (1000, 20, 0.0), (4001, 1, 3.0), (4001, 10, 0.0),
                                           (4001, 20, -2.0)])
def test_matrix_loglike_grad_predict(n, d, log_alpha):
    o, g, X, y, rng = make_pair(n, d, log_alpha, seed=n + d)
    assert g.get_parameter_names() == o.get_parameter_names()
    np.testing.assert_allclose(g.get_parameter_vector(), o.get_parameter_vector(), rtol=1e-14, atol=1e-15)
    sub = X[:min(n, 600)]
    np.testing.assert_allclose(g.kernel.get_value(sub, X), o.get_matrix(sub, X), rtol=1e-12, atol=1e-300)
    ll_o, ll_g = o.log_likelihood(y), g.log_likelihood(y)
    assert abs(ll_g - ll_o) <= 1e-9 * abs(ll_o), (ll_g, ll_o)
    assert abs(g.solver.log_determinant - o.log_determinant) <= 1e-9 * abs(o.log_determinant) + 1e-9
    go, gg = o.grad_log_likelihood(y), g.grad_log_likelihood(y)
    assert len(gg) == len(go) == len(o.get_parameter_vector())
    scale = np.maximum(np.abs(go), 1e-6 * np.max(np.abs(go)))
    assert np.max(np.abs(gg - go) / scale) < 1e-7, (gg, go)
    amp = np.exp(o.log_const)
    t = rng.uniform(-1.1, 1.1, size=(3000, d))
    mu_o, var_o = o.predict(y, t, return_var=True)
    mu_g, var_g = g.predict(y, t, return_var=True)
    assert rel_to_scale(mu_g, mu_o) < 1e-9
    assert np.max(np.abs(var_g - var_o)) < 1e-9 * amp
    mu_p, var_p, dmu_g, dvar_g = g.predict_grad(y, t[:200])
    np.testing.assert_array_equal(mu_p, mu_g[:200])
    dmu_o, dvar_o = o.predict_grad(y, t[:40])
    assert np.max(np.abs(dmu_g[:40] - dmu_o)) <= 1e-8 * np.max(np.abs(dmu_o))
    assert np.max(np.abs(dvar_g[:40] - dvar_o)) <= 1e-8 * max(np.max(np.abs(dvar_o)), 1e-6 * amp)
    # a new log_alpha alone marks the factor stale and is refactorised
    p = g.get_parameter_vector()
    p[3] += 0.5
    o.set_parameter_vector(p)
    g.set_parameter_vector(p)
    ll_o, ll_g = o.log_likelihood(y), g.log_likelihood(y)
    assert abs(ll_g - ll_o) <= 1e-9 * abs(ll_o)


@pytest.mark.parametrize("n,d,log_alpha", [(150, 1, 0.0), (1000, 3, -2.0), (4001, 10, 3.0)])
def test_few_query_path_reproduces_batched_bits(n, d, log_alpha):
    o, g, X, y, rng = make_pair(n, d, log_alpha, seed=n + 3)
    t = rng.uniform(-1.05, 1.05, size=(3000, d))
    t[3] = X[7]
    mu_big, var_big = g.predict(y, t, return_var=True)
    big = g.predict_grad(y, t[:300])
    hd = g._hd
    for m in (1, 3, 8):
        hd.lib.ab_gp_set_few_query_path(hd.h, 1)
        mu_f, var_f = g.predict(y, t[:m], return_var=True)
        few = g.predict_grad(y, t[:m])
        hd.lib.ab_gp_set_few_query_path(hd.h, 0)
        mu_b, var_b = g.predict(y, t[:m], return_var=True)
        bat = g.predict_grad(y, t[:m])
        hd.lib.ab_gp_set_few_query_path(hd.h, 1)
        np.testing.assert_array_equal(mu_f, mu_b)
        np.testing.assert_array_equal(var_f, var_b)
        np.testing.assert_array_equal(mu_f, mu_big[:m])
        np.testing.assert_array_equal(var_f, var_big[:m])
        for a, b_, c in zip(few, bat, big):
            np.testing.assert_array_equal(a, b_)
            np.testing.assert_array_equal(a, c[:m])


@pytest.mark.parametrize("n0,nadd,d,log_alpha", [(126, 4, 3, 0.0), (1000, 3, 10, -2.0)])
def test_append_point_equals_refactorisation(n0, nadd, d, log_alpha):
    import alabi_b200 as ab
    o, g, X, y, rng = make_pair(n0 + nadd, d, log_alpha, seed=11)
    mk = lambda: ab.GP(kernel=rq_kernel(log_alpha, o.log_M, d) * (np.exp(o.log_const) * d), fit_mean=True, mean=o.mean,
                       white_noise=o.white_noise, fit_white_noise=True)
    ga = mk()
    ga.compute(X[:n0])
    t = rng.uniform(-1, 1, size=(300, d))
    for k in range(nadd):
        ga.append_point(X[n0 + k])
        m = n0 + k + 1
        gf = mk()
        gf.compute(X[:m])
        oo = rq.OracleGP(RQ, d, o.log_M, log_const=o.log_const, mean=o.mean, fit_mean=True, white_noise=o.white_noise,
                         fit_white_noise=True, log_alpha=log_alpha).compute(X[:m])
        ll_a, ll_f, ll_o = ga.log_likelihood(y[:m]), gf.log_likelihood(y[:m]), oo.log_likelihood(y[:m])
        assert abs(ll_a - ll_f) <= 1e-10 * abs(ll_f)
        assert abs(ll_a - ll_o) <= 1e-9 * abs(ll_o)
        mu_a, var_a = ga.predict(y[:m], t, return_var=True)
        mu_f, var_f = gf.predict(y[:m], t, return_var=True)
        assert rel_to_scale(mu_a, mu_f) < 1e-10
        assert np.max(np.abs(var_a - var_f)) < 1e-10 * np.exp(o.log_const)


@pytest.mark.parametrize("n,d", [(150, 1), (1000, 3), (333, 10)])
def test_cv_batch_matches_oracle_folds(n, d):
    from sklearn.model_selection import KFold
    o, g, X, y, rng = make_pair(n, d, 0.5, seed=n + 3 * d)
    base = g.get_parameter_vector()
    assert g.get_parameter_names()[3] == "kernel:k2:log_alpha"
    ncand, k = 5, 5
    cands = base + rng.normal(0, 0.3, size=(ncand, len(base)))
    cands[0] = base
    cands[1, 3] = -2.0                                     # log_alpha across the range
    cands[2, 3] = 3.0
    folds, job_cand = [], []
    for c in range(ncand):
        for tr, va in KFold(n_splits=k, shuffle=True, random_state=c).split(X):
            folds.append((tr, va))
            job_cand.append(c)
    preds, lls, status = g.cv_batch(X, y, cands, folds, job_cand=job_cand)
    np.testing.assert_array_equal(g.get_parameter_vector(), base)
    assert np.all(status == 0)
    for b, (tr, va) in enumerate(folds):
        oc = rq.make_gp(RQ, X[tr], y[tr], np.zeros(d), amp=1.0, compute=False, log_alpha=0.0)
        oc.set_parameter_vector(cands[job_cand[b]])
        oc.compute(X[tr])
        ll_o = oc.log_likelihood(y[tr])
        mu_o = oc.predict(y[tr], X[va])
        assert abs(lls[b] - ll_o) <= 1e-9 * abs(ll_o), (b, lls[b], ll_o)
        np.testing.assert_allclose(preds[b], mu_o, rtol=1e-8, atol=1e-8 * np.max(np.abs(mu_o)))


def test_large_alpha_approaches_exp_squared():
    """(1 + x)^(-alpha) -> exp(-r^2 / 2) as alpha -> inf; the difference is below r^4 / (8 alpha)
    (+ rounding) at log_alpha = 12, with the device's own ExpSquared matrix as the yardstick."""
    import alabi_b200 as ab
    rng = np.random.default_rng(12)
    d = 4
    X = rng.uniform(-1, 1, size=(700, d))
    log_M = rng.uniform(-0.5, 0.5, size=d)
    k_rq = ab.kernels.RationalQuadraticKernel(12.0, metric=np.exp(log_M), ndim=d).get_value(X)
    k_se = ab.kernels.ExpSquaredKernel(metric=np.exp(log_M), ndim=d).get_value(X)
    r2 = rq.ogp.scaled_sqdist(X, X, log_M)
    bound = r2 * r2 / (8.0 * np.exp(12.0)) + 1e-15
    assert np.all(np.abs(k_rq - k_se) <= bound)
    assert np.max(np.abs(k_rq - k_se)) > 0.0


def _surrogate(n, d, seed, log_alpha):
    import alabi_b200 as ab
    from alabi_b200.ensemble import SurrogateLogProb
    rng = np.random.default_rng(seed)
    b = np.array([(-2.0, 2.0)] * d)
    X = rng.uniform(b[:, 0], b[:, 1], size=(n, d))
    y = -0.5 * np.sum((X / 0.7) ** 2, axis=1) + 0.3 * np.sin(2.0 * X[:, 0])
    log_M = np.full(d, 1.0)
    o = rq.make_gp(RQ, X, y, log_M, amp=np.var(y), white_noise=-8.0, log_alpha=log_alpha)
    g = ab.GP(kernel=rq_kernel(log_alpha, log_M, d) * np.var(y), fit_mean=True, mean=np.median(y), white_noise=-8.0,
              fit_white_noise=True)
    g.compute(X)
    return g, o, X, y, rng, b, SurrogateLogProb


@pytest.mark.parametrize("n,d,nw,nsteps,log_alpha", [(300, 3, 32, 40, 0.0), (8192, 10, 67, 8, -2.0)])
def test_sampler_chain_replays_on_the_cpu(n, d, nw, nsteps, log_alpha):
    """A resident training set, and a streamed one (N = 8192, d = 10, few walkers: spread mode)."""
    from alabi_b200.ensemble import EnsembleSampler
    g, o, X, y, rng, b, SLP = _surrogate(n, d, 17, log_alpha)
    lp = SLP(g, y, b)

    def lp_oracle(q):
        q = np.atleast_2d(q)
        inside = np.all((q > b[:, 0]) & (q < b[:, 1]), axis=1)
        return np.where(inside, o.predict(y, q), -np.inf)
    p0 = rng.uniform(-1.5, 1.5, size=(nw, d))
    seed = 987654321
    s = EnsembleSampler(nw, d, lp, seed=seed)
    s.run_mcmc(p0, nsteps)
    chain, lps, nacc, _ = oem.replay_device_chain(p0, lp_oracle, nsteps, seed)
    np.testing.assert_allclose(s.get_chain(), chain, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(s.get_log_prob(), lps, rtol=1e-9, atol=1e-9)
    assert np.array_equal(s._naccepted, nacc) and nacc.sum() > 0


def test_nested_walk_replays_on_the_cpu():
    from alabi_b200.nested import DeviceWalker
    d, nchains = 3, 37
    g, o, X, y, rng, b, SLP = _surrogate(500, d, 5, 1.0)
    lp = SLP(g, y, b, y_scale=1.5, y_offset=-0.25)
    like_o = lambda t: o.predict(y, np.atleast_2d(t)) * 1.5 - 0.25
    w = DeviceWalker(lp, b, seed=424242)
    u0 = rng.uniform(0.2, 0.8, size=(nchains, d))
    th0 = w.transform(u0)
    l0 = like_o(th0)
    np.testing.assert_allclose(w.like(th0), l0, rtol=1e-9, atol=1e-9)
    lmin = float(np.quantile(l0, 0.3))
    A = rng.normal(size=(d, d))
    chol = np.linalg.cholesky(A @ A.T / d + 0.5 * np.eye(d)) * 0.08
    walks, scale = 12, 0.9
    cnt = w.counter
    u, th, ll, acc = w.walk(u0, th0, l0, lmin, scale, chol, walks)
    ur, thr, llr, naccr, margin = onest.replay_walk(u0, th0, l0, lmin, scale, chol, walks, 424242, cnt, w.transform, like_o)
    assert margin > 1e-7
    np.testing.assert_allclose(u, ur, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(th, thr, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(ll, llr, rtol=1e-9, atol=1e-9)
    assert 0.02 < acc < 0.98


def test_set_kernel_rq_rejects_bad_alpha_and_set_kernel_rejects_id_3():
    import ctypes
    import torch
    from alabi_b200 import _lib
    from alabi_b200.gp import _Handle
    hd = _Handle(torch.cuda.current_device())
    x = torch.zeros((4, 2), dtype=torch.float64, device="cuda")
    assert hd.lib.ab_gp_set_inputs(hd.h, _lib.ptr(x), 4, 2) == 0
    lm = (ctypes.c_double * 2)(0.0, 0.0)
    assert hd.lib.ab_gp_set_kernel(hd.h, 3, 1.0, lm, 0.0, -8.0, 0.0) == -1
    for bad in (np.inf, 800.0, np.nan, -800.0):
        assert hd.lib.ab_gp_set_kernel_rq(hd.h, 1.0, bad, lm, 0.0, -8.0, 0.0) == -1
    assert hd.lib.ab_gp_set_kernel_rq(hd.h, 1.0, 0.5, lm, 0.0, -8.0, 0.0) == 0
    assert hd.lib.ab_version() == 100


def lnlike(theta):
    theta = np.asarray(theta).flatten()
    return -0.5 * np.sum((theta / np.array([0.6, 0.9])) ** 2)


@pytest.mark.parametrize("hyperopt", ["ml", "cv"])
def test_surrogate_model_workflow(tmp_path, hyperopt):
    import alabi_b200 as ab
    np.random.seed(3)
    sm = ab.SurrogateModel(lnlike_fn=lnlike, bounds=[(-3.0, 3.0), (-3.0, 3.0)], savedir=str(tmp_path), cache=True,
                           verbose=False)
    sm.init_samples(ntrain=60, ntest=20, sampler="lhs")
    kw = dict(hyperopt_method=hyperopt, gp_nopt=2)
    if hyperopt == "cv":
        kw.update(cv_n_candidates=12, cv_stage2_candidates=6, cv_stage3_candidates=4, gp_amp_rng=[-2, -1])
    test_mse = sm.init_gp(kernel=RQ, fit_amp=True, fit_mean=True, fit_white_noise=False, white_noise=-10,
                          gp_scale_rng=[-1, 3], **kw)
    assert np.isfinite(test_mse)
    assert "kernel:k2:log_alpha" in sm.param_names_full
    la = sm.gp.get_parameter_dict()["kernel:k2:log_alpha"]
    assert np.isfinite(la) and -2.0 <= la <= 2.0
    sm.active_train(niter=4, algorithm="bape", gp_opt_freq=2, nopt=1, show_progress=False)
    assert sm.ntrain == 64
    t = np.random.uniform(-2.5, 2.5, size=(50, 2))
    mu = sm.surrogate_log_likelihood(t)
    truth = np.array([lnlike(p) for p in t])
    assert np.sqrt(np.mean((mu - truth) ** 2)) < 0.5 * np.std(truth)
    sm.run_emcee(nwalkers=40, nsteps=200, min_ess=50)
    assert np.all(np.isfinite(sm.emcee_samples)) and 0.1 < sm.acc_frac < 0.95
    sm2 = pickle.loads(pickle.dumps(sm))
    np.testing.assert_array_equal(sm2.surrogate_log_likelihood(t), mu)
    assert sm2.gp.get_parameter_dict()["kernel:k2:log_alpha"] == sm.gp.get_parameter_dict()["kernel:k2:log_alpha"]
