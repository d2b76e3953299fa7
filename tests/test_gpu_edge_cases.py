"""Edge cases of the GPU path (through the C ABI): smallest and ragged sizes, the
padding boundaries of the 128-row blocking, the maximum dimension, empty query
sets, duplicated training points, non-finite inputs, the ill-conditioned default
white noise, and both unit sizes of the sampler."""
import numpy as np
import pytest

from oracle import gp as ogp, emcee as oem

pytestmark = pytest.mark.gpu


def _pair(kind, X, y, log_M, wn=-6.0):
    import alabi_b200 as ab
    d = X.shape[1]
    o = ogp.make_gp(kind, X, y, log_M, amp=np.var(y) if len(y) > 1 and np.var(y) > 0 else 1.0, white_noise=wn)
    k = getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d) * (np.exp(o.log_const) * d)
    g = ab.GP(kernel=k, fit_mean=True, mean=o.mean, white_noise=wn, fit_white_noise=True)
    g.compute(X)
    return o, g


def _check(o, g, y, t, tol=1e-9):
    ll_o, ll_g = o.log_likelihood(y), g.log_likelihood(y)
    assert abs(ll_g - ll_o) <= tol * max(abs(ll_o), 1.0)
    mu_o, var_o = o.predict(y, t, return_var=True)
    mu_g, var_g = g.predict(y, t, return_var=True)
    assert np.max(np.abs(mu_g - mu_o)) <= tol * max(np.max(np.abs(mu_o)), 1e-3)
    assert np.max(np.abs(var_g - var_o)) <= tol * np.exp(o.log_const)
    go, gg = o.grad_log_likelihood(y), g.grad_log_likelihood(y)
    assert np.max(np.abs(gg - go)) <= 1e-7 * max(np.max(np.abs(go)), 1e-3)


@pytest.mark.parametrize("n", [1, 2, 3, 127, 128, 129, 255, 256, 257, 385])
def test_ragged_sizes_around_the_block_boundaries(n):
    rng = np.random.default_rng(n)
    X = rng.uniform(-1, 1, size=(n, 2))
    y = np.cos(X[:, 0]) + 0.5 * X[:, 1] + 0.01 * rng.normal(size=n)
    o, g = _pair("Matern32Kernel", X, y, np.array([0.2, -0.1]))
    _check(o, g, y, rng.uniform(-1, 1, size=(17, 2)))


# both ends of every compiled dimension bucket (2, 4, 8, 12, 16, 20, 24, 32)
@pytest.mark.parametrize("d", [1, 2, 3, 4, 5, 8, 9, 12, 13, 16, 17, 20, 21, 24, 25, 32])
def test_dimensions_up_to_the_maximum(d):
    rng = np.random.default_rng(d)
    n = 200
    X = rng.uniform(-1, 1, size=(n, d))
    y = np.sin(X.sum(axis=1)) + 0.01 * rng.normal(size=n)
    o, g = _pair("ExpSquaredKernel", X, y, rng.uniform(0.5, 1.5, size=d))
    t = rng.uniform(-1, 1, size=(33, d))
    _check(o, g, y, t)
    amp = np.exp(o.log_const)
    # one query (the few-query kernels)
    m1, v1 = g.predict(y, t[:1], return_var=True)
    mo, vo = o.predict(y, t[:1], return_var=True)
    assert abs(m1[0] - mo[0]) <= 1e-9 * max(abs(mo[0]), 1e-3) and abs(v1[0] - vo[0]) <= 1e-9 * amp
    # gradients of the mean and variance: few-query and batched kernels
    for tq in (t[:3], t):
        _, _, dmu_g, dvar_g = g.predict_grad(y, tq)
        dmu_o, dvar_o = o.predict_grad(y, tq)
        assert np.max(np.abs(dmu_g - dmu_o)) <= 1e-8 * np.max(np.abs(dmu_o))
        assert np.max(np.abs(dvar_g - dvar_o)) <= 1e-8 * max(np.max(np.abs(dvar_o)), 1e-6 * amp)
    import alabi_b200 as ab
    with pytest.raises(Exception):
        ab.GP(kernel=ab.kernels.ExpSquaredKernel(metric=np.ones(33), ndim=33)).compute(rng.uniform(size=(10, 33)))


def test_empty_and_single_query_sets():
    rng = np.random.default_rng(0)
    X = rng.uniform(-1, 1, size=(90, 2))
    y = X[:, 0] ** 2 - X[:, 1]
    o, g = _pair("Matern52Kernel", X, y, np.zeros(2))
    mu, var = g.predict(y, np.empty((0, 2)), return_var=True)
    assert mu.shape == (0,) and var.shape == (0,)
    mu = g.predict(y, np.empty((0, 2)), return_cov=False)
    assert mu.shape == (0,)
    m1, v1 = g.predict(y, np.array([[0.1, 0.2]]), return_var=True)
    mo, vo = o.predict(y, np.array([[0.1, 0.2]]), return_var=True)
    assert abs(m1[0] - mo[0]) <= 1e-9 * abs(mo[0]) and abs(v1[0] - vo[0]) <= 1e-9 * np.exp(o.log_const)
    idx, val = g.utility_argmin(y, np.empty((0, 2)), np.array([(-1.0, 1.0)] * 2), algorithm="bape")
    assert idx == -1
    # every candidate outside the prior box: no finite utility, index -1 (the caller falls back)
    idx, val = g.utility_argmin(y, np.full((5, 2), 3.0), np.array([(-1.0, 1.0)] * 2), algorithm="agp")
    assert idx == -1


def test_duplicated_points_and_default_white_noise():
    """Exact duplicates make K singular up to the white noise: with the reference default
    (white_noise = -12) the factorisation must still succeed and agree with LAPACK to the
    accuracy the conditioning allows; with no white noise at all it must fail like george
    (LinAlgError from compute, -inf / zero gradient with quiet=True)."""
    import alabi_b200 as ab
    rng = np.random.default_rng(3)
    X = rng.uniform(-1, 1, size=(140, 2))
    X[70:] = X[:70]                                            # every point twice
    y = np.sin(3 * X[:, 0]) + X[:, 1]
    o, g = _pair("ExpSquaredKernel", X, y, np.array([-1.0, -1.0]), wn=-12.0)
    ll_o, ll_g = o.log_likelihood(y), g.log_likelihood(y)
    assert np.isfinite(ll_g) and abs(ll_g - ll_o) <= 1e-6 * abs(ll_o)
    k = ab.kernels.ExpSquaredKernel(metric=np.exp([-1.0, -1.0]), ndim=2) * 1.0
    gs = ab.GP(kernel=k, fit_mean=True, mean=0.0, white_noise=-745.0, fit_white_noise=True)
    with pytest.raises(np.linalg.LinAlgError):
        gs.compute(X)
    assert gs.log_likelihood(y, quiet=True) == -np.inf
    assert np.all(gs.grad_log_likelihood(y, quiet=True) == 0.0)
    # appending an exact duplicate with the default white noise: the bordered update and a
    # fresh factorisation agree to what the conditioning (~1e12) allows
    ga = ab.GP(kernel=k, fit_mean=True, mean=0.0, white_noise=-12.0, fit_white_noise=True)
    ga.compute(X[:70])
    ga.append_point(X[0])
    gf = ab.GP(kernel=k, fit_mean=True, mean=0.0, white_noise=-12.0, fit_white_noise=True)
    gf.compute(np.vstack([X[:70], X[:1]]))
    yy = np.append(y[:70], y[0])
    assert abs(ga.log_likelihood(yy) - gf.log_likelihood(yy)) <= 1e-5 * abs(gf.log_likelihood(yy))


def test_non_finite_inputs_are_reported():
    import alabi_b200 as ab
    from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb
    rng = np.random.default_rng(4)
    X = rng.uniform(-1, 1, size=(60, 2))
    y = X[:, 0] - X[:, 1] ** 2
    o, g = _pair("Matern32Kernel", X, y, np.zeros(2))
    lp = SurrogateLogProb(g, y, [(-1, 1), (-1, 1)])
    s = EnsembleSampler(16, 2, lp, seed=1)
    p0 = rng.uniform(-0.5, 0.5, size=(16, 2))
    p0[3, 1] = np.nan
    with pytest.raises(ValueError):
        s.run_mcmc(p0, 5)
    yn = y.copy()
    yn[5] = np.nan
    assert not np.isfinite(g.log_likelihood(yn, quiet=True)) or g.log_likelihood(yn, quiet=True) == -np.inf


def test_sampler_proposals_per_unit_variants_replay():
    """P = 2 proposals per unit (90 walkers) and the wide 32-proposal unit (one lane per proposal,
    the large-ensemble configuration: 32 walkers per SM plus 26, so the last unit is partly
    filled), each replayed on the CPU from the same draws; a configuration with
    ab_ensemble_config.reserved != 0 is refused."""
    import alabi_b200 as ab
    from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb
    rng = np.random.default_rng(8)
    n, d = 700, 3
    X = rng.uniform(-2, 2, size=(n, d))
    y = -0.5 * np.sum((X / 0.9) ** 2, axis=1)
    o, g = _pair("ExpSquaredKernel", X, y, np.array([0.3, 0.1, 0.5]))
    b = np.array([(-2.0, 2.0)] * d)
    lp = SurrogateLogProb(g, y, b)

    def lp_o(q):
        q = np.atleast_2d(q)
        inside = np.all((q > b[:, 0]) & (q < b[:, 1]), axis=1)
        return np.where(inside, o.predict(y, q), -np.inf)
    nsm = ab._lib.load().ab_device_sm_count(g._hd.device)
    assert nsm > 0
    for nw in (90, 32 * nsm + 26):
        p0 = rng.uniform(-1, 1, size=(nw, d))
        s = EnsembleSampler(nw, d, lp, seed=21)
        s.run_mcmc(p0, 25)
        ref, _, _, _ = oem.replay_device_chain(p0, lp_o, 25, 21)
        assert np.allclose(s.get_chain(), ref, rtol=1e-9, atol=1e-12)

    s = EnsembleSampler(90, d, lp, seed=21)
    config = s._config

    def reserved_config(*args, **kwargs):
        cfg = config(*args, **kwargs)
        cfg.reserved = 1
        return cfg
    s._config = reserved_config
    with pytest.raises(ab._lib.AlabiB200Error, match="reserved must be 0"):
        s.run_mcmc(rng.uniform(-1, 1, size=(90, d)), 5)


def test_round2_paths_at_their_smallest_sizes():
    """The round-2 device paths on degenerate shapes: batched CV with ragged folds that straddle a
    128-row padding boundary and a one-block factor; nested walks in one dimension; a wide streamed
    sampler whose (unit, chunk) ranges cut units in the middle with thinning."""
    import alabi_b200 as ab
    from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb
    from alabi_b200.nested import DeviceWalker
    from oracle import nested as onest
    rng = np.random.default_rng(9)
    # (1) CV: n = 161, 5 folds of 33 / 32 rows -> 128 or 129 training rows (one or two 128-blocks)
    n, d = 161, 2
    X = rng.uniform(-1, 1, size=(n, d))
    y = np.cos(2 * X[:, 0]) + X[:, 1]
    o, g = _pair("ExpSquaredKernel", X, y, np.array([0.1, 0.3]), wn=-8.0)
    base = g.get_parameter_vector()
    idx = rng.permutation(n)
    folds = [(np.sort(np.setdiff1d(idx, f)), np.sort(f)) for f in np.array_split(idx, 5)]
    preds, lls, st = g.cv_batch(X, y, np.array([base, base + 0.1]), folds * 2)
    assert np.all(st == 0) and len(preds) == 10
    for b, (tr, va) in enumerate(folds * 2):
        oc = ogp.make_gp("ExpSquaredKernel", X[tr], y[tr], np.zeros(d), amp=1.0, compute=False)
        oc.set_parameter_vector(base + (0.1 if b >= 5 else 0.0))
        oc.compute(X[tr])
        assert abs(lls[b] - oc.log_likelihood(y[tr])) <= 1e-9 * abs(oc.log_likelihood(y[tr]))
        np.testing.assert_allclose(preds[b], oc.predict(y[tr], X[va]), rtol=1e-8, atol=1e-9)
    # (2) nested walk in one dimension
    X1 = rng.uniform(-2, 2, size=(60, 1))
    y1 = -0.5 * (X1[:, 0] / 0.5) ** 2
    o1, g1 = _pair("Matern52Kernel", X1, y1, np.array([0.0]), wn=-8.0)
    b1 = np.array([(-2.0, 2.0)])
    w = DeviceWalker(SurrogateLogProb(g1, y1, b1), b1, seed=5)
    u0 = rng.uniform(0.3, 0.7, size=(9, 1))
    th0 = w.transform(u0)
    l0 = o1.predict(y1, th0)
    cnt = w.counter
    u, th, ll, acc = w.walk(u0, th0, l0, float(np.min(l0)) - 1.0, 0.5, np.array([[0.2]]), 7)
    ur, thr, llr, nacc, margin = onest.replay_walk(u0, th0, l0, float(np.min(l0)) - 1.0, 0.5, np.array([[0.2]]), 7, 5, cnt,
                                                   w.transform, lambda t: o1.predict(y1, t))
    np.testing.assert_allclose(u, ur, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(ll, llr, rtol=1e-9, atol=1e-9)
    # (3) wide streamed sampler, ranges cutting units, thinning: continuing a run reproduces the long run
    n3, d3, nw = 5000, 16, 4736
    X3 = rng.uniform(-1, 1, size=(n3, d3))
    y3 = -0.5 * np.sum((X3 / 0.6) ** 2, axis=1)
    o3, g3 = _pair("ExpSquaredKernel", X3, y3, np.full(d3, 0.5), wn=-8.0)
    lp = SurrogateLogProb(g3, y3, [(-1.0, 1.0)] * d3)
    p0 = rng.uniform(-0.5, 0.5, size=(nw, d3))
    s = EnsembleSampler(nw, d3, lp, seed=3)
    s.run_mcmc(p0, 3, thin_by=2)
    s2 = EnsembleSampler(nw, d3, lp, seed=3)
    s2.run_mcmc(p0, 1, thin_by=2)
    s2.run_mcmc(None, 2, thin_by=2)
    np.testing.assert_array_equal(s.get_chain(), s2.get_chain())
    lp_last = o3.predict(y3, s.get_chain()[-1][:200])
    np.testing.assert_allclose(s.get_log_prob()[-1][:200], lp_last, rtol=1e-9, atol=1e-9)
