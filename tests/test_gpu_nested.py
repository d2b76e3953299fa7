"""GPU checks for nested sampling on the surrogate (SURVEY 8a14 / 8f-2): the constrained random
walks of ``ab_nested_walk`` replayed on the CPU from the same Philox draws against the oracle GP,
and the static / dynamic samplers on the c3 surrogate (evidence within its error, posteriors
consistent by KS)."""
import numpy as np
import pytest
from scipy import stats

from oracle import gp as ogp, nested as onest

pytestmark = pytest.mark.gpu


def _surrogate(kind, n, d, seed, bounds, y_scale=1.0, y_offset=0.0):
    import alabi_b200 as ab
    from alabi_b200.ensemble import SurrogateLogProb
    rng = np.random.default_rng(seed)
    b = np.asarray(bounds, dtype=np.float64)
    X = rng.uniform(b[:, 0], b[:, 1], size=(n, d))
    y = -0.5 * np.sum((X / 0.7) ** 2, axis=1) + 0.3 * np.sin(2.0 * X[:, 0])
    log_M = np.full(d, 0.8)
    o = ogp.make_gp(kind, X, y, log_M, amp=np.var(y), white_noise=-8.0)
    g = ab.GP(kernel=getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d) * np.var(y), fit_mean=True, mean=np.median(y),
              white_noise=-8.0, fit_white_noise=True)
    g.compute(X)
    lp = SurrogateLogProb(g, y, b, y_scale=y_scale, y_offset=y_offset)
    like_o = lambda t: o.predict(y, np.atleast_2d(t)) * y_scale + y_offset
    return g, lp, like_o, rng, b


@pytest.mark.parametrize("kind,n,d,nchains,normal", [("ExpSquaredKernel", 300, 2, 37, False),
                                                     ("Matern52Kernel", 900, 5, 96, True),
                                                     ("Matern32Kernel", 2600, 12, 64, False),
                                                     ("Matern52Kernel", 500, 14, 48, True),
                                                     ("ExpSquaredKernel", 600, 22, 40, False)])
def test_device_walk_replays_on_the_cpu(kind, n, d, nchains, normal):
    from alabi_b200.nested import DeviceWalker
    g, lp, like_o, rng, b = _surrogate(kind, n, d, 5, [(-2.0, 2.0)] * d, y_scale=1.5, y_offset=-0.25)
    data = None
    if normal:
        data = [(0.2, 0.5), (None, None)] + [(-0.3, 0.8)] * (d - 2)
    w = DeviceWalker(lp, b, prior_data=data, seed=424242)
    u0 = rng.uniform(0.2, 0.8, size=(nchains, d))
    th0 = w.transform(u0)
    l0 = like_o(th0)
    # the device's own batched likelihood agrees with the oracle
    np.testing.assert_allclose(w.like(th0), l0, rtol=1e-9, atol=1e-9)
    lmin = float(np.quantile(l0, 0.3))
    A = rng.normal(size=(d, d))
    chol = np.linalg.cholesky(A @ A.T / d + 0.5 * np.eye(d)) * 0.08
    walks, scale = 12, 0.9
    cnt = w.counter
    u, th, ll, acc = w.walk(u0, th0, l0, lmin, scale, chol, walks)
    ur, thr, llr, naccr, margin = onest.replay_walk(u0, th0, l0, lmin, scale, chol, walks, 424242, cnt, w.transform, like_o)
    assert margin > 1e-7                                  # no accept decision sits on the rounding edge
    np.testing.assert_allclose(u, ur, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(th, thr, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(ll, llr, rtol=1e-9, atol=1e-9)
    assert abs(acc - naccr.sum() / (nchains * walks)) < 1e-12 and 0.02 < acc < 0.98
    assert np.all((u > 0) & (u < 1)) and np.all(ll[naccr > 0] > lmin)
    # a second launch draws new numbers (launch counter) and keeps the constraint
    u2, th2, ll2, _ = w.walk(u, th, ll, lmin, scale, chol, walks)
    assert not np.allclose(u2, u) and np.all(ll2 >= np.minimum(ll, ll2)) and np.all(ll2[np.any(u2 != u, axis=1)] > lmin)


def test_static_and_dynamic_sampler_on_c3_surrogate():
    """c3 (2-D eggbox, Matern-5/2, N = 4000): evidence of the dynamic run within the combined error
    of the static run's, posteriors consistent (KS on both marginals), one launch per batch."""
    from alabi_b200 import _lib, workloads
    from alabi_b200.ensemble import SurrogateLogProb
    from alabi_b200.nested import BatchedNestedSampler, DeviceWalker, resample_equal
    cfg = workloads.make_config("c3")
    g = workloads.build_gp(cfg)
    g.compute(cfg["X"])
    lp = SurrogateLogProb(g, cfg["y"], cfg["bounds"])
    lib = _lib.load()
    s1 = BatchedNestedSampler(DeviceWalker(lp, cfg["bounds"], seed=11), 2, nlive=2000, walks=25, rstate=12)
    n0 = lib.ab_launch_counter()
    r1 = s1.run_nested(dlogz=0.02)
    launches = lib.ab_launch_counter() - n0
    # every batch of nbatch x walks proposals is ONE walk launch (the only other launches are the
    # three kernels of the batched predict for the initial live points)
    assert launches <= 3 + r1.ncall / (s1.nbatch * s1.walks) + 1, (launches, r1.ncall)
    s2 = BatchedNestedSampler(DeviceWalker(lp, cfg["bounds"], seed=21), 2, nlive=1000, walks=25, rstate=22)
    r2 = s2.run_dynamic(dlogz_init=0.5, n_effective=6000, pfrac=1.0)
    z1, e1, z2, e2 = r1.logz[-1], r1.logzerr[-1], r2.logz[-1], r2.logzerr[-1]
    assert abs(z1 - z2) < 4.0 * np.hypot(e1, e2) + 0.05, (z1, e1, z2, e2)
    assert r2.nbatch >= 1 and r2.n_effective >= 6000
    # quadrature of exp(surrogate) over the unit square is the evidence both estimate
    ng = 400
    gx = (np.arange(ng) + 0.5) / ng
    grid = np.stack(np.meshgrid(gx, gx, indexing="ij"), axis=-1).reshape(-1, 2)
    mu = g.predict(cfg["y"], grid, return_cov=False)
    z_quad = np.log(np.mean(np.exp(mu - mu.max()))) + mu.max()
    assert abs(z1 - z_quad) < 4.0 * e1 + 0.05 and abs(z2 - z_quad) < 4.0 * e2 + 0.05, (z1, e1, z2, e2, z_quad)
    # posteriors: the eggbox has 25 modes whose weights every run estimates with its own noise, and
    # resampled points are not independent, so the KS STATISTIC against the quadrature marginals is
    # bounded (and between the two runs), not a p-value
    post = np.exp(mu - mu.max()).reshape(ng, ng)
    q1 = resample_equal(r1.samples, np.exp(r1.logwt - z1), np.random.default_rng(1))
    q2 = resample_equal(r2.samples, np.exp(r2.logwt - z2), np.random.default_rng(2))
    for k in range(2):
        marg = post.sum(axis=1 - k)
        cdf = np.cumsum(marg) / marg.sum()
        for q in (q1, q2):
            emp = np.searchsorted(np.sort(q[:, k]), gx + 0.5 / ng, side="right") / len(q)
            assert np.max(np.abs(emp - cdf)) < 0.1, (k, np.max(np.abs(emp - cdf)))
        assert stats.ks_2samp(q1[:, k], q2[:, k]).statistic < 0.12


def test_run_dynesty_modes_and_kwargs(tmp_path):
    """SurrogateModel.run_dynesty: both modes run on the device walker, a user prior transform is
    honoured point by point, unsupported keywords raise, save_iter writes a checkpoint."""
    import alabi_b200 as ab
    np.random.seed(2)
    fn = lambda th: -0.5 * float(np.sum((np.asarray(th).flatten() / np.array([0.6, 0.9])) ** 2))
    sm = ab.SurrogateModel(lnlike_fn=fn, bounds=[(-3.0, 3.0)] * 2, savedir=str(tmp_path), cache=False, verbose=False)
    sm.init_samples(ntrain=150, ntest=0, sampler="lhs")
    sm.init_gp(kernel="ExpSquaredKernel", fit_amp=True, fit_mean=True, fit_white_noise=False, white_noise=-10,
               gp_scale_rng=[-1, 3], hyperopt_method="ml", gp_nopt=2)
    want = np.log(2 * np.pi * 0.6 * 0.9 / 36.0)
    sm.run_dynesty(mode="static", sampler_kwargs={"nlive": 300, "seed": 5}, run_kwargs={"dlogz": 0.05}, min_ess=300)
    assert abs(sm.dynesty_logz - want) < 3 * sm.dynesty_logz_err + 0.2
    st = sm.dynesty_samples.std(axis=0)
    assert abs(st[0] - 0.6) < 0.1 and abs(st[1] - 0.9) < 0.12
    sm.run_dynesty(mode="dynamic", sampler_kwargs={"nlive": 150, "seed": 6}, run_kwargs={"n_effective": 3000},
                   min_ess=300, save_iter=500)
    assert abs(sm.dynesty_logz - want) < 3 * sm.dynesty_logz_err + 0.25 and sm.dynesty_results.nbatch >= 1
    st = sm.dynesty_samples.std(axis=0)
    assert abs(st[0] - 0.6) < 0.1 and abs(st[1] - 0.9) < 0.12
    assert (tmp_path / "dynesty_sampler_surrogate_run1.pkl").exists()
    # user transform with dynesty's one-point contract (indexes dimensions)
    seen = []

    def my_transform(u):
        seen.append(np.ndim(u))
        return np.array([6.0 * u[0] - 3.0, 6.0 * u[1] - 3.0])
    sm.run_dynesty(mode="static", prior_transform=my_transform, sampler_kwargs={"nlive": 100, "seed": 7, "walks": 10},
                   run_kwargs={"dlogz": 0.5}, min_ess=50)
    assert set(seen) == {1} and abs(sm.dynesty_logz - want) < 3 * sm.dynesty_logz_err + 0.5
    with pytest.raises(TypeError):
        sm.run_dynesty(sampler_kwargs={"nlive": 50, "first_update": {}}, min_ess=10)
    with pytest.raises(NotImplementedError):
        sm.run_dynesty(sampler_kwargs={"nlive": 50, "sample": "slice"}, min_ess=10)
    with pytest.raises(ValueError):
        sm.run_dynesty(mode="adaptive")
