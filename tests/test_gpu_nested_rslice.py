"""GPU checks for random-direction slice sampling in the built-in nested sampler (dynesty's
sample="rslice", ``ab_nested_rslice``): the device launch replayed on the CPU by
``tests/rslice_oracle.replay_rslice`` against the oracle GP for all four kernels (resident and chunked
training sets), batch independence, the caps, one launch per batch, and the samplers on the c3
eggbox, on an 8-D surrogate against rwalk, and through ``SurrogateModel.run_dynesty``."""
import os
import sys

import numpy as np
import pytest
from scipy import stats

from oracle import gp as ogp

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import rq_oracle as rq  # noqa: E402
import rslice_oracle as ors  # noqa: E402

pytestmark = pytest.mark.gpu


def _surrogate(kind, n, d, seed, y_scale=1.0, y_offset=0.0):
    import alabi_b200 as ab
    from alabi_b200.ensemble import SurrogateLogProb
    rng = np.random.default_rng(seed)
    b = np.array([(-2.0, 2.0)] * d)
    X = rng.uniform(b[:, 0], b[:, 1], size=(n, d))
    y = -0.5 * np.sum((X / 0.7) ** 2, axis=1) + 0.3 * np.sin(2.0 * X[:, 0])
    log_M = np.full(d, 0.8 if d < 20 else 1.5)
    if kind == "RationalQuadraticKernel":
        o = rq.make_gp(kind, X, y, log_M, amp=np.var(y), white_noise=-8.0, log_alpha=0.5)
        kern = ab.kernels.RationalQuadraticKernel(0.5, metric=np.exp(log_M), ndim=d)
    else:
        o = ogp.make_gp(kind, X, y, log_M, amp=np.var(y), white_noise=-8.0)
        kern = getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d)
    g = ab.GP(kernel=kern * np.var(y), fit_mean=True, mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
    g.compute(X)
    lp = SurrogateLogProb(g, y, b, y_scale=y_scale, y_offset=y_offset)
    like_o = lambda t: o.predict(y, np.atleast_2d(t)) * y_scale + y_offset
    return g, lp, like_o, rng, b


def _start(w, like_o, rng, nchains, d):
    u0 = rng.uniform(0.2, 0.8, size=(nchains, d))
    th0 = w.transform(u0)
    l0 = like_o(th0)
    A = rng.normal(size=(d, d))
    chol = np.linalg.cholesky(A @ A.T / d + 0.5 * np.eye(d)) * 0.08
    return u0, th0, l0, chol


@pytest.mark.parametrize("kind,n,d,nchains,normal", [("ExpSquaredKernel", 300, 2, 37, False),
                                                     ("Matern52Kernel", 900, 5, 96, True),
                                                     ("Matern32Kernel", 2600, 12, 64, False),
                                                     ("RationalQuadraticKernel", 1200, 24, 40, False)])
def test_device_rslice_replays_on_the_cpu(kind, n, d, nchains, normal):
    """Matern32 at N = 2600, d = 12 does not fit the shared-memory budget: chunked training points."""
    from alabi_b200.nested import DeviceWalker
    g, lp, like_o, rng, b = _surrogate(kind, n, d, 5, y_scale=1.5, y_offset=-0.25)
    data = [(0.2, 0.5), (None, None)] + [(-0.3, 0.8)] * (d - 2) if normal else None
    w = DeviceWalker(lp, b, prior_data=data, seed=8642)
    u0, th0, l0, chol = _start(w, like_o, rng, nchains, d)
    np.testing.assert_allclose(w.like(th0), l0, rtol=1e-9, atol=1e-9)
    lmin = float(np.quantile(l0, 0.3))
    slices, scale = 4, 0.9
    cnt = w.counter
    u, th, ll, counts = w.rslice(u0, th0, l0, lmin, scale, chol, slices)
    ur, thr, llr, cr, margin = ors.replay_rslice(u0, th0, l0, lmin, scale, chol, slices, 8642, cnt, w.transform, like_o)
    assert margin > 1e-7                                  # no branch sits on the rounding edge
    np.testing.assert_array_equal(counts, cr)
    np.testing.assert_allclose(u, ur, rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(th, thr, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(ll, llr, rtol=1e-9, atol=1e-9)
    # chains that start below lmin (30 %) shrink onto their start and end at the contraction cap
    moved = counts[:, 0] > 0
    assert np.all(counts[l0 > lmin, 0] == slices) and counts[:, 1].sum() > 0 and counts[:, 2].sum() > 0
    assert np.all(ll[moved] > lmin) and np.all((u > 0) & (u < 1))
    assert np.array_equal(u[~moved], u0[~moved]) and np.array_equal(ll[~moved], l0[~moved])


def test_rslice_chain_does_not_depend_on_its_batch():
    from alabi_b200.nested import DeviceWalker
    d = 6
    g, lp, like_o, rng, b = _surrogate("Matern52Kernel", 700, d, 9)
    w = DeviceWalker(lp, b, seed=77)
    u0, th0, l0, chol = _start(w, like_o, rng, 200, d)
    lmin = float(np.quantile(l0, 0.4))
    cnt = w.counter
    full = w.rslice(u0, th0, l0, lmin, 1.3, chol, 5)
    for k in (0, 45, 168):
        w.counter = cnt
        part = w.rslice(u0[k:k + 32], th0[k:k + 32], l0[k:k + 32], lmin, 1.3, chol, 5, chain_offset=k)
        for a, p in zip(full, part):
            assert np.array_equal(a[k:k + 32], p), k


def test_rslice_launch_is_bounded_and_single():
    """lmin above the surrogate's maximum: every slice fails, the caps end the launch, the start
    points stay.  lmin = -inf: stepping out stops at the cube's faces and every slice completes.
    Each call is one kernel launch."""
    from alabi_b200 import _lib
    from alabi_b200.nested import RSLICE_MAX_CONTRACT, DeviceWalker
    d = 3
    g, lp, like_o, rng, b = _surrogate("ExpSquaredKernel", 400, d, 13)
    w = DeviceWalker(lp, b, seed=5)
    u0, th0, l0, chol = _start(w, like_o, rng, 70, d)
    lib = _lib.load()
    n0 = lib.ab_launch_counter()
    u, th, ll, counts = w.rslice(u0, th0, l0, float(l0.max()) + 1e3, 1.0, chol, 3)
    assert lib.ab_launch_counter() - n0 == 1
    assert np.array_equal(u, u0) and np.array_equal(th, th0) and np.array_equal(ll, l0)
    assert np.all(counts[:, 0] == 0) and np.all(counts[:, 1] == 0) and np.all(counts[:, 2] == RSLICE_MAX_CONTRACT)
    assert np.all(counts[:, 3] <= RSLICE_MAX_CONTRACT + 2)
    u, th, ll, counts = w.rslice(u0, th0, l0, -np.inf, 1.0, chol, 3)
    assert np.all(counts[:, 0] == 3) and np.all((u > 0) & (u < 1)) and np.all(counts[:, 1] < 1024)
    np.testing.assert_allclose(ll, like_o(th), rtol=1e-9, atol=1e-9)


def _c3():
    from alabi_b200 import workloads
    from alabi_b200.ensemble import SurrogateLogProb
    cfg = workloads.make_config("c3")
    g = workloads.build_gp(cfg)
    g.compute(cfg["X"])
    return cfg, g, SurrogateLogProb(g, cfg["y"], cfg["bounds"])


def test_static_and_dynamic_rslice_on_c3_surrogate():
    """c3 (2-D eggbox, Matern-5/2, N = 4000) with the tolerances of the rwalk test: evidence against
    the quadrature of exp(surrogate), KS statistics of both marginals, one launch per batch."""
    from alabi_b200 import _lib
    from alabi_b200.nested import BatchedNestedSampler, DeviceWalker, resample_equal
    cfg, g, lp = _c3()
    lib = _lib.load()
    w1 = DeviceWalker(lp, cfg["bounds"], seed=31)
    calls = []
    rs = w1.rslice
    w1.rslice = lambda *a, **k: calls.append(1) or rs(*a, **k)
    s1 = BatchedNestedSampler(w1, 2, nlive=2000, sample="rslice", slices=5, rstate=32)
    n0 = lib.ab_launch_counter()
    r1 = s1.run_nested(dlogz=0.02)
    assert lib.ab_launch_counter() - n0 <= 3 + len(calls), (lib.ab_launch_counter() - n0, len(calls))
    assert r1.ncall > len(calls) * s1.nbatch * s1.slices
    s2 = BatchedNestedSampler(DeviceWalker(lp, cfg["bounds"], seed=41), 2, nlive=1000, sample="rslice", rstate=42)
    r2 = s2.run_dynamic(dlogz_init=0.5, n_effective=6000, pfrac=1.0)
    z1, e1, z2, e2 = r1.logz[-1], r1.logzerr[-1], r2.logz[-1], r2.logzerr[-1]
    assert abs(z1 - z2) < 4.0 * np.hypot(e1, e2) + 0.05, (z1, e1, z2, e2)
    assert r2.nbatch >= 1 and r2.n_effective >= 6000
    ng = 400
    gx = (np.arange(ng) + 0.5) / ng
    grid = np.stack(np.meshgrid(gx, gx, indexing="ij"), axis=-1).reshape(-1, 2)
    mu = g.predict(cfg["y"], grid, return_cov=False)
    z_quad = np.log(np.mean(np.exp(mu - mu.max()))) + mu.max()
    assert abs(z1 - z_quad) < 4.0 * e1 + 0.05 and abs(z2 - z_quad) < 4.0 * e2 + 0.05, (z1, e1, z2, e2, z_quad)
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


def test_rslice_against_rwalk_on_8d_gaussian_surrogate():
    import alabi_b200 as ab
    from alabi_b200.ensemble import SurrogateLogProb
    from alabi_b200.nested import BatchedNestedSampler, DeviceWalker, resample_equal
    d = 8
    rng = np.random.default_rng(21)
    sd = np.linspace(0.5, 1.0, d)
    cov = 0.3 ** np.abs(np.subtract.outer(np.arange(d), np.arange(d))) * np.outer(sd, sd)
    P = np.linalg.inv(cov)
    b = np.array([(-4.0, 4.0)] * d)
    X = np.vstack([rng.uniform(-4.0, 4.0, size=(1500, d)), rng.multivariate_normal(np.zeros(d), 2.0 * cov, size=1500)])
    X = np.clip(X, -4.0, 4.0)
    y = -0.5 * np.einsum("ij,jk,ik->i", X, P, X)
    g = ab.GP(kernel=ab.kernels.ExpSquaredKernel(metric=np.full(d, 9.0), ndim=d) * np.var(y), fit_mean=True,
              mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
    g.compute(X)
    lp = SurrogateLogProb(g, y, b)
    runs = []
    for kw, seed in ((dict(sample="rslice", slices=d), 51), (dict(sample="rwalk", walks=25), 61)):
        s = BatchedNestedSampler(DeviceWalker(lp, b, seed=seed), d, nlive=600, rstate=seed + 1, **kw)
        r = s.run_nested(dlogz=0.05)
        q = resample_equal(r.samples, np.exp(r.logwt - r.logz[-1]), np.random.default_rng(seed))
        runs.append((r.logz[-1], r.logzerr[-1], q.mean(axis=0), q.std(axis=0)))
    (z1, e1, m1, s1), (z2, e2, m2, s2) = runs
    assert abs(z1 - z2) < 4.0 * np.hypot(e1, e2) + 0.05, (z1, e1, z2, e2)
    assert np.all(np.abs(m1 - m2) < 0.1 * sd + 0.03), (m1, m2)
    np.testing.assert_allclose(s1, s2, rtol=0.1)
    np.testing.assert_allclose(s1, sd, rtol=0.15)


def test_run_dynesty_rslice(tmp_path):
    """SurrogateModel.run_dynesty(sample="rslice", slices=...) in both modes on the device, a user
    prior transform through the host chains, and sample="slice" still raises."""
    import alabi_b200 as ab
    np.random.seed(2)
    fn = lambda th: -0.5 * float(np.sum((np.asarray(th).flatten() / np.array([0.6, 0.9])) ** 2))
    sm = ab.SurrogateModel(lnlike_fn=fn, bounds=[(-3.0, 3.0)] * 2, savedir=str(tmp_path), cache=False, verbose=False)
    sm.init_samples(ntrain=150, ntest=0, sampler="lhs")
    sm.init_gp(kernel="ExpSquaredKernel", fit_amp=True, fit_mean=True, fit_white_noise=False, white_noise=-10,
               gp_scale_rng=[-1, 3], hyperopt_method="ml", gp_nopt=2)
    want = np.log(2 * np.pi * 0.6 * 0.9 / 36.0)
    sm.run_dynesty(mode="static", sampler_kwargs={"nlive": 300, "seed": 5, "sample": "rslice", "slices": 6},
                   run_kwargs={"dlogz": 0.05}, min_ess=300)
    assert isinstance(sm.dynesty_sampler.walker, ab.nested.DeviceWalker) and sm.dynesty_sampler.slices == 6
    assert abs(sm.dynesty_logz - want) < 3 * sm.dynesty_logz_err + 0.2
    st = sm.dynesty_samples.std(axis=0)
    assert abs(st[0] - 0.6) < 0.1 and abs(st[1] - 0.9) < 0.12
    sm.run_dynesty(mode="dynamic", sampler_kwargs={"nlive": 150, "seed": 6, "sample": "rslice"},
                   run_kwargs={"n_effective": 3000}, min_ess=300)
    assert sm.dynesty_sampler.sample == "rslice" and sm.dynesty_sampler.slices == 5
    assert abs(sm.dynesty_logz - want) < 3 * sm.dynesty_logz_err + 0.25 and sm.dynesty_results.nbatch >= 1
    st = sm.dynesty_samples.std(axis=0)
    assert abs(st[0] - 0.6) < 0.1 and abs(st[1] - 0.9) < 0.12
    seen = []

    def my_transform(u):
        seen.append(np.ndim(u))
        return np.array([6.0 * u[0] - 3.0, 6.0 * u[1] - 3.0])
    sm.run_dynesty(mode="static", prior_transform=my_transform,
                   sampler_kwargs={"nlive": 100, "seed": 7, "sample": "rslice", "slices": 3}, run_kwargs={"dlogz": 0.5},
                   min_ess=50)
    assert isinstance(sm.dynesty_sampler.walker, ab.nested.HostWalker)
    assert set(seen) == {1} and abs(sm.dynesty_logz - want) < 3 * sm.dynesty_logz_err + 0.5
    with pytest.raises(NotImplementedError):
        sm.run_dynesty(sampler_kwargs={"nlive": 50, "sample": "slice"}, min_ess=10)
