"""Host side of random-direction slice sampling (dynesty's sample="rslice") in the built-in nested
sampler: HostWalker.rslice on an analytic 20-D correlated Gaussian, the caps, the scale rule,
keyword validation and pickling.  No GPU needed."""
import pickle
from functools import partial

import numpy as np
import pytest

from alabi_b200 import nested as ns, utility as ut


def _gaussian(d, seed):
    rng = np.random.default_rng(seed)
    sd = rng.uniform(0.5, 1.5, size=d)
    R = 0.5 ** np.abs(np.subtract.outer(np.arange(d), np.arange(d)))       # AR(1) correlations
    cov = R * np.outer(sd, sd)
    P = np.linalg.inv(cov)
    logn = -0.5 * (d * np.log(2.0 * np.pi) + np.linalg.slogdet(cov)[1])

    def loglike(th):
        th = np.atleast_2d(th)
        return logn - 0.5 * np.einsum("ij,jk,ik->i", th, P, th)
    bounds = np.stack([-6.0 * sd, 6.0 * sd], axis=1)                        # holds all but ~1e-8 of the mass
    return loglike, bounds, sd


def test_host_rslice_evidence_and_widths_20d():
    d = 20
    loglike, bounds, sd = _gaussian(d, 3)
    w = ns.HostWalker(loglike, partial(ut.prior_transform_uniform, bounds=bounds), d, rng=np.random.default_rng(4))
    # 2 d slices: with dynesty's default of 5 (or 25 rwalk steps) the chains decorrelate too little
    # in 20 dimensions and ln Z comes out about 1.3 high
    s = ns.BatchedNestedSampler(w, d, nlive=300, sample="rslice", slices=2 * d, rstate=5)
    r = s.run_nested(dlogz=0.1)
    want = -np.sum(np.log(bounds[:, 1] - bounds[:, 0]))                     # L is a normalised density
    assert abs(r.logz[-1] - want) < 3.0 * r.logzerr[-1] + 0.1, (r.logz[-1], r.logzerr[-1], want)
    q = ns.resample_equal(r.samples, np.exp(r.logwt - r.logz[-1]), np.random.default_rng(6))
    np.testing.assert_allclose(q.std(axis=0), sd, rtol=0.10)
    assert r.ncall == w.ncall and r.ncall > 0


def test_host_rslice_counts_and_constraint():
    d, k = 3, 40
    loglike, bounds, _ = _gaussian(d, 7)
    w = ns.HostWalker(loglike, partial(ut.prior_transform_uniform, bounds=bounds), d, rng=np.random.default_rng(8))
    u0 = np.random.default_rng(9).uniform(0.4, 0.6, size=(k, d))
    th0 = w.transform(u0)
    l0 = w.like(th0)
    lmin = float(np.quantile(l0, 0.2))
    n0 = w.ncall
    u, th, ll, counts = w.rslice(u0, th0, l0, lmin, 1.0, np.eye(d) * 0.1, 4)
    assert counts.shape == (k, 4) and counts[:, 3].sum() == w.ncall - n0
    # a chain that starts below lmin shrinks onto its own start and ends at the contraction cap
    done = counts[:, 0] == 4
    assert np.all(done[l0 > lmin]) and np.all(counts[~done, 2] % ns.RSLICE_MAX_CONTRACT == 0)
    assert np.all(ll[counts[:, 0] > 0] > lmin)
    assert np.all((u > 0) & (u < 1)) and np.allclose(th, w.transform(u)) and np.allclose(ll, loglike(th))
    assert np.all(counts[:, 2] <= 4 * ns.RSLICE_MAX_CONTRACT) and np.all(counts[:, 1] <= 4 * ns.RSLICE_MAX_EXPAND)


def test_host_rslice_caps_bound_a_hopeless_slice():
    """lmin above the maximum: no slice completes, every chain keeps its start point after exactly
    RSLICE_MAX_CONTRACT failed shrink draws (no expansion ever succeeds)."""
    d, k = 4, 9
    loglike, bounds, _ = _gaussian(d, 10)
    w = ns.HostWalker(loglike, partial(ut.prior_transform_uniform, bounds=bounds), d, rng=np.random.default_rng(11))
    u0 = np.random.default_rng(12).uniform(0.3, 0.7, size=(k, d))
    th0 = w.transform(u0)
    l0 = w.like(th0)
    u, th, ll, counts = w.rslice(u0, th0, l0, 1e3, 0.5, np.eye(d) * 0.2, 3)
    assert np.array_equal(u, u0) and np.array_equal(th, th0) and np.array_equal(ll, l0)
    assert np.all(counts[:, 0] == 0) and np.all(counts[:, 1] == 0) and np.all(counts[:, 2] == ns.RSLICE_MAX_CONTRACT)
    # a flat likelihood with lmin = -inf: stepping out ends at the cube's faces, every slice completes
    w2 = ns.HostWalker(lambda t: np.zeros(len(t)), partial(ut.prior_transform_uniform, bounds=bounds), d,
                       rng=np.random.default_rng(13))
    u, th, ll, counts = w2.rslice(u0, th0, np.zeros(k), -np.inf, 1.0, np.eye(d) * 0.05, 3)
    assert np.all(counts[:, 0] == 3) and np.all(counts[:, 1] > 0) and np.all((u > 0) & (u < 1))


def test_rslice_scale_rule():
    c = lambda e, n: np.array([[1, e, n, 0]])
    assert ns.rslice_scale(0.7, c(5, 5)) == pytest.approx(0.7)
    assert ns.rslice_scale(0.7, c(9, 3)) == pytest.approx(0.7 * 1.5)
    assert ns.rslice_scale(0.7, c(1, 3)) == pytest.approx(0.7 * 0.5)
    assert ns.rslice_scale(8.0, c(10, 0)) == 10.0 and ns.rslice_scale(0.3, c(0, 4)) == 1e-6
    assert ns.rslice_scale(0.3, np.zeros((3, 4), dtype=np.int64)) == 0.3


def test_sampler_keywords_and_pickle():
    loglike, bounds, _ = _gaussian(2, 14)
    w = ns.HostWalker(loglike, partial(ut.prior_transform_uniform, bounds=bounds), 2)
    with pytest.raises(ValueError):
        ns.BatchedNestedSampler(w, 2, sample="slice")
    with pytest.raises(ValueError):
        ns.BatchedNestedSampler(w, 2, sample="rslice", slices=0)
    s = ns.BatchedNestedSampler(w, 2, nlive=50, sample="rslice", slices=7, rstate=1)
    s.scale = 0.37
    t = pickle.loads(pickle.dumps(s))
    assert (t.sample, t.slices, t.scale, t.walker) == ("rslice", 7, 0.37, None)
    assert ns.BatchedNestedSampler(w, 2).sample == "rwalk"


def test_run_dynesty_rslice_keywords_on_the_host(tmp_path):
    """run_dynesty's built-in runner with a host likelihood: sample="rslice" and slices reach the
    sampler and a static run lands on the analytic evidence; every other sample= keeps raising,
    naming both methods."""
    import alabi_b200 as ab
    fn = lambda th: -0.5 * float(np.sum((np.asarray(th).flatten() / np.array([0.6, 0.9])) ** 2))
    sm = ab.SurrogateModel(lnlike_fn=fn, bounds=[(-3.0, 3.0)] * 2, savedir=str(tmp_path), cache=False, verbose=False)
    sm.prior_transform = partial(ut.prior_transform_uniform, bounds=sm.bounds)
    batch_like = lambda th: np.array([fn(t) for t in np.atleast_2d(th)])
    run = sm._builtin_nested_runner(ns, batch_like, None, "static", {"nlive": 200, "seed": 3, "sample": "rslice", "slices": 4},
                                    {"dlogz": 0.1}, None)
    ds, res = run(1)
    assert isinstance(ds.walker, ns.HostWalker) and (ds.sample, ds.slices) == ("rslice", 4)
    want = np.log(2 * np.pi * 0.6 * 0.9 / 36.0)
    assert abs(res.logz[-1] - want) < 3 * res.logzerr[-1] + 0.2, (res.logz[-1], res.logzerr[-1], want)
    assert res.ncall == ds.walker.ncall
    ds, _ = sm._builtin_nested_runner(ns, batch_like, None, "static", {"nlive": 30, "sample": "auto"}, {"dlogz": 5.0}, None)(1)
    assert ds.sample == "rwalk" and ds.slices == 5
    for bad in ("slice", "unif", "rstagger"):
        with pytest.raises(NotImplementedError, match="rslice"):
            sm.run_dynesty(like_fn="true", sampler_kwargs={"nlive": 50, "sample": bad}, min_ess=10)
