"""GPU parity for K5: the device stretch-move chain replayed on the CPU from
the same Philox draws (oracle/philox.py + oracle/emcee.py), per-proposal
log-probabilities against the oracle GP, and posterior consistency (KS)."""
import numpy as np
import pytest
from scipy import stats

from oracle import gp as ogp, emcee as oem

pytestmark = pytest.mark.gpu


def surrogate(kind, n, d, seed, bounds):
    import alabi_b200 as ab
    from alabi_b200.ensemble import SurrogateLogProb
    rng = np.random.default_rng(seed)
    b = np.asarray(bounds, dtype=np.float64)
    X = rng.uniform(b[:, 0], b[:, 1], size=(n, d))
    y = -0.5 * np.sum((X / 0.7) ** 2, axis=1)          # Gaussian log-density, sigma = 0.7
    log_M = np.full(d, 1.0)
    o = ogp.make_gp(kind, X, y, log_M, amp=np.var(y), white_noise=-8.0)
    k = getattr(ab.kernels, kind)(metric=np.exp(log_M), ndim=d) * np.var(y)
    g = ab.GP(kernel=k, fit_mean=True, mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
    g.compute(X)
    lp = SurrogateLogProb(g, y, b)

    def lp_oracle(q):
        q = np.atleast_2d(q)
        inside = np.all((q > b[:, 0]) & (q < b[:, 1]), axis=1)
        return np.where(inside, o.predict(y, q), -np.inf)
    return g, lp, lp_oracle, rng, b


@pytest.mark.parametrize("kind,n,d,nw,rs,wpu", [("ExpSquaredKernel", 200, 2, 32, True, 0),
                                                ("Matern32Kernel", 300, 3, 41, False, 1),
                                                ("Matern52Kernel", 700, 5, 64, True, 2),
                                                ("ExpSquaredKernel", 150, 2, 10, True, 8),
                                                ("Matern32Kernel", 250, 15, 48, True, 0),
                                                ("ExpSquaredKernel", 300, 23, 64, False, 0)])
def test_chain_replay_and_per_proposal_logp(kind, n, d, nw, rs, wpu):
    from alabi_b200.ensemble import EnsembleSampler
    bounds = [(-2.0, 2.0)] * d
    g, lp, lp_oracle, rng, b = surrogate(kind, n, d, 17, bounds)
    p0 = rng.uniform(-1.9, 1.9, size=(nw, d))
    nsteps, seed = 60, 987654321987
    s = EnsembleSampler(nw, d, lp, seed=seed, randomize_split=rs, warps_per_unit=wpu, live_dangerously=True)
    s.run_mcmc(p0, nsteps, record_proposals=True)
    chain, lps, nacc, rec = oem.replay_device_chain(p0, lp_oracle, nsteps, seed, randomize_split=rs)
    rq, rl = s.proposal_record
    # (1) given the same proposals the log-probabilities are identical to 1e-9
    n_checked = 0
    for t in range(nsteps):
        ok = np.isfinite(rq[t, :, 0])
        lo = lp_oracle(rq[t, ok])
        fin = np.isfinite(lo)
        assert np.array_equal(np.isfinite(rl[t, ok]), fin)
        np.testing.assert_allclose(rl[t, ok][fin], lo[fin], rtol=1e-9, atol=1e-9)
        n_checked += ok.sum()
    assert n_checked == nsteps * nw
    # (2) the whole chain replays (same draws, same accept decisions)
    np.testing.assert_allclose(s.get_chain(), chain, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(s.get_log_prob(), lps, rtol=1e-9, atol=1e-9)
    assert np.array_equal(s._naccepted, nacc)
    np.testing.assert_allclose(rq[5][np.isfinite(rq[5, :, 0])], rec[5]["q"][np.isfinite(rec[5]["q"][:, 0])], rtol=1e-12)
    # continuing the run keeps the counter-based stream going
    s.run_mcmc(None, 5)
    chain2, _, _, _ = oem.replay_device_chain(p0, lp_oracle, nsteps + 5, seed, randomize_split=rs)
    np.testing.assert_allclose(s.get_chain()[-1], chain2[-1], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("kind,n,d,nw", [("ExpSquaredKernel", 200, 2, 32), ("Matern52Kernel", 400, 5, 4800)])
def test_normal_prior_chain_replay(kind, n, d, nw):
    """Box times independent normals (ut.lnprior_normal) evaluated inside the kernel: same
    replay / per-proposal checks as above, narrow and wide units (4800 walkers: one lane per
    proposal), with a uniform dimension mixed in."""
    from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb
    from oracle import utility as ou
    bounds = [(-2.0, 2.0)] * d
    g, lp0, lp_oracle0, rng, b = surrogate(kind, n, d, 23, bounds)
    data = [(0.3, 0.4), (None, None)] + [(-0.5, 0.25)] * (d - 2)
    mu = np.array([np.nan if m is None else m for m, _ in data])
    sd = np.array([np.nan if s_ is None else s_ for _, s_ in data])
    lp = SurrogateLogProb(g, lp0.y, b, prior_data=data)

    def lp_oracle(q):
        q = np.atleast_2d(q)
        with np.errstate(invalid="ignore"):
            return lp_oracle0(q) + ou.lnprior_normal(q, b, mu, sd)
    p0 = rng.uniform(-1.9, 1.9, size=(nw, d))
    nsteps, seed = 25, 55443322
    s = EnsembleSampler(nw, d, lp, seed=seed)
    s.run_mcmc(p0, nsteps, record_proposals=True)
    chain, lps, nacc, _ = oem.replay_device_chain(p0, lp_oracle, nsteps, seed)
    rq, rl = s.proposal_record
    for t in range(0, nsteps, 6):
        ok = np.isfinite(rq[t, :, 0])
        lo = lp_oracle(rq[t, ok])
        fin = np.isfinite(lo)
        assert np.array_equal(np.isfinite(rl[t, ok]), fin)
        np.testing.assert_allclose(rl[t, ok][fin], lo[fin], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(s.get_chain(), chain, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(s.get_log_prob(), lps, rtol=1e-9, atol=1e-9)
    assert np.array_equal(s._naccepted, nacc)
    # the host-callable form agrees with the device log-probabilities
    np.testing.assert_allclose(lp(chain[-1]), s.get_log_prob()[-1], rtol=1e-9, atol=1e-9)
    # and the prior really acts: the same seed without it walks elsewhere
    s0 = EnsembleSampler(nw, d, lp0, seed=seed)
    s0.run_mcmc(p0, nsteps)
    assert not np.allclose(s0.get_chain()[-1], s.get_chain()[-1])


def test_posterior_moments_ks_and_api():
    from alabi_b200.ensemble import EnsembleSampler
    from alabi_b200.mcmc_utils import estimate_burnin
    d, nw = 2, 200
    g, lp, lp_oracle, rng, b = surrogate("ExpSquaredKernel", 400, d, 3, [(-3.0, 3.0)] * d)
    s = EnsembleSampler(nw, d, lp, seed=42)
    st = s.run_mcmc(rng.uniform(-1, 1, size=(nw, d)), 1500, progress=True)
    assert st.coords.shape == (nw, d) and s.get_chain().shape == (1500, nw, d)
    burn, thin = estimate_burnin(s)
    tau = s.get_autocorr_time(tol=0)
    assert 1 < tau.max() < 100 and 0.2 < s.acceptance_fraction.mean() < 0.9
    flat = s.get_chain(discard=max(burn, 100), thin=int(2 * tau.max()) + 1, flat=True)
    # the surrogate interpolates a N(0, 0.7^2 I) log-density
    assert abs(flat.mean()) < 0.05 and abs(flat.std() - 0.7) < 0.05
    assert stats.kstest(flat[:, 0] / 0.7, "norm").pvalue > 1e-4
    # CPU emcee-order sampler on the oracle surrogate gives the same moments
    ref = oem.StretchEnsemble(40, d, lp_oracle, seed=1, vectorize=True)
    ref.run_mcmc(rng.uniform(-1, 1, size=(40, d)), 1500)
    rflat = ref.get_chain(discard=300, thin=10, flat=True)
    assert stats.ks_2samp(flat[::3, 1], rflat[:, 1]).pvalue > 1e-4
    # thin_by stores every k-th step only
    s2 = EnsembleSampler(nw, d, lp, seed=42)
    s2.run_mcmc(s.get_chain()[0], 10, thin_by=3)
    assert s2.get_chain().shape == (10, nw, d) and s2._step_counter == 30


def test_large_nonresident_training_set():
    """N too large for shared memory: the chunked path gives the same chain."""
    from alabi_b200.ensemble import EnsembleSampler
    d, nw = 12, 96
    g, lp, lp_oracle, rng, b = surrogate("ExpSquaredKernel", 2600, d, 9, [(-2.0, 2.0)] * d)
    p0 = rng.uniform(-1, 1, size=(nw, d))
    s = EnsembleSampler(nw, d, lp, seed=5)
    s.run_mcmc(p0, 12)
    chain, lps, nacc, _ = oem.replay_device_chain(p0, lp_oracle, 12, 5)
    np.testing.assert_allclose(s.get_chain(), chain, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("d,n", [(12, 6000), (10, 6000), (32, 700)])
def test_wide_streamed_split_units_replay(d, n):
    """Large ensemble on a training set that does not fit shared memory: the wide unit streams the
    points (per-warp rings filled by bulk copies; d = 10 runs the d = 12 kernel with two zero-padded
    dimensions; d = 32, N = 700 runs the run-time chunk length with 33 row slices per warp and chunk),
    and the points of one 32-proposal unit are split over several CTAs whose slice sums
    are combined in slice order by the CTA that completes the unit.  The chain must still replay on
    the CPU, and must not depend on how a run is cut into pieces."""
    from alabi_b200.ensemble import EnsembleSampler
    nw = 4800
    g, lp, lp_oracle, rng, b = surrogate("ExpSquaredKernel", n, d, 31, [(-2.0, 2.0)] * d)
    p0 = rng.uniform(-1, 1, size=(nw, d))
    s = EnsembleSampler(nw, d, lp, seed=77)
    s.run_mcmc(p0, 5)
    chain, lps, nacc, _ = oem.replay_device_chain(p0, lp_oracle, 5, 77)
    np.testing.assert_allclose(s.get_chain(), chain, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(s.get_log_prob(), lps, rtol=1e-9, atol=1e-9)
    assert np.array_equal(s._naccepted, nacc)
    s2 = EnsembleSampler(nw, d, lp, seed=77)
    s2.run_mcmc(p0, 2)
    s2.run_mcmc(None, 3)
    np.testing.assert_array_equal(s2.get_chain(), s.get_chain())


@pytest.mark.parametrize("kind,n,d,nw,rs,wpu,nsteps,thin", [("Matern32Kernel", 1000, 2, 1000, True, 0, 150, 1),
                                                            ("ExpSquaredKernel", 300, 3, 41, False, 2, 97, 1),
                                                            ("Matern52Kernel", 500, 5, 333, True, 4, 64, 3),
                                                            ("ExpSquaredKernel", 150, 2, 10, True, 8, 200, 1)])
def test_dataflow_schedule_gives_the_barrier_schedules_chain(kind, n, d, nw, rs, wpu, nsteps, thin):
    """Small ensembles: the dataflow schedule (a proposal waits for its partner's versioned record,
    progress barrier every 15 steps, ring of 32 versions) must reproduce the chain of the grid-barrier
    schedule bit for bit -- stored rows, log-probabilities, acceptance counts and the final state --
    over more steps than the ring holds versions, for odd ensembles, thinning and cut runs."""
    from alabi_b200.ensemble import EnsembleSampler
    g, lp, lp_oracle, rng, b = surrogate(kind, n, d, 23, [(-2.0, 2.0)] * d)
    p0 = rng.uniform(-1.9, 1.9, size=(nw, d))
    runs = []
    for schedule in (1, 0):
        s = EnsembleSampler(nw, d, lp, seed=4242, randomize_split=rs, warps_per_unit=wpu, schedule=schedule,
                            live_dangerously=True)
        s.run_mcmc(p0, nsteps, thin_by=thin)
        st = s.run_mcmc(None, 40, thin_by=thin)              # continued run: versions restart, step counter goes on
        runs.append((s.get_chain().copy(), s.get_log_prob().copy(), s._naccepted.copy(), st.coords.copy(), st.log_prob.copy()))
    for a, b_ in zip(runs[0], runs[1]):
        np.testing.assert_array_equal(a, b_)
    # without a stored chain (final state only) the dataflow run ends in the same state
    s = EnsembleSampler(nw, d, lp, seed=4242, randomize_split=rs, warps_per_unit=wpu, live_dangerously=True)
    s.run_mcmc(p0, nsteps * thin, store=False)
    st = s.run_mcmc(None, 40 * thin, store=False)
    np.testing.assert_array_equal(st.coords, runs[0][3])
    np.testing.assert_array_equal(st.log_prob, runs[0][4])


@pytest.mark.parametrize("nw,n,d", [(64, 300, 3), (4800, 700, 2)])
def test_gathered_chain_layout_and_second_destination(nw, n, d):
    """The fused all_gather of chain blocks on one GPU: the kernel writes its stored rows as columns
    [column, column + nwalkers) of wider rows, into its own buffer AND into a second destination (the
    role a peer GPU's buffer plays over NVLink).  Both must hold exactly the chain of a plain run, the
    other columns stay untouched; small units (dataflow schedule) and the wide unit."""
    import torch
    from alabi_b200.ensemble import EnsembleSampler
    g, lp, lp_oracle, rng, b = surrogate("ExpSquaredKernel", n, d, 5, [(-2.0, 2.0)] * d)
    p0 = rng.uniform(-1.5, 1.5, size=(nw, d))
    steps, thin, col, total = 9, 2, 5, nw + 11
    plain = EnsembleSampler(nw, d, lp, seed=31)
    plain.run_mcmc(p0, steps, thin_by=thin, walker_offset=col)
    dev = f"cuda:{g._hd.device}"
    own_c = torch.full((steps, total, d), -7.0, dtype=torch.float64, device=dev)
    own_l = torch.full((steps, total), -7.0, dtype=torch.float64, device=dev)
    peer_c, peer_l = own_c.clone(), own_l.clone()
    spec = {"chain": own_c, "log_prob": own_l, "nwalkers_total": total, "column": col,
            "peer_chain_ptrs": [peer_c.data_ptr()], "peer_log_prob_ptrs": [peer_l.data_ptr()]}
    s = EnsembleSampler(nw, d, lp, seed=31)
    s.run_mcmc(p0, steps, thin_by=thin, walker_offset=col, store="device", gather=spec)
    torch.cuda.synchronize()
    for c_, l_ in ((own_c, own_l), (peer_c, peer_l)):
        np.testing.assert_array_equal(c_[:, col:col + nw].cpu().numpy(), plain.get_chain())
        np.testing.assert_array_equal(l_[:, col:col + nw].cpu().numpy(), plain.get_log_prob())
        assert bool((c_[:, :col] == -7.0).all()) and bool((c_[:, col + nw:] == -7.0).all())
        assert bool((l_[:, :col] == -7.0).all()) and bool((l_[:, col + nw:] == -7.0).all())
    np.testing.assert_array_equal(s.get_chain(), plain.get_chain())


@pytest.mark.parametrize("kind,n,d,nw", [("ExpSquaredKernel", 2600, 12, 150), ("Matern32Kernel", 5000, 8, 67)])
def test_spread_mode_gives_the_streaming_units_chain(kind, n, d, nw):
    """Small ensemble on a training set that does not fit shared memory: the automatic choice (wide unit,
    short chunks, (unit, chunk) pairs dealt over the GPU, segment sums combined in segment order) must give
    the chain of the 2-proposal units that stream the whole training set (schedule=3), up to the summation
    order of the surrogate mean: same accept decisions, positions within 1e-12, and the CPU replay holds."""
    from alabi_b200.ensemble import EnsembleSampler
    g, lp, lp_oracle, rng, b = surrogate(kind, n, d, 41, [(-2.0, 2.0)] * d)
    p0 = rng.uniform(-1.5, 1.5, size=(nw, d))
    runs = []
    for schedule in (3, 0):
        s = EnsembleSampler(nw, d, lp, seed=777, schedule=schedule)
        s.run_mcmc(p0, 24, thin_by=2)
        s.run_mcmc(None, 6, thin_by=2)
        runs.append((s.get_chain().copy(), s.get_log_prob().copy(), s._naccepted.copy()))
    np.testing.assert_array_equal(runs[0][2], runs[1][2])
    np.testing.assert_allclose(runs[0][0], runs[1][0], rtol=0, atol=1e-12)
    np.testing.assert_allclose(runs[0][1], runs[1][1], rtol=1e-10, atol=1e-10)
    chain, lps, nacc, _ = oem.replay_device_chain(p0, lp_oracle, 60, 777)
    np.testing.assert_allclose(runs[1][0], chain[1::2], rtol=1e-9, atol=1e-12)
