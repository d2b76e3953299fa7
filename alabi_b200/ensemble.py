"""emcee.EnsembleSampler look-alike running the stretch move on the GPU (K5).

Mirrors the protocol alabi uses (alabi/core.py:2319-2387, alabi/mcmc_utils.py:45):
``EnsembleSampler(nwalkers, ndim, log_prob_fn, pool=None, **kw)``,
``run_mcmc(p0, nsteps, progress=True)``, ``get_chain(discard, thin, flat)``,
``get_last_sample().coords``, ``acceptance_fraction``, ``get_autocorr_time``.

``log_prob_fn`` must be a :class:`SurrogateLogProb` (GP predictive mean +
uniform prior box, optionally times independent normals as in ``ut.lnprior_normal``,
i.e. ``SurrogateModel.lnprob`` of alabi/core.py:2073-2100):
the whole step then runs on the device with no host round trip.  A plain
Python callable cannot be evaluated inside a CUDA kernel; it is rejected
instead of silently falling back to a CPU sampler.
"""
import ctypes

import numpy as np

from . import _lib
from .mcmc_utils import integrated_time

__all__ = ["EnsembleSampler", "SurrogateLogProb", "State"]


class State:
    def __init__(self, coords, log_prob=None, random_state=None):
        self.coords = np.array(coords, dtype=np.float64)
        self.log_prob = None if log_prob is None else np.array(log_prob, dtype=np.float64)
        self.blobs = None
        self.random_state = random_state

    def __iter__(self):
        return iter((self.coords, self.log_prob, self.random_state))


class _DeviceState(State):
    """The sampler's state after a run, left in HBM: ``coords`` / ``log_prob`` are downloaded on first
    access (emcee's State holds NumPy arrays), and a run that continues from it (``initial_state=None``)
    hands the device tensors straight back to the kernel — no download, finiteness scan and upload of
    the ensemble between the pieces of a long chain (10 MB each way at 65 536 walkers x 20)."""

    def __init__(self, coords_dev, log_prob_dev):
        self._dev = (coords_dev, log_prob_dev)
        self._host = None
        self.blobs = None
        self.random_state = None

    def _get(self):
        if self._host is None:
            self._host = (self._dev[0].cpu().numpy(), self._dev[1].cpu().numpy())
        return self._host

    @property
    def coords(self):
        return self._get()[0]

    @property
    def log_prob(self):
        return self._get()[1]

    def __reduce__(self):                       # pickles / copies as a plain host State
        return (State, (self.coords, self.log_prob))


class SurrogateLogProb:
    """ln P(theta) = GP mean(theta_scaler(theta)) mapped back by the y scaler,
    plus a uniform prior on the open box ``bounds`` (unscaled theta) and, with
    ``prior_data = [(mean, std) | (None, None), ...]``, independent normal priors on the
    dimensions that name a mean (``ut.lnprior_normal``, alabi/utility.py:370-378).

    theta_scaled = theta * theta_scale + theta_offset;
    y = ys * y_scale + y_offset (y_kind 0), -10**ys (1) or 10**ys (2)."""

    def __init__(self, gp, y, bounds, theta_scale=None, theta_offset=None, y_kind=0, y_scale=1.0, y_offset=0.0,
                 prior_data=None):
        self.gp = gp
        self.y = np.ascontiguousarray(np.asarray(y, dtype=np.float64).reshape(-1))
        self.bounds = np.asarray(bounds, dtype=np.float64).reshape(-1, 2)
        d = len(self.bounds)
        self.theta_scale = np.ones(d) if theta_scale is None else np.asarray(theta_scale, dtype=np.float64).reshape(d)
        self.theta_offset = np.zeros(d) if theta_offset is None else np.asarray(theta_offset, dtype=np.float64).reshape(d)
        self.y_kind, self.y_scale, self.y_offset = int(y_kind), float(y_scale), float(y_offset)
        # normal priors: mean / std per dimension, std = 0 marks a uniform dimension
        self.prior_mu, self.prior_sd = np.zeros(d), np.zeros(d)
        if prior_data is not None:
            if len(prior_data) != d:
                raise ValueError("prior_data needs one (mean, std) pair per dimension")
            for k, (m, sd) in enumerate(prior_data):
                if m is not None:
                    if sd is None or not (np.isfinite(m) and np.isfinite(sd) and sd > 0):
                        raise ValueError(f"prior_data[{k}]: a normal prior needs a finite mean and std > 0")
                    self.prior_mu[k], self.prior_sd[k] = float(m), float(sd)
        self.use_normal_prior = bool(np.any(self.prior_sd > 0))

    def __call__(self, theta):
        """Host-callable form (one device predict per call) for callers that
        need a Python function, e.g. a nested sampler's likelihood."""
        theta = np.asarray(theta, dtype=np.float64)
        one = theta.ndim == 1
        t = np.atleast_2d(theta)
        ys = self.gp.predict(self.y, t * self.theta_scale + self.theta_offset, return_cov=False)
        yv = ys * self.y_scale + self.y_offset if self.y_kind == 0 else (-10.0 ** ys if self.y_kind == 1 else 10.0 ** ys)
        inside = np.all((t > self.bounds[:, 0]) & (t < self.bounds[:, 1]), axis=1)
        for k in np.nonzero(self.prior_sd > 0)[0]:
            z = (t[:, k] - self.prior_mu[k]) / self.prior_sd[k]
            yv = yv + ((-(z * z) / 2.0 - 0.9189385332046727) - np.log(self.prior_sd[k]))
        lp = np.where(inside, yv, -np.inf)
        return lp[0] if one else lp


class EnsembleSampler:
    def __init__(self, nwalkers, ndim, log_prob_fn, pool=None, moves=None, args=None, kwargs=None,
                 backend=None, vectorize=False, blobs_dtype=None, parameter_names=None, a=2.0, seed=None,
                 randomize_split=True, live_dangerously=False, warps_per_unit=0, schedule=0):
        if not isinstance(log_prob_fn, SurrogateLogProb):
            raise TypeError("alabi_b200.EnsembleSampler runs on the GPU and needs a SurrogateLogProb "
                            "(GP surrogate + uniform prior); arbitrary Python log-probabilities are not supported")
        if moves is not None:
            raise NotImplementedError("only the default StretchMove(a) is implemented")
        self.nwalkers, self.ndim = int(nwalkers), int(ndim)
        if self.nwalkers < 2 * self.ndim and not live_dangerously:
            raise ValueError("It is unadvisable to use a red-blue move with fewer walkers than twice the number of dimensions.")
        if ndim != len(log_prob_fn.bounds):
            raise ValueError("ndim does not match the surrogate's bounds")
        self.log_prob_fn = log_prob_fn
        self.a = float(a)
        self.seed = int(np.random.SeedSequence().entropy % (2 ** 63)) if seed is None else int(seed)
        self.randomize_split = bool(randomize_split)
        self.warps_per_unit = int(warps_per_unit)
        # small ensembles: 0 = dataflow on the partner's versioned record (default), 1 = a grid barrier
        # per half-step (ab_ensemble_config.schedule); the chains are identical
        self.schedule = int(schedule)
        self.pinned_limit_bytes = 4 << 30      # larger stored chains land in pageable host memory
        self.reset()

    def reset(self):
        self.iteration = 0
        self._chain = np.empty((0, self.nwalkers, self.ndim))
        self._log_prob = np.empty((0, self.nwalkers))
        self._naccepted = np.zeros(self.nwalkers, dtype=np.int64)
        self._last = None
        self._step_counter = 0
        self.last_run_device_seconds = None
        self.device_chain = self.device_log_prob = None
        self._device_rows_pending = False

    # ------------------------------------------------------------------------------------
    def _config(self, nsteps, thin_by, init_logp, walker_offset=0):
        lp = self.log_prob_fn
        cfg = _lib.EnsembleConfig()
        cfg.nwalkers, cfg.nsteps, cfg.thin_by = self.nwalkers, int(nsteps), int(thin_by)
        cfg.init_logp, cfg.randomize_split = int(init_logp), int(self.randomize_split)
        cfg.warps_per_unit, cfg.y_kind = self.warps_per_unit, lp.y_kind
        cfg.a, cfg.seed = self.a, self.seed
        cfg.first_step, cfg.walker_offset = self._step_counter, int(walker_offset)
        cfg.y_scale, cfg.y_offset = lp.y_scale, lp.y_offset
        for k in range(self.ndim):
            cfg.lo[k], cfg.hi[k] = lp.bounds[k, 0], lp.bounds[k, 1]
            cfg.theta_scale[k], cfg.theta_offset[k] = lp.theta_scale[k], lp.theta_offset[k]
            cfg.prior_mu[k], cfg.prior_sd[k] = lp.prior_mu[k], lp.prior_sd[k]
        cfg.use_normal_prior = int(lp.use_normal_prior)
        cfg.schedule = self.schedule
        return cfg

    def run_mcmc(self, initial_state, nsteps, progress=False, thin_by=1, store=True, record_proposals=False,
                 walker_offset=0, gather=None, **kwargs):
        """Run ``nsteps * thin_by`` ensemble steps on the device, storing every
        ``thin_by``-th.  Returns the final :class:`State`.  ``store``: True (chain and
        log-probabilities end up in host arrays, emcee's backend), False (final state only) or
        ``"device"`` (the stored chain stays in HBM as ``device_chain`` / ``device_log_prob``
        torch tensors: what ``parallel.sharded_ensemble`` all_gathers over NVLink).  ``gather`` (with
        ``store="device"``): a ``parallel.PeerChainBuffers`` spec — the kernel writes the stored rows
        straight into the gathered (nsteps, nwalkers_total, ndim) buffers of this rank AND of the
        other ranks (peer memory over NVLink), the fused form of the chain-block all_gather."""
        import torch
        gp = self.log_prob_fn.gp
        gp.recompute()
        gp._set_targets(self.log_prob_fn.y)
        hd = gp._hd
        dev = f"cuda:{hd.device}"
        if initial_state is None:
            if self._last is None:
                raise ValueError("Cannot have `initial_state=None` if run_mcmc has never been called.")
            initial_state = self._last
        # a run that continues from this sampler's own last state takes it from HBM as it is (the kernel
        # left finite, independent walkers there); a host copy the caller already looked at stays valid
        # because the kernel updates fresh clones
        resume = isinstance(initial_state, _DeviceState) and initial_state is self._last and \
            initial_state._dev[0].device.index == hd.device
        if resume:
            have_lp, p0 = True, None
        else:
            have_lp = isinstance(initial_state, State) and initial_state.log_prob is not None
            p0 = initial_state.coords if isinstance(initial_state, State) else np.asarray(initial_state, dtype=np.float64)
            if p0.shape != (self.nwalkers, self.ndim):
                raise ValueError("incompatible input dimensions")
            if not np.all(np.isfinite(p0)):
                raise ValueError("At least one parameter value was infinite or NaN")
            if self.nwalkers > 1 and not self._independent(p0):
                raise ValueError("Initial state has a large condition number. Make sure that your walkers are linearly independent for the best performance")
        on_device = isinstance(store, str) and store == "device"
        store = bool(store)
        if store:
            self._materialise()              # rows of an earlier store="device" run join the host chain first
        total = int(nsteps) * int(thin_by)
        if resume:
            coords, logp = initial_state._dev[0].clone(), initial_state._dev[1].clone()
        else:
            coords = torch.from_numpy(np.ascontiguousarray(p0)).to(dev)
            logp = torch.from_numpy(np.ascontiguousarray(initial_state.log_prob)).to(dev) if have_lp \
                else torch.empty(self.nwalkers, dtype=torch.float64, device=dev)
        nacc = torch.zeros(self.nwalkers, dtype=torch.int64, device=dev)
        if gather is not None:
            if not on_device or record_proposals:
                raise ValueError("gather needs store='device' and no proposal record")
            chain, lpc = gather["chain"], gather["log_prob"]            # gathered buffers of THIS rank
            if tuple(chain.shape) != (int(nsteps), gather["nwalkers_total"], self.ndim) or chain.dtype != torch.float64:
                raise ValueError("gather buffers do not match (nsteps, nwalkers_total, ndim)")
        else:
            chain = torch.empty((int(nsteps), self.nwalkers, self.ndim), dtype=torch.float64, device=dev) if store else None
            lpc = torch.empty((int(nsteps), self.nwalkers), dtype=torch.float64, device=dev) if store else None
        rq = torch.full((total, self.nwalkers, self.ndim), float("nan"), dtype=torch.float64, device=dev) if record_proposals else None
        rl = torch.full((total, self.nwalkers), float("nan"), dtype=torch.float64, device=dev) if record_proposals else None
        cfg = self._config(total, thin_by, not have_lp, walker_offset)
        if gather is not None:
            cfg.chain_row_walkers, cfg.chain_walker_offset = int(gather["nwalkers_total"]), int(gather["column"])
            cfg.n_chain_peers = len(gather["peer_chain_ptrs"])
            for q, (pc, pl) in enumerate(zip(gather["peer_chain_ptrs"], gather["peer_log_prob_ptrs"])):
                cfg.chain_peers[q], cfg.logp_chain_peers[q] = pc, pl
        lib = hd.lib
        prof_prev = lib.ab_gp_set_profiling(hd.h, 1)
        if store and not record_proposals and not on_device:
            # chain delivered to host arrays by the library: the run is cut into pieces, piece b is
            # copied out while piece b + 1 runs.  The host arrays are page-locked (torch's pinned
            # allocator caches the block, so repeated runs reuse touched, locked pages); very large
            # chains fall back to pageable memory.
            nbytes = chain.numel() * 8
            ch_t = lh_t = None
            if nbytes <= self.pinned_limit_bytes:
                try:
                    ch_t = torch.empty(tuple(chain.shape), dtype=torch.float64, pin_memory=True)
                    lh_t = torch.empty(tuple(lpc.shape), dtype=torch.float64, pin_memory=True)
                except RuntimeError:
                    ch_t = lh_t = None
            if ch_t is None:
                ch_t = torch.empty(tuple(chain.shape), dtype=torch.float64)
                lh_t = torch.empty(tuple(lpc.shape), dtype=torch.float64)
            nblocks = int(min(16, max(1, nbytes // (8 << 20)))) if int(nsteps) > 1 else 1
            rc = _lib.check(lib.ab_ensemble_run_host(hd.h, ctypes.byref(cfg), _lib.ptr(coords), _lib.ptr(logp), _lib.ptr(nacc),
                                                     _lib.ptr(chain), _lib.ptr(lpc), _lib.ptr(ch_t), _lib.ptr(lh_t), nblocks),
                            "ab_ensemble_run_host")
            hbufs = (ch_t.numpy(), lh_t.numpy())
        else:
            _lib.check(lib.ab_ensemble_launch(hd.h, ctypes.byref(cfg), _lib.ptr(coords), _lib.ptr(logp), _lib.ptr(nacc),
                                              _lib.ptr(chain), _lib.ptr(lpc), _lib.ptr(rq), _lib.ptr(rl)),
                       "ab_ensemble_launch")
            rc = _lib.check(lib.ab_ensemble_finish(hd.h), "ab_ensemble_finish")
            hbufs = None
            if store and not on_device:
                hbufs = (chain.cpu().numpy(), lpc.cpu().numpy())
        # device time of the sampler kernels alone (events around the launches, on the handle's stream)
        kms, kcnt = ctypes.c_double(), ctypes.c_longlong()
        lib.ab_gp_profile_read(hd.h, 4, ctypes.byref(kms), ctypes.byref(kcnt))
        lib.ab_gp_set_profiling(hd.h, prof_prev)
        self.last_run_device_seconds = kms.value * 1e-3
        self.last_run_launches = int(kcnt.value)
        if rc == 1:
            raise ValueError("Probability function returned NaN")
        self._step_counter += total
        self._naccepted += nacc.cpu().numpy()
        if on_device:
            # the stored rows stay in HBM; get_chain() / get_log_prob() copy them on first use
            if gather is not None and not gather.get("keep_local", True):
                pass                             # the caller (parallel.sharded_ensemble) attaches the rows when all pieces are in
            else:
                if gather is not None:
                    # own columns of the gathered buffers, copied: the buffers are reused by the next gather
                    c0 = int(gather["column"])
                    chain, lpc = chain[:, c0:c0 + self.nwalkers].clone(), lpc[:, c0:c0 + self.nwalkers].clone()
                self.device_chain, self.device_log_prob = chain, lpc
                self._device_rows_pending = True
                self.iteration += int(nsteps)
        elif store:
            ch, lh = hbufs
            self._chain = ch if len(self._chain) == 0 else np.concatenate([self._chain, ch])
            self._log_prob = lh if len(self._log_prob) == 0 else np.concatenate([self._log_prob, lh])
            self.iteration += int(nsteps)
        if record_proposals:
            self.proposal_record = (rq.cpu().numpy(), rl.cpu().numpy())
        self._last = _DeviceState(coords, logp)
        return self._last

    def _independent(self, p0):
        """emcee's start-up check: the walkers must span the space.  Rank of the centred positions
        through their ndim x ndim triangular factor (O(nwalkers ndim^2)), not an SVD of the tall
        matrix; skipped when the run continues from this sampler's own last state."""
        last = self._last
        if isinstance(last, _DeviceState):
            last = last._host[0] if last._host is not None else None      # (no download just for this test)
        else:
            last = getattr(last, "coords", None)
        if p0 is last:
            return True
        c = p0 - p0.mean(axis=0)
        r = np.linalg.qr(c, mode="r") if c.shape[0] >= c.shape[1] else c
        return np.linalg.matrix_rank(r) >= min(self.ndim, self.nwalkers - 1)

    def sample(self, initial_state, iterations=1, **kwargs):
        for _ in range(int(iterations)):
            yield self.run_mcmc(initial_state, 1, **kwargs)
            initial_state = None

    # ------------------------------------------------------------------------------------
    def _materialise(self):
        if getattr(self, "_device_rows_pending", False):
            ch, lh = self.device_chain.cpu().numpy(), self.device_log_prob.cpu().numpy()
            self._chain = ch if len(self._chain) == 0 else np.concatenate([self._chain, ch])
            self._log_prob = lh if len(self._log_prob) == 0 else np.concatenate([self._log_prob, lh])
            self._device_rows_pending = False

    def get_chain(self, discard=0, thin=1, flat=False):
        self._materialise()
        v = self._chain[discard + thin - 1:self.iteration:thin]
        return v.reshape(-1, self.ndim) if flat else v

    def get_log_prob(self, discard=0, thin=1, flat=False):
        self._materialise()
        v = self._log_prob[discard + thin - 1:self.iteration:thin]
        return v.reshape(-1) if flat else v

    def get_last_sample(self):
        if self._last is None:
            raise AttributeError("you must run the sampler before accessing the results")
        return self._last

    @property
    def chain(self):
        return np.swapaxes(self.get_chain(), 0, 1)

    @property
    def flatchain(self):
        return self.get_chain(flat=True)

    @property
    def lnprobability(self):
        return np.swapaxes(self.get_log_prob(), 0, 1)

    @property
    def acceptance_fraction(self):
        return self._naccepted / max(float(self._step_counter), 1.0)

    def get_autocorr_time(self, discard=0, thin=1, **kwargs):
        return thin * integrated_time(self.get_chain(discard=discard, thin=thin), **kwargs)
