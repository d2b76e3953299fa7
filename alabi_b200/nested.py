"""Nested sampling for ``SurrogateModel.run_dynesty`` (SURVEY 8f-2) when dynesty itself is not
importable, and the batching shim that feeds real dynesty when it is.

The reference hands ``self.like_fn`` to ``dynesty.DynamicNestedSampler`` (``mode="dynamic"``, the
default) or ``dynesty.NestedSampler`` (``mode="static"``) and reads
``results.{samples, logwt, logz, logzerr, niter}`` plus ``dynesty.utils.resample_equal``
(alabi/core.py:2549-2706); dynesty calls the likelihood one point at a time (or ``queue_size`` at a
time through ``pool.map``).  This module provides

* :class:`BatchedNestedSampler` — static nested sampling (Skilling 2006) and dynesty's *dynamic*
  scheme (Higson et al. 2019; Speagle 2020): a baseline run, then batches of extra live points over
  the likelihood range that carries the posterior mass (importance = ``pfrac`` posterior +
  (1 - ``pfrac``) evidence, the reference passes ``pfrac = 1``), merged by birth / death likelihood
  until the requested effective sample size is reached.  Replacement points come from constrained
  random walks (dynesty's ``sample="rwalk"``) or random-direction slice sampling
  (``sample="rslice"``), a whole batch of chains at a time:
* :class:`DeviceWalker` — surrogate likelihood with one of the two prior transforms the reference
  ships: the whole batch of ``walks``-step chains (or ``slices``-slice chains) is ONE kernel launch
  (``ab_nested_walk`` / ``ab_nested_rslice``), no host round trip per step;
* :class:`HostWalker` — any Python likelihood / prior transform (e.g. the true likelihood): chains
  advance in lock-step on the host, one batched likelihood call per walk step (per slice-sampling
  round);
* :class:`BatchPool` — ``pool``-shaped object for real dynesty: ``map`` turns the ``queue_size``
  points of one dynesty iteration into one batched surrogate predict (K3).

Volumes use ln X_i = sum_k ln(n_k / (n_k + 1)) with n_k the number of live points when sample k
died (from the birth / death likelihoods, so merged runs and the final live points need no special
case), weights w_i = L_i (X_{i-1} - X_i), and logzerr^2 = sum dH / n.
"""
import ctypes
import pickle
import warnings

import numpy as np

__all__ = ["BatchedNestedSampler", "DeviceWalker", "HostWalker", "BatchPool", "NestedResults", "resample_equal",
           "compute_weights", "rslice_scale"]

# Step-out moves and failed shrink draws allowed per slice (the caps of ab_nested_rslice): a chain
# that would need more stops at the end point of its last completed slice.
RSLICE_MAX_EXPAND = 1024
RSLICE_MAX_CONTRACT = 256


class NestedResults(dict):
    __getattr__ = dict.get


def resample_equal(samples, weights, rstate=None):
    """Systematic resampling to equally weighted samples (dynesty.utils.resample_equal)."""
    rstate = np.random.default_rng() if rstate is None else rstate
    w = np.asarray(weights, dtype=np.float64)
    w = w / w.sum()
    n = len(w)
    positions = (rstate.random() + np.arange(n)) / n
    idx = np.minimum(np.searchsorted(np.cumsum(w), positions), n - 1)
    out = np.asarray(samples)[idx]
    return out[rstate.permutation(n)]


def compute_weights(logl, birth):
    """Volumes, weights and evidence of a set of dead points given their death and birth
    log-likelihoods (any mixture of runs).  Returns dict(order, nlive, logvol, logwt, logz, logzerr)
    with arrays in death order."""
    logl = np.asarray(logl, dtype=np.float64)
    birth = np.asarray(birth, dtype=np.float64)
    order = np.argsort(logl, kind="stable")
    L = logl[order]
    sb = np.sort(birth)
    # alive when sample i dies: born strictly below L_i, not dead before it (ties die in order)
    born = np.searchsorted(sb, L, side="left")
    nlive = np.maximum(born - np.arange(len(L)), 1).astype(np.float64)
    dlv = np.log(nlive / (nlive + 1.0))
    logvol = np.cumsum(dlv)
    prev = np.concatenate([[0.0], logvol[:-1]])
    logdvol = prev + np.log1p(-np.exp(logvol - prev))          # ln (X_{i-1} - X_i)
    logwt = L + logdvol
    logz = np.logaddexp.accumulate(logwt)
    # information and its contribution to the evidence variance
    with np.errstate(invalid="ignore", over="ignore"):
        h_terms = np.where(np.isfinite(L), np.exp(logwt - logz[-1]) * L, 0.0)
    h_cum = np.cumsum(h_terms)                                  # running sum of w_i L_i / Z_final
    zfrac = np.exp(logz - logz[-1])
    with np.errstate(invalid="ignore", divide="ignore"):
        H = np.where(zfrac > 0, h_cum / zfrac - logz, 0.0)      # H_i = sum_{k<=i} (w_k / Z_i) L_k - ln Z_i
    H = np.maximum(np.nan_to_num(H, nan=0.0, posinf=0.0, neginf=0.0), 0.0)
    dH = np.diff(np.concatenate([[0.0], H]))
    logzvar = np.maximum(np.cumsum(dH / nlive), 0.0)           # signed increments: H / n for constant n
    return dict(order=order, nlive=nlive, logvol=logvol, logwt=logwt, logz=logz, logzerr=np.sqrt(logzvar), H=H)


# -------------------------------------------------------------------------------------------------
# walkers: produce replacement points inside the hard constraint
# -------------------------------------------------------------------------------------------------
def _builtin_transform(fn):
    """(kind, bounds, data) when ``fn`` is a functools.partial of one of the two prior transforms the
    reference ships (alabi/utility.py:278-345, 381-486); None otherwise."""
    from functools import partial
    from . import utility as ut
    if not isinstance(fn, partial):
        return None
    names = {ut.prior_transform_uniform: ("uniform", ("bounds",)), ut.prior_transform_normal: ("normal", ("bounds", "data"))}
    if fn.func not in names:
        return None
    kind, argn = names[fn.func]
    kw = dict(zip(argn, fn.args))
    kw.update(fn.keywords or {})
    if any(a not in kw for a in argn):
        return None
    return kind, np.asarray(kw["bounds"], dtype=np.float64), kw.get("data")


class HostWalker:
    """Random walks with an arbitrary Python likelihood and prior transform.

    ``loglike_batch`` maps (m, ndim) -> (m,).  ``prior_transform`` follows dynesty's contract — ONE
    1-D point per call — unless it is one of the reference's own (vectorised) transforms."""

    def __init__(self, loglike_batch, prior_transform, ndim, rng=None):
        self.loglike = loglike_batch
        self.ndim = int(ndim)
        self.rng = np.random.default_rng() if rng is None else rng
        self._pt = prior_transform
        self._vectorised = _builtin_transform(prior_transform) is not None
        self.ncall = 0

    def transform(self, u):
        u = np.atleast_2d(u)
        if self._vectorised:
            return np.atleast_2d(self._pt(u))
        return np.array([np.asarray(self._pt(row), dtype=np.float64).reshape(-1) for row in u]).reshape(len(u), self.ndim)

    def like(self, theta):
        self.ncall += len(theta)
        return np.asarray(self.loglike(theta), dtype=np.float64).reshape(-1)

    def initial(self, n):
        u = self.rng.random((n, self.ndim))
        theta = self.transform(u)
        return u, theta, self.like(theta)

    def walk(self, u0, theta0, logl0, lmin, scale, chol, walks):
        u, theta, logl = u0.copy(), theta0.copy(), logl0.copy()
        k, d = u.shape
        nacc = 0
        for _ in range(int(walks)):
            prop = u + scale * (self.rng.standard_normal((k, d)) @ chol.T)
            inside = np.all((prop > 0.0) & (prop < 1.0), axis=1)
            if inside.any():
                t_in = self.transform(prop[inside])
                l_in = self.like(t_in)
                ok_in = l_in > lmin
                idx = np.nonzero(inside)[0][ok_in]
                u[idx], theta[idx], logl[idx] = prop[idx], t_in[ok_in], l_in[ok_in]
                nacc += int(ok_in.sum())
        return u, theta, logl, nacc / float(max(k * int(walks), 1))

    def _rslice_chain(self, c, u, theta, logl, counts, lmin, scale, chol, slices):
        """Slice-sampling state machine of chain ``c`` (the algorithm of ``ab_nested_rslice``, with
        draws from ``self.rng``): yields each in-cube proposal, is sent back its (theta, logl)."""
        d = self.ndim
        v = None

        def F(x):
            # point u + x v with its image and likelihood; outside the unit cube: -inf, no call
            p = u[c] + x * v
            if np.all((p > 0.0) & (p < 1.0)):
                th, y = yield p
                return p, th, y
            return p, None, -np.inf
        for _ in range(int(slices)):
            z = self.rng.standard_normal(d)
            v = (chol @ z) * (scale / np.sqrt(z @ z))
            r0 = self.rng.random()
            xl, xr = -r0, 1.0 - r0
            nexp = 0
            for left in (True, False):
                while True:
                    _, _, y = yield from F(xl if left else xr)
                    if not y > lmin:
                        break
                    if nexp == RSLICE_MAX_EXPAND:
                        return
                    nexp += 1
                    counts[c, 1] += 1
                    if left:
                        xl -= 1.0
                    else:
                        xr += 1.0
            ncon = 0
            while True:
                x = xl + self.rng.random() * (xr - xl)
                p, th, y = yield from F(x)
                if y > lmin:
                    u[c], theta[c], logl[c] = p, th, y
                    counts[c, 0] += 1
                    break
                ncon += 1
                counts[c, 2] += 1
                if x < 0.0:
                    xl = x
                elif x > 0.0:
                    xr = x
                if ncon == RSLICE_MAX_CONTRACT:
                    return

    def rslice(self, u0, theta0, logl0, lmin, scale, chol, slices):
        """``slices`` random-direction slices per chain (dynesty's ``sample="rslice"``).  All
        unfinished chains advance in lock step, one batched likelihood call per round.  Returns
        (u, theta, logl, counts) with counts (k, 4): slices completed, nexpand, ncontract, evaluations."""
        u, theta, logl = u0.copy(), theta0.copy(), logl0.copy()
        k = len(u)
        counts = np.zeros((k, 4), dtype=np.int64)
        chains = [self._rslice_chain(c, u, theta, logl, counts, lmin, scale, chol, slices) for c in range(k)]

        def step(c, sent):
            try:
                return chains[c].send(sent)
            except StopIteration:
                return None
        pending = {c: p for c in range(k) if (p := step(c, None)) is not None}
        while pending:
            idx = list(pending)
            th = self.transform(np.array([pending[c] for c in idx]))
            y = self.like(th)
            counts[idx, 3] += 1
            pending = {c: p for j, c in enumerate(idx) if (p := step(c, (th[j], y[j]))) is not None}
        return u, theta, logl, counts


def rslice_scale(scale, counts):
    """Slice-scale update after one batch: scale * 2 E / (E + C) with E expansions and C
    contractions summed over the batch (dynesty's rule as recalled: a window that had to grow asks for
    a larger scale, one that had to shrink for a smaller), kept in [1e-6, 10]."""
    e, c = float(np.sum(counts[:, 1])), float(np.sum(counts[:, 2]))
    if e + c == 0.0:
        return float(scale)
    return float(np.clip(scale * 2.0 * e / (e + c), 1e-6, 10.0))


class DeviceWalker:
    """Random walks on the surrogate, one launch per batch (``ab_nested_walk``).

    ``logprob`` is an ``alabi_b200.ensemble.SurrogateLogProb`` (GP + theta / y scalers: the
    surrogate likelihood itself, its prior terms are not used); the prior transform is the uniform
    box ``bounds`` or, with ``prior_data``, ``ut.prior_transform_normal``."""

    def __init__(self, logprob, bounds, prior_data=None, seed=None):
        import torch
        from . import _lib
        self._lib = _lib
        self.lp = logprob
        self.gp = logprob.gp
        self.bounds = np.asarray(bounds, dtype=np.float64).reshape(-1, 2)
        self.ndim = len(self.bounds)
        self.prior_mu, self.prior_sd = np.zeros(self.ndim), np.zeros(self.ndim)
        if prior_data is not None:
            for k, (m, sd) in enumerate(prior_data):
                if m is not None:
                    self.prior_mu[k], self.prior_sd[k] = float(m), float(sd)
        self.seed = int(np.random.SeedSequence().entropy % (2 ** 63)) if seed is None else int(seed)
        self.rng = np.random.default_rng(self.seed)
        self.counter = 0
        self.ncall = 0
        self.gp.recompute()
        self.gp._set_targets(self.lp.y)
        self._torch = torch
        self._dev = f"cuda:{self.gp._hd.device}"

    def transform(self, u):
        from scipy.stats import norm
        u = np.atleast_2d(u)
        b = self.bounds
        out = (b[:, 1] - b[:, 0]) * u + b[:, 0]
        for k in np.nonzero(self.prior_sd > 0)[0]:
            out[:, k] = norm.ppf(u[:, k], self.prior_mu[k], self.prior_sd[k])
        return out

    def like(self, theta):
        """Surrogate log-likelihood of a batch (K3 mean through the scalers)."""
        lp = self.lp
        theta = np.atleast_2d(theta)
        self.ncall += len(theta)
        ys = self.gp.predict(lp.y, theta * lp.theta_scale + lp.theta_offset, return_cov=False)
        return ys * lp.y_scale + lp.y_offset if lp.y_kind == 0 else (-10.0 ** ys if lp.y_kind == 1 else 10.0 ** ys)

    def initial(self, n):
        u = self.rng.random((n, self.ndim))
        theta = self.transform(u)
        return u, theta, self.like(theta)

    def _launch(self, entry, u0, theta0, logl0, lmin, scale, chol, steps, ncount, chain_offset=0):
        """One ``entry`` launch (ab_nested_walk / ab_nested_rslice) over the batch: the end points on the
        host and the device counts (k x ncount int32)."""
        torch, _lib = self._torch, self._lib
        hd = self.gp._hd
        k, d = u0.shape
        cfg = _lib.NestedConfig()
        cfg.nchains, cfg.walks, cfg.y_kind = int(k), int(steps), int(self.lp.y_kind)
        cfg.use_normal_prior = int(np.any(self.prior_sd > 0))
        cfg.scale, cfg.lmin = float(scale), float(lmin) if np.isfinite(lmin) else -1.7976931348623157e308
        cfg.seed, cfg.counter, cfg.chain_offset = self.seed, self.counter, int(chain_offset)
        self.counter += 1
        cfg.y_scale, cfg.y_offset = self.lp.y_scale, self.lp.y_offset
        for i in range(d):
            cfg.lo[i], cfg.hi[i] = self.bounds[i, 0], self.bounds[i, 1]
            cfg.prior_mu[i], cfg.prior_sd[i] = self.prior_mu[i], self.prior_sd[i]
            cfg.theta_scale[i], cfg.theta_offset[i] = self.lp.theta_scale[i], self.lp.theta_offset[i]
        cl = np.ascontiguousarray(np.tril(chol), dtype=np.float64).reshape(-1)
        ctypes.memmove(cfg.chol, cl.ctypes.data, cl.nbytes)
        # one device block in, one out: [u | theta | logl] and the counts
        blk = torch.from_numpy(np.concatenate([u0.reshape(-1), theta0.reshape(-1), logl0.reshape(-1)])).to(self._dev)
        du, dth, dl = blk[:k * d], blk[k * d:2 * k * d], blk[2 * k * d:]
        cnt = torch.zeros(k * ncount, dtype=torch.int32, device=self._dev)
        _lib.check(getattr(hd.lib, entry)(hd.h, ctypes.byref(cfg), _lib.ptr(du), _lib.ptr(dl), _lib.ptr(dth), _lib.ptr(cnt)),
                   entry)
        host = blk.cpu().numpy()
        return host[:k * d].reshape(k, d), host[k * d:2 * k * d].reshape(k, d), host[2 * k * d:], cnt

    def walk(self, u0, theta0, logl0, lmin, scale, chol, walks):
        k = len(u0)
        u, theta, logl, nacc = self._launch("ab_nested_walk", u0, theta0, logl0, lmin, scale, chol, walks, 1)
        self.ncall += k * int(walks)
        return u, theta, logl, float(nacc.sum().item()) / float(max(k * int(walks), 1))

    def rslice(self, u0, theta0, logl0, lmin, scale, chol, slices, chain_offset=0):
        """``slices`` random-direction slices per chain, one launch (``ab_nested_rslice``); returns
        (u, theta, logl, counts) as :meth:`HostWalker.rslice`.  Row i draws the random numbers of
        chain ``chain_offset + i``, so a sub-batch reproduces its rows of a larger batch."""
        u, theta, logl, cnt = self._launch("ab_nested_rslice", u0, theta0, logl0, lmin, scale, chol, slices, 4,
                                           chain_offset)
        counts = cnt.cpu().numpy().reshape(-1, 4).astype(np.int64)
        self.ncall += int(counts[:, 3].sum())
        return u, theta, logl, counts


class BatchPool:
    """``pool`` for real dynesty (``NestedSampler(..., pool=BatchPool(f), queue_size=q)``): dynesty
    maps its likelihood wrapper over the ``queue_size`` points proposed in one iteration; when that
    wrapper is (a wrapper of) ``f.one`` the points are stacked and evaluated by ONE batched call
    ``f.batch`` (one K3 launch) instead of ``queue_size`` one-point predicts.  Anything else is
    mapped serially."""

    def __init__(self, like, size=64):
        self.like = like
        self.size = int(size)

    def map(self, func, iterable):
        items = list(iterable)
        target = getattr(func, "func", func)
        if len(items) > 0 and (target is self.like or getattr(target, "__self__", None) is self.like) \
                and not getattr(func, "args", None) and not getattr(func, "kwargs", None):
            pts = np.array([np.asarray(p, dtype=np.float64).reshape(-1) for p in items])
            return [float(v) for v in self.like.batch(pts)]
        return [func(p) for p in items]

    def close(self):
        pass

    def join(self):
        pass


class BatchLikelihood:
    """Callable the samplers see: ``__call__(theta)`` for one point (dynesty's contract),
    ``batch(thetas)`` for many (used by :class:`BatchPool` and the built-in sampler)."""

    def __init__(self, batch_fn):
        self.batch = batch_fn

    def __call__(self, theta):
        return float(np.asarray(self.batch(np.asarray(theta, dtype=np.float64).reshape(1, -1))).reshape(-1)[0])


# -------------------------------------------------------------------------------------------------
# the sampler
# -------------------------------------------------------------------------------------------------
class BatchedNestedSampler:
    """``walker``: :class:`DeviceWalker` or :class:`HostWalker`.  ``nbatch`` chains are advanced
    together whenever the queue of replacement candidates runs dry, by ``walks`` random-walk steps
    (``sample="rwalk"``) or ``slices`` random-direction slices (``sample="rslice"``)."""

    def __init__(self, walker, ndim, nlive=500, walks=25, nbatch=None, rstate=None, max_failed_rounds=50,
                 sample="rwalk", slices=5):
        if sample not in ("rwalk", "rslice"):
            raise ValueError(f"sample={sample!r}: choose 'rwalk' or 'rslice'")
        if int(slices) < 1:
            raise ValueError(f"slices={slices!r}: at least one slice per chain")
        self.walker = walker
        self.ndim = int(ndim)
        self.nlive = int(nlive)
        self.walks = int(walks)
        self.sample = sample
        self.slices = int(slices)
        self.nbatch = int(nbatch) if nbatch else max(self.nlive // 4, 32)
        self.rng = np.random.default_rng(rstate)
        self.max_failed_rounds = int(max_failed_rounds)
        self.results = None
        self.scale = 1.0
        self.checkpoint = None          # optional callable(sampler, iteration)
        self.checkpoint_every = None

    @property
    def ncall(self):
        return self.walker.ncall

    # ---------------------------------------------------------------------------------------------
    def _proposal_chol(self, live_u):
        d = self.ndim
        cov = np.cov(live_u.T) + 1e-12 * np.eye(d) if d > 1 else np.atleast_2d(np.var(live_u) + 1e-12)
        try:
            return np.linalg.cholesky(cov)
        except np.linalg.LinAlgError:
            return np.sqrt(np.diag(np.diag(cov)))

    def _candidates(self, live_u, live_t, live_l, lmin):
        """One batch of walks from random live points; adapts the proposal scale."""
        k = self.nbatch
        start = self.rng.integers(0, len(live_l), size=k)
        if self.sample == "rslice":
            u, theta, logl, counts = self.walker.rslice(live_u[start], live_t[start], live_l[start], lmin, self.scale,
                                                        self._proposal_chol(live_u), self.slices)
            self.scale = rslice_scale(self.scale, counts)
            moved = counts[:, 0] > 0             # a chain with no completed slice is a copy of a live point
            return [(u[i], theta[i], logl[i]) for i in range(k) if moved[i] and logl[i] > lmin]
        u, theta, logl, acc = self.walker.walk(live_u[start], live_t[start], live_l[start], lmin, self.scale,
                                               self._proposal_chol(live_u), self.walks)
        self.scale = float(np.clip(self.scale * np.exp((acc - 0.5) / max(self.ndim, 1)), 1e-6, 10.0))
        # a chain that never moved is a copy of a live point: not a new sample
        moved = np.any(u != live_u[start], axis=1)
        return [(u[i], theta[i], logl[i]) for i in range(k) if moved[i] and logl[i] > lmin]

    def _segment(self, live_u, live_t, live_l, live_b, stop, maxiter, maxcall, it0=0):
        """Kill worst points / replace them until ``stop(lmin, logvol_est, live_l, it)`` says so, then
        retire the remaining live points.  Returns the dead points of this segment."""
        dead_u, dead_t, dead_l, dead_b = [], [], [], []
        queue, it, failed = [], 0, 0
        while it < maxiter:
            worst = int(np.argmin(live_l))
            lmin = live_l[worst]
            if stop(lmin, live_l, it):
                break
            dead_u.append(live_u[worst].copy()); dead_t.append(live_t[worst].copy())
            dead_l.append(lmin); dead_b.append(live_b[worst])
            it += 1
            new = None
            while new is None:
                while queue:
                    cand = queue.pop()
                    if cand[2] > lmin:
                        new = cand
                        break
                if new is not None:
                    break
                queue = self._candidates(live_u, live_t, live_l, lmin)
                failed = failed + 1 if not queue else 0
                if failed >= self.max_failed_rounds or (maxcall and self.ncall > maxcall):
                    break
            if new is None:
                # likelihood plateau / exhausted budget: the worst point stays dead, the run ends
                if failed >= self.max_failed_rounds:
                    moves = f"{self.slices} slices" if self.sample == "rslice" else f"{self.walks} walk steps"
                    warnings.warn(f"nested sampling: no point above L = {lmin:.6g} found in {failed} rounds of "
                                  f"{self.nbatch} x {moves} (likelihood plateau?); ending the run")
                live_u, live_t = np.delete(live_u, worst, axis=0), np.delete(live_t, worst, axis=0)
                live_l, live_b = np.delete(live_l, worst), np.delete(live_b, worst)
                break
            live_u[worst], live_t[worst], live_l[worst], live_b[worst] = new[0], new[1], new[2], lmin
            if self.checkpoint is not None and self.checkpoint_every and (it0 + it) % self.checkpoint_every == 0:
                self._partial = (dead_u, dead_t, dead_l, dead_b)
                self.checkpoint(self, it0 + it)
        for i in np.argsort(live_l):
            dead_u.append(live_u[i].copy()); dead_t.append(live_t[i].copy()); dead_l.append(live_l[i]); dead_b.append(live_b[i])
        return (np.array(dead_u).reshape(-1, self.ndim), np.array(dead_t).reshape(-1, self.ndim), np.array(dead_l),
                np.array(dead_b), it)

    def _finish(self, U, T, L, B, niter, extra=None):
        w = compute_weights(L, B)
        o = w["order"]
        self.results = NestedResults(samples=T[o], samples_u=U[o], logl=L[o], birth_logl=B[o], logwt=w["logwt"],
                                     logz=w["logz"], logzerr=w["logzerr"], logvol=w["logvol"], samples_n=w["nlive"],
                                     information=w["H"], niter=int(niter), ncall=int(self.ncall),
                                     eff=100.0 * niter / max(self.ncall, 1), nlive=self.nlive)
        if extra:
            self.results.update(extra)
        return self.results

    # ---------------------------------------------------------------------------------------------
    def run_nested(self, dlogz=0.01, maxiter=None, maxcall=None, print_progress=False, nlive=None):
        """Static nested sampling: ``nlive`` points, stop when the live points can add less than
        ``dlogz`` to ln Z."""
        nl = int(nlive or self.nlive)
        u, t, l = self.walker.initial(nl)
        b = np.full(nl, -np.inf)
        state = {"logz": -1e300, "logvol": 0.0}

        def stop(lmin, live_l, it):
            # evidence so far and the bound on what is left: max(L_live) X
            if it > 0:
                dlv = np.log1p(-np.exp(-1.0 / nl))
                state["logz"] = np.logaddexp(state["logz"], state["logvol"] + dlv + state["last"])
                state["logvol"] -= 1.0 / nl
            state["last"] = lmin
            if it == 0:
                return False
            dz = np.logaddexp(state["logz"], np.max(live_l) + state["logvol"]) - state["logz"]
            if print_progress and it % 500 == 0:
                print(f"iter {it} logz {state['logz']:.3f} dlogz {dz:.4f} ncall {self.ncall}")
            return dz < dlogz
        U, T, L, B, it = self._segment(u, t, l, b, stop, int(maxiter) if maxiter else 10 ** 9, maxcall)
        return self._finish(U, T, L, B, it)

    def run_dynamic(self, dlogz_init=0.01, nlive_init=None, nlive_batch=None, maxiter=None, maxcall=None, maxbatch=None,
                    n_effective=None, pfrac=1.0, maxfrac=0.8, pad=1, print_progress=False):
        """Dynamic nested sampling: baseline run (``nlive_init`` points, ``dlogz_init``), then batches of
        ``nlive_batch`` points over the likelihood range where the importance
        ``pfrac`` * posterior + (1 - ``pfrac``) * evidence exceeds ``maxfrac`` of its maximum (widened by
        ``pad`` samples), until the posterior's effective sample size reaches ``n_effective``
        (dynesty's default: max(ndim^2, 10000)), ``maxbatch`` batches, ``maxiter`` or ``maxcall``."""
        nl0 = int(nlive_init or self.nlive)
        nlb = int(nlive_batch or self.nlive)
        maxiter = int(maxiter) if maxiter else 10 ** 9
        maxbatch = 200 if maxbatch is None else int(maxbatch)
        n_eff_target = max(self.ndim ** 2, 10000) if n_effective is None else float(n_effective)
        res = self.run_nested(dlogz=dlogz_init, maxiter=maxiter, maxcall=maxcall, print_progress=print_progress, nlive=nl0)
        U, T, L, B = res.samples_u, res.samples, res.logl, res.birth_logl
        niter, nb = res.niter, 0
        neff = 0.0
        while nb < maxbatch and niter < maxiter and not (maxcall and self.ncall > maxcall):
            w = compute_weights(L, B)
            o = w["order"]
            U, T, L, B = U[o], T[o], L[o], B[o]
            logwt, logz = w["logwt"], w["logz"]
            post = np.exp(logwt - logz[-1])
            neff = float(post.sum() ** 2 / np.sum(post ** 2))
            if neff >= n_eff_target:
                break
            # importance of every dead point: posterior mass and (remaining) evidence
            zrem = 1.0 - np.exp(logz - logz[-1])
            imp = pfrac * post / post.sum() + (1.0 - pfrac) * (zrem / max(zrem.sum(), 1e-300))
            sel = np.nonzero(imp > maxfrac * imp.max())[0]
            i_lo, i_hi = max(int(sel[0]) - pad, 0), min(int(sel[-1]) + pad, len(L) - 1)
            l_lo = L[i_lo] if i_lo > 0 else -np.inf
            l_hi = L[i_hi]
            # starting live set: points uniformly distributed inside L > l_lo
            if np.isfinite(l_lo):
                alive = np.nonzero((B < l_lo) & (L > l_lo))[0]   # alive when the contour l_lo was crossed
                if len(alive) < 2:
                    alive = np.nonzero(L > l_lo)[0][:max(2, nlb)]
                start = self.rng.choice(alive, size=nlb, replace=True)
                chol = self._proposal_chol(U[alive]) if len(alive) > self.ndim else np.eye(self.ndim) * 0.1
                if self.sample == "rslice":
                    u, t, l, _ = self.walker.rslice(U[start], T[start], L[start], l_lo, self.scale, chol, self.slices)
                else:
                    u, t, l, _ = self.walker.walk(U[start], T[start], L[start], l_lo, self.scale, chol,
                                                  max(self.walks, 2 * self.ndim))
                b = np.full(nlb, l_lo)
            else:
                u, t, l = self.walker.initial(nlb)
                b = np.full(nlb, -np.inf)
            stop = lambda lmin, live_l, it, l_hi=l_hi: lmin >= l_hi      # the batch ends at the upper contour
            u2, t2, l2, b2, it = self._segment(u, t, l, b, stop, maxiter - niter, maxcall, it0=niter)
            U, T = np.vstack([U, u2]), np.vstack([T, t2])
            L, B = np.concatenate([L, l2]), np.concatenate([B, b2])
            niter += it
            nb += 1
            if it == 0:
                break                                            # nothing left to add in that range
            if print_progress:
                print(f"batch {nb}: L in ({l_lo:.4g}, {l_hi:.4g}), {len(l2)} samples, ESS {neff:.0f}, ncall {self.ncall}")
        out = self._finish(U, T, L, B, niter, extra={"nbatch": nb})
        post = np.exp(out.logwt - out.logz[-1])
        out["n_effective"] = float(post.sum() ** 2 / np.sum(post ** 2))
        return out

    # ---------------------------------------------------------------------------------------------
    def __getstate__(self):
        st = self.__dict__.copy()
        st["walker"] = None              # device handles / user callables do not travel
        st["checkpoint"] = None
        return st


def save_checkpoint(path):
    """Checkpoint callback for ``BatchedNestedSampler.checkpoint``: pickles the dead points so far."""
    def cb(sampler, it):
        du, dt, dl, db = sampler._partial
        with open(path, "wb") as f:
            pickle.dump({"iteration": it, "samples_u": np.array(du), "samples": np.array(dt), "logl": np.array(dl),
                         "birth_logl": np.array(db), "scale": sampler.scale, "ncall": sampler.ncall}, f)
    return cb
