import os, sys, json, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alabi_b200 as ab
from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb
rng = np.random.default_rng(2)
X = rng.uniform(-6, 6, size=(1000, 2))
y = -0.5 * np.sum((X / 2.0) ** 2, axis=1)
k = ab.kernels.Matern32Kernel(metric=np.full(2, 9.0), ndim=2) * np.var(y)
g = ab.GP(kernel=k, fit_mean=True, mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
g.compute(X)
lp = SurrogateLogProb(g, y, [(-6, 6), (-6, 6)])
p0 = rng.uniform(-5, 5, size=(1000, 2))
for sched in ((1, 0) if not os.environ.get('ENS_SKIP_SMALL') else ()):
    for wpu in (0, 4, 8):
        s = EnsembleSampler(1000, 2, lp, seed=1, warps_per_unit=wpu, schedule=sched)
        s.run_mcmc(p0, 50, store=False)
        st = s.run_mcmc(None, 2000, store=False)
        print(json.dumps({"schedule": sched, "wpu": wpu, "walker_steps_per_s": 1000 * 2000 / s.last_run_device_seconds,
                          "us_per_step": s.last_run_device_seconds / 2000 * 1e6, "state_sum": float(st.coords.sum())}), flush=True)
# other small-ensemble shapes (the reference's usual sizes): walkers x training points
for nw_s, n_s in (((100, 150), (200, 1000), (1000, 4000), (2000, 1000)) if not os.environ.get('ENS_SKIP_SMALL') else ()):
    Xs = rng.uniform(-6, 6, size=(n_s, 2)); ys = -0.5 * np.sum((Xs / 2.0) ** 2, axis=1)
    gs = ab.GP(kernel=ab.kernels.Matern32Kernel(metric=np.full(2, 9.0), ndim=2) * np.var(ys), fit_mean=True, mean=np.median(ys), white_noise=-8.0, fit_white_noise=True)
    gs.compute(Xs)
    lps = SurrogateLogProb(gs, ys, [(-6, 6), (-6, 6)])
    p0s = rng.uniform(-5, 5, size=(nw_s, 2))
    for sched in (1, 0):
        s = EnsembleSampler(nw_s, 2, lps, seed=1, schedule=sched)
        s.run_mcmc(p0s, 50, store=False)
        s.run_mcmc(None, 2000, store=False)
        print(json.dumps({"nw": nw_s, "n": n_s, "schedule": sched, "walker_steps_per_s": nw_s * 2000 / s.last_run_device_seconds,
                          "us_per_step": s.last_run_device_seconds / 2000 * 1e6}), flush=True)
if os.environ.get('ENS_SMALL_ONLY'):
    sys.exit(0)

# c5-like per-GPU share: N = 16384, d = 20, 8192 walkers
import time
d, n, nw = 20, 16384, int(os.environ.get('ENS_NW', '8192'))
X = rng.uniform(0, 1, size=(n, d))
y = -0.5 * np.sum(((X - 0.5) / 0.2) ** 2, axis=1)
k = ab.kernels.ExpSquaredKernel(metric=np.full(d, 4.0), ndim=d) * np.var(y)
g = ab.GP(kernel=k, fit_mean=True, mean=np.median(y), white_noise=-6.0, fit_white_noise=True)
g.compute(X)
lp = SurrogateLogProb(g, y, [(0, 1)] * d)
s = EnsembleSampler(nw, d, lp, seed=1)
s.run_mcmc(rng.uniform(0.3, 0.7, size=(nw, d)), 2, store=False)
s.run_mcmc(None, 20, store=False)
ws = nw * 20 / s.last_run_device_seconds
print(json.dumps({"c5_like": True, "walker_steps_per_s": ws, "fp64_instr_rate_frac": ws * n * (2 * d + 22) / 1.8e13,
                  "acc": float(s.acceptance_fraction.mean())}), flush=True)
