"""Development probe (GPU box): device timings of every kernel family at a few
sizes, next to cuBLAS DGEMM / HBM copy yard-sticks.  Not part of the product."""
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alabi_b200 as ab
from alabi_b200 import _lib
from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb


def ev_time(fn, reps=3, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    return best


def main():
    out = {}
    lib = _lib.load()
    # yard-sticks
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    t = ev_time(lambda: torch.matmul(a, b), reps=3)
    out["cublas_dgemm_8192_tflops"] = 2 * n ** 3 / t * 1e-12
    t = ev_time(lambda: b.copy_(a), reps=5)
    out["copy_gbs"] = 2 * a.numel() * 8 / t * 1e-9
    del a, b
    print(json.dumps(out), flush=True)

    sizes = [int(s) for s in os.environ.get("PROBE_SIZES", "1024,4096,8192,16384").split(",")]
    for n in sizes:
        d = 10
        rng = np.random.default_rng(n)
        X = rng.uniform(-1, 1, size=(n, d))
        y = -0.5 * np.sum(X ** 2, axis=1) + 0.01 * rng.normal(size=n)
        k = ab.kernels.ExpSquaredKernel(metric=np.full(d, 4.0), ndim=d) * np.var(y)
        g = ab.GP(kernel=k, fit_mean=True, mean=np.median(y), white_noise=-6.0, fit_white_noise=True)
        g.compute(X)
        h = g._hd.h
        res = {"n": n}
        K = torch.empty((n, n), dtype=torch.float64, device="cuda")
        t = ev_time(lambda: lib.ab_gp_build_cov(h, _lib.ptr(K), 1), reps=5)
        res["cov_ms"] = t * 1e3
        res["cov_gbs"] = 8.0 * n * n / t * 1e-9
        del K
        t = ev_time(lambda: lib.ab_gp_factor(h), reps=3)
        res["factor_ms"] = t * 1e3
        res["factor_tflops"] = n ** 3 / 3 / t * 1e-12
        yd = torch.from_numpy(y).cuda()
        ll = ctypes.c_double()
        t = ev_time(lambda: lib.ab_gp_log_likelihood(h, _lib.ptr(yd), ctypes.byref(ll)), reps=3)
        res["factor+solve_ms(loglike after factor)"] = t * 1e3
        gr = (ctypes.c_double * (d + 3))()

        def full_grad():
            lib.ab_gp_factor(h)
            lib.ab_gp_grad_log_likelihood(h, _lib.ptr(yd), gr)
        t = ev_time(full_grad, reps=2)
        res["factor+grad_ms"] = t * 1e3
        res["factor+grad_tflops"] = n ** 3 / t * 1e-12
        m = 1 << 20 if n <= 4096 else 1 << 18
        Xq = torch.from_numpy(rng.uniform(-1, 1, size=(m, d))).cuda()
        mu = torch.empty(m, dtype=torch.float64, device="cuda")
        var = torch.empty(m, dtype=torch.float64, device="cuda")
        t = ev_time(lambda: lib.ab_gp_predict(h, _lib.ptr(Xq), m, _lib.ptr(mu), None), reps=3)
        res["predict_mean_pts_s"] = m / t
        mv = m if n <= 4096 else 148 * 128 * 2
        t = ev_time(lambda: lib.ab_gp_predict(h, _lib.ptr(Xq), mv, _lib.ptr(mu), _lib.ptr(var)), reps=2)
        res["predict_var_pts_s"] = mv / t
        res["predict_var_tflops"] = mv * float(n) ** 2 / t * 1e-12
        print(json.dumps(res), flush=True)
        del g

    # sampler: c2-like (N = 1000, d = 2, 1000 walkers)
    rng = np.random.default_rng(2)
    X = rng.uniform(-6, 6, size=(1000, 2))
    y = -0.5 * np.sum((X / 2.0) ** 2, axis=1)
    k = ab.kernels.Matern32Kernel(metric=np.full(2, 9.0), ndim=2) * np.var(y)
    g = ab.GP(kernel=k, fit_mean=True, mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
    g.compute(X)
    lp = SurrogateLogProb(g, y, [(-6, 6), (-6, 6)])
    for wpu in (0, 1, 2, 4, 8):
        s = EnsembleSampler(1000, 2, lp, seed=1, warps_per_unit=wpu)
        s.run_mcmc(rng.uniform(-5, 5, size=(1000, 2)), 50, store=False)
        s.run_mcmc(None, 2000, store=False)
        print(json.dumps({"ensemble_c2_wpu": wpu, "walker_steps_per_s": 1000 * 2000 / s.last_run_device_seconds,
                          "acc": float(s.acceptance_fraction.mean())}), flush=True)


if __name__ == "__main__":
    main()
