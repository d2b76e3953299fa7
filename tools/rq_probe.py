"""Cost of the rational quadratic kernel (RQ, log_alpha = 0) against ExpSquared on identical inputs,
on the GPU: covariance build and gradient at N = 8192, d = 10 (the c4 training set); predict mean +
variance for one 18944-point wave (148 SMs x 128) on the c4 model; sampler walker-steps/s at the c5
shape (N = 16384, d = 20) with 8192 and 65536 walkers and at the c2 shape (N = 1000, d = 2, 1000
walkers).  Device times come from the library's per-family event marks (ab_gp_set_profiling /
ab_gp_profile_read) and, for the gradient and the sampler, from CUDA events around the calls.  The
two kernels alternate (ES, RQ, ES, RQ) so that run-to-run spread shows.  Prints JSON lines, the
first with the GPU name and power limit read in the same run.

    python tools/rq_probe.py [--reps 2]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alabi_b200 as ab  # noqa: E402
from alabi_b200 import _lib, workloads  # noqa: E402
from alabi_b200.ensemble import EnsembleSampler, SurrogateLogProb  # noqa: E402

PROF_COV, PROF_FACTOR, PROF_PANEL, PROF_VAR, PROF_ENS = range(5)
WAVE = 148 * 128


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read ({e})"
    return info


def make_gp(cfg, rq, n=None):
    hp = cfg["hp"]
    d = cfg["ndim"]
    base = (ab.kernels.RationalQuadraticKernel(0.0, metric=np.exp(hp["log_M"]), ndim=d) if rq else
            ab.kernels.ExpSquaredKernel(metric=np.exp(hp["log_M"]), ndim=d))
    return ab.GP(kernel=base * hp["amp"], fit_mean=True, mean=hp["mean"], white_noise=hp["white_noise"],
                 fit_white_noise=True)


def prof_read(h, fam):
    ms, cnt = ctypes.c_double(), ctypes.c_longlong()
    _lib.check(_lib.load().ab_gp_profile_read(h, fam, ctypes.byref(ms), ctypes.byref(cnt)), "ab_gp_profile_read")
    return ms.value, cnt.value


def events(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def gp_families(rq, reps):
    """K1 covariance (inside ab_gp_factor), K2 gradient and one predict wave on the c4 model."""
    lib = _lib.load()
    cfg = workloads.make_config("c4")
    g = make_gp(cfg, rq)
    g.compute(cfg["X"])
    h = g._hd.h
    y = torch.from_numpy(cfg["y"]).cuda()
    out = (ctypes.c_double * (cfg["ndim"] + 4))()
    _lib.check(lib.ab_gp_grad_log_likelihood(h, _lib.ptr(y), out), "grad")          # warm-up: K^-1, alpha
    lib.ab_gp_set_profiling(h, 1)
    for _ in range(reps):
        _lib.check(lib.ab_gp_factor(h), "factor")
    cov_ms, ncov = prof_read(h, PROF_COV)
    fac_ms, nfac = prof_read(h, PROF_FACTOR)
    _lib.check(lib.ab_gp_set_targets(h, _lib.ptr(y)), "targets")
    _lib.check(lib.ab_gp_grad_log_likelihood(h, None, out), "grad")                  # K^-1 of the new factor
    grad_ms = min(events(lambda: _lib.check(lib.ab_gp_grad_log_likelihood(h, None, out), "grad")) for _ in range(reps))
    rng = np.random.default_rng(44)
    xq = torch.from_numpy(rng.uniform(-3, 3, size=(WAVE, cfg["ndim"]))).cuda()
    mu = torch.empty(WAVE, dtype=torch.float64, device="cuda")
    var = torch.empty(WAVE, dtype=torch.float64, device="cuda")
    _lib.check(lib.ab_gp_predict(h, _lib.ptr(xq), WAVE, _lib.ptr(mu), _lib.ptr(var)), "predict")   # warm-up
    prof_read(h, PROF_PANEL), prof_read(h, PROF_VAR)
    tot = min(events(lambda: _lib.check(lib.ab_gp_predict(h, _lib.ptr(xq), WAVE, _lib.ptr(mu), _lib.ptr(var)), "predict"))
              for _ in range(reps))
    panel_ms, npanel = prof_read(h, PROF_PANEL)
    var_ms, nvar = prof_read(h, PROF_VAR)
    lib.ab_gp_set_profiling(h, 0)
    return {"cov_ms": cov_ms / ncov, "factor_ms": fac_ms / nfac, "grad_ms": grad_ms,
            "predict_wave_ms": tot, "predict_mean_panel_ms": panel_ms / max(npanel, 1),
            "predict_var_ms": var_ms / max(nvar, 1)}


def sampler(rq, name, nwalkers, nsteps):
    cfg = workloads.make_config(name)
    g = make_gp(cfg, rq)
    g.compute(cfg["X"])
    lp = SurrogateLogProb(g, cfg["y"], cfg["bounds"])
    rng = np.random.default_rng(7)
    c = cfg["bounds"]
    p0 = rng.uniform(0.5 * c[:, 0], 0.5 * c[:, 1], size=(nwalkers, cfg["ndim"]))
    s = EnsembleSampler(nwalkers, cfg["ndim"], lp, seed=11)
    s.run_mcmc(p0, max(2, nsteps // 10), store=False)                                  # warm-up
    s.run_mcmc(None, nsteps, store=False)
    return nwalkers * nsteps / s.last_run_device_seconds


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=2, help="timed repetitions per measurement (the minimum is reported)")
    ap.add_argument("--alternations", type=int, default=2, help="ES / RQ alternations")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rq_probe.py needs a CUDA device")
    print(json.dumps(gpu_info()), flush=True)
    for rnd in range(args.alternations):
        for rq in (False, True):
            kern = "RationalQuadratic" if rq else "ExpSquared"
            res = {"round": rnd, "kernel": kern, "c4_N8192_d10": gp_families(rq, args.reps)}
            res["c5_N16384_d20_w8192_walker_steps_s"] = sampler(rq, "c5", 8192, 60)
            res["c5_N16384_d20_w65536_walker_steps_s"] = sampler(rq, "c5", 65536, 12)
            res["c2_N1000_d2_w1000_walker_steps_s"] = sampler(rq, "c2", 1000, 1000)
            print(json.dumps(res), flush=True)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
