"""Per-phase device times of the full predictive covariance (ab_gp_predict_cov) and of the
multivariate-normal draws (ab_mvn_sample) on the GPU, at (N, M) = (1000, 1000), (4000, 2048) and
(8192, 4096) with d = 10 and ExpSquared, S = 1000 draws.

Whole calls are timed with CUDA events after warm-up (median of --reps).  Phases come from a separate
torch.profiler pass (CUDA activities; kernel durations summed per phase):
  panel     predict_mean_kernel + combine_splits_kernel      cross-covariance panel P and the mean
  W         tri_gemm_kernel (inside predict_cov)             W = L^-1 P, M N^2 flop (lower triangle)
  prior     scale_points_kernel + cov_kernel                 K(t, t)
  syrk      syrk_lower_kernel                                K(t, t) - W^T W, about M^2 N flop (lower tile pairs)
  diagonal  var_from_w_kernel + set_diag_kernel              sigma^2 from W
  mirror    mirror_lower_kernel + mirror_diag_tiles_kernel
  factor    mvn_pad_kernel + chol_dataflow_kernel            Cholesky of Sigma, M^3 / 3 flop
  draws     mvn_normals_kernel + tri_gemm_kernel + mvn_finish_kernel   Y = L Z, M^2 S flop
Flop rates are stated against the FP64 DMMA issue-rate peak measured in the same run
(ab_fp64_tensor_peak).  The first JSON line names the GPU and its power limit, read in the same run.

    python tools/predict_cov_probe.py [--reps 5] [--out FILE]
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
from alabi_b200 import _lib  # noqa: E402

SIZES = [(1000, 1000), (4000, 2048), (8192, 4096)]
D, S = 10, 1000
PHASES = {
    "panel": ("predict_mean_kernel", "combine_splits_kernel"),
    "W": ("tri_gemm_kernel",),
    "prior": ("scale_points_kernel", "cov_kernel"),
    "syrk": ("syrk_lower_kernel",),
    "diagonal": ("var_from_w_kernel", "set_diag_kernel"),
    "mirror": ("mirror_lower_kernel", "mirror_diag_tiles_kernel"),
    "factor": ("mvn_pad_kernel", "chol_dataflow_kernel"),
    "draws": ("mvn_normals_kernel", "tri_gemm_kernel", "mvn_finish_kernel"),
}


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = f"not read ({e})"
    pk = ctypes.c_double()
    _lib.check(_lib.load().ab_fp64_tensor_peak(0, ctypes.byref(pk)), "ab_fp64_tensor_peak")
    info["fp64_dmma_peak_tflops_measured"] = pk.value
    return info


def event_ms(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def kernel_ms(fn, phases):
    """Device time per phase (ms) of one call of fn, from torch.profiler kernel records."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in phases}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for k, names in phases.items():
            if any(nm in ev.name for nm in names):
                out[k] += ev.time_range.elapsed_us() / 1e3
                break
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = [gpu_info()]
    peak = lines[0]["fp64_dmma_peak_tflops_measured"]
    print(json.dumps(lines[0]), flush=True)
    lib = _lib.load()
    for n, m in SIZES:
        rng = np.random.default_rng(n)
        X = rng.uniform(-1, 1, size=(n, D))
        y = np.sin(X.sum(axis=1)) + 0.05 * rng.normal(size=n)
        g = ab.GP(kernel=ab.kernels.ExpSquaredKernel(metric=np.full(D, 2.0), ndim=D) * np.var(y), fit_mean=True,
                  mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
        g.compute(X)
        tq = torch.from_numpy(rng.uniform(-1, 1, size=(m, D))).cuda()
        g.predict(y, tq, return_cov=False)                       # targets set, L^-1 built by the warm-up below
        hd = g._hd
        mu = torch.empty(m, dtype=torch.float64, device="cuda")
        cov = torch.empty((m, m), dtype=torch.float64, device="cuda")
        out = torch.empty((S, m), dtype=torch.float64, device="cuda")
        info = ctypes.c_int()

        def pcov():
            _lib.check(lib.ab_gp_predict_cov(hd.h, _lib.ptr(tq), m, _lib.ptr(mu), _lib.ptr(cov), m), "ab_gp_predict_cov")

        def draw():
            rc = _lib.check(lib.ab_mvn_sample(hd.h, _lib.ptr(cov), m, m, _lib.ptr(mu), 1e-6 * g.kernel.spec()[1], S, 7,
                                              _lib.ptr(out), ctypes.byref(info)), "ab_mvn_sample")
            assert rc == 0, rc

        for _ in range(2):                                      # warm-up: modules, scratch, L^-1
            pcov()
            draw()
        torch.cuda.synchronize()
        t_cov = event_ms(pcov, args.reps)
        t_draw = event_ms(draw, args.reps)
        ph = kernel_ms(pcov, {k: PHASES[k] for k in ("panel", "W", "prior", "syrk", "diagonal", "mirror")})
        ph.update(kernel_ms(draw, {k: PHASES[k] for k in ("factor", "draws")}))
        flop = {"W": float(m) * n * n, "syrk": float(m) * m * n, "factor": float(m) ** 3 / 3.0,
                "draws": float(m) * m * S}
        rates = {k: {"tflops": flop[k] / (ph[k] * 1e-3) / 1e12, "of_dmma_peak": flop[k] / (ph[k] * 1e-3) / 1e12 / peak}
                 for k in flop if ph[k] > 0}
        rec = {"N": n, "M": m, "d": D, "S": S, "predict_cov_ms": t_cov, "mvn_sample_ms": t_draw,
               "phase_ms": ph, "rates": rates,
               "workspace_bytes_predict_cov": 16 * hd.lib.ab_gp_padded_size(hd.h) * ((m + 255) // 256 * 256)}
        lines.append(rec)
        print(json.dumps(rec), flush=True)
        del g
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
