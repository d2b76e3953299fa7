"""Random-direction slice sampling (ab_nested_rslice) against the random walk (ab_nested_walk) on
two surrogates: c3 (2-D eggbox, Matern-5/2, N = 4000, training points resident in shared memory)
and a d = 24 ExpSquared surrogate of a Gaussian log-likelihood at N = 8192 (chunked).

Per surrogate:
  launch   rwalk (walks = 25) and rslice (slices = 5) over the same NCHAINS start points inside
           L > lmin (lmin = median of L at uniform draws), proposal factor from their covariance,
           scale 1.  Kernel time from torch.profiler (CUDA activities, summed kernel durations of
           REPS launches after a warm-up launch).  Evaluations: nchains x walks for rwalk (every
           lane evaluates every step), the reported counts for rslice.  Lane utilisation of rslice:
           evaluations / (32 x rounds), a CTA running as many rounds as its busiest chain has
           evaluations.
  e2e      BatchedNestedSampler.run_nested wall time (host clock, the run ends in device
           synchronisation), ncall and ln Z of both methods at the same dlogz.

The first JSON line names the GPU and its power limit, read in the same run.

    python tools/nested_rslice_probe.py [--reps 5] [--out profiles/nested_rslice_probe.txt]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alabi_b200 as ab  # noqa: E402
from alabi_b200 import workloads  # noqa: E402
from alabi_b200.ensemble import SurrogateLogProb  # noqa: E402
from alabi_b200.nested import BatchedNestedSampler, DeviceWalker  # noqa: E402

NCHAINS = 148 * 32          # one CTA per SM
WALKS, SLICES = 25, 5


def surrogates():
    cfg = workloads.make_config("c3")
    g = workloads.build_gp(cfg)
    g.compute(cfg["X"])
    yield "c3", SurrogateLogProb(g, cfg["y"], cfg["bounds"]), np.asarray(cfg["bounds"]), 2000, 0.02
    d, n = 24, 8192
    rng = np.random.default_rng(24)
    b = np.array([(-2.0, 2.0)] * d)
    X = rng.uniform(-2.0, 2.0, size=(n, d))
    y = -0.5 * np.sum((X / 0.7) ** 2, axis=1)
    g = ab.GP(kernel=ab.kernels.ExpSquaredKernel(metric=np.full(d, 16.0), ndim=d) * np.var(y), fit_mean=True,
              mean=np.median(y), white_noise=-8.0, fit_white_noise=True)
    g.compute(X)
    yield "d24", SurrogateLogProb(g, y, b), b, 500, 0.5


def kernel_ms(fn, name, reps):
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if name in e.key)
    return us / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "nested_rslice_probe.txt"))
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0].split(", ")
    lines = [{"gpu": smi[0], "power_limit": smi[1], "max_sm_clock": smi[2], "nchains": NCHAINS, "walks": WALKS,
              "slices": SLICES}]
    for name, lp, b, nlive, dlogz in surrogates():
        d = len(b)
        w = DeviceWalker(lp, b, seed=7)
        u = w.rng.random((8 * NCHAINS, d))
        th = w.transform(u)
        ll = w.like(th)
        lmin = float(np.median(ll))
        keep = np.nonzero(ll > lmin)[0][:NCHAINS]
        u0, th0, l0 = u[keep], th[keep], ll[keep]
        chol = BatchedNestedSampler(w, d)._proposal_chol(u0)
        row = {"surrogate": name, "N": int(lp.gp._x.shape[0]) if hasattr(lp.gp, "_x") else None, "d": d, "lmin": lmin}
        walk_ms = kernel_ms(lambda: w.walk(u0, th0, l0, lmin, 1.0, chol, WALKS), "nested_walk_kernel", args.reps)
        _, _, _, acc = w.walk(u0, th0, l0, lmin, 1.0, chol, WALKS)
        slice_ms = kernel_ms(lambda: w.rslice(u0, th0, l0, lmin, 1.0, chol, SLICES), "nested_rslice_kernel", args.reps)
        _, _, _, counts = w.rslice(u0, th0, l0, lmin, 1.0, chol, SLICES)
        ev = counts[:, 3]
        pad = (-len(ev)) % 32
        rounds = np.concatenate([ev, np.zeros(pad, dtype=ev.dtype)]).reshape(-1, 32).max(axis=1)
        walk_ev = NCHAINS * WALKS
        row["rwalk"] = {"kernel_ms": walk_ms, "evaluations": walk_ev, "evals_per_s": walk_ev / (walk_ms / 1e3),
                        "acceptance": acc, "lane_utilisation": 1.0}
        row["rslice"] = {"kernel_ms": slice_ms, "evaluations": int(ev.sum()), "evals_per_s": float(ev.sum()) / (slice_ms / 1e3),
                         "evals_per_chain": float(ev.mean()), "nexpand_per_slice": float(counts[:, 1].sum() / max(counts[:, 0].sum(), 1)),
                         "ncontract_per_slice": float(counts[:, 2].sum() / max(counts[:, 0].sum(), 1)),
                         "chains_finished": float(np.mean(counts[:, 0] == SLICES)),
                         "lane_utilisation": float(ev.sum() / (32.0 * rounds.sum()))}
        for sample in ("rwalk", "rslice"):
            s = BatchedNestedSampler(DeviceWalker(lp, b, seed=11), d, nlive=nlive, walks=WALKS, slices=SLICES,
                                     sample=sample, rstate=12)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = s.run_nested(dlogz=dlogz)
            torch.cuda.synchronize()
            row[sample]["e2e"] = {"nlive": nlive, "dlogz": dlogz, "wall_s": time.perf_counter() - t0, "ncall": int(r.ncall),
                                  "niter": int(r.niter), "logz": float(r.logz[-1]), "logzerr": float(r.logzerr[-1])}
        lines.append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
    print(json.dumps(lines[0]))


if __name__ == "__main__":
    main()
