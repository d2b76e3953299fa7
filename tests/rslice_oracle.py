"""CPU reference for the device's random-direction slice sampling (ab_nested_rslice).

TEST INFRASTRUCTURE ONLY.  Builds on ``oracle.nested.walk_normals`` (the walk's normals) and
``oracle.philox`` and leaves the ``oracle`` package unchanged.  The algorithm and draw layout are
restated here independently of the CUDA source:

Random-direction slice sampling of ``ab_nested_rslice`` (dynesty's ``sample="rslice"``
as recalled, Neal 2003 stepping out and shrinking; parity with dynesty unpinned like rwalk's).
Slice s of chain c, with F(x) = L(T(u + x v)) inside (0, 1)^d and -inf (no call) outside:

    z = the walk's normals at step s;  v = (C z) * (scale / |z|)
    r0 = u53(w0, w1) of Philox block j0 = ceil(d / 2), counter (chain_offset + c, s, j0, launch counter)
    x_l = -r0, x_r = 1 - r0
    while F(x_l) > L_min: x_l -= 1;  then while F(x_r) > L_min: x_r += 1        (nexpand += 1 each)
    for i = 0, 1, ...: x = x_l + u_i (x_r - x_l), u_i = u53(w0, w1) of block j0 + 1 + i
        F(x) > L_min: u <- u + x v, the slice is complete
        else: x_l = x if x < 0, x_r = x if x > 0                                (ncontract += 1)
    a slice needing more than ``max_expand`` expansions or ``max_contract`` contractions ends the
    chain at the end point of its last completed slice.

Window and point arithmetic are single IEEE operations here (no fused multiply-add), as on the
device.
"""
import numpy as np

from oracle.nested import walk_normals
from oracle.philox import philox4x32, u53


def replay_rslice(u0, theta0, logl0, lmin, scale, chol, slices, seed, counter, transform, loglike, chain_offset=0,
                  max_expand=1024, max_contract=256):
    """End points (u, theta, logl), counts (nchains, 4: slices completed, nexpand, ncontract,
    likelihood calls) and the smallest margin of any comparison that decided a branch (L vs L_min
    and the cube edges) of ``slices`` slices from (u0, theta0, logl0).  Chains advance in lock step so
    that ``loglike`` sees one batch per round."""
    u, theta, logl = np.array(u0, dtype=np.float64), np.array(theta0, dtype=np.float64), np.array(logl0, dtype=np.float64)
    k, d = u.shape
    C = np.tril(np.asarray(chol, dtype=np.float64))
    j0 = (d + 1) // 2
    counts = np.zeros((k, 4), dtype=np.int64)
    margins = [np.inf]
    st = [{"done": int(slices) == 0} for _ in range(k)]

    def uniform(c, j):
        r = philox4x32(np.uint64(chain_offset + c), int(counts[c, 0]), j, counter, seed & 0xFFFFFFFF, seed >> 32)
        return float(u53(r[0], r[1]))

    def begin(c):
        S = st[c]
        z = walk_normals(seed, counter, [c], int(counts[c, 0]), d, chain_offset)[0]
        S["v"] = (C @ z) * (scale / np.sqrt(np.sum(z * z)))
        r0 = uniform(c, j0)
        S.update(xl=-r0, xr=1.0 - r0, x=-r0, phase=0, i=0, ne=0, nc=0)

    def shrink_draw(c):
        S = st[c]
        return S["xl"] + uniform(c, j0 + 1 + S["i"]) * (S["xr"] - S["xl"])

    def point(c):
        return u[c] + st[c]["x"] * st[c]["v"]

    def advance(c, ok, th=None, y=None):
        S = st[c]
        if S["phase"] < 2:                       # stepping out, left then right
            if ok:
                if S["ne"] == max_expand:
                    S["done"] = True
                    return
                S["ne"] += 1
                counts[c, 1] += 1
                if S["phase"] == 0:
                    S["xl"] -= 1.0
                    S["x"] = S["xl"]
                else:
                    S["xr"] += 1.0
                    S["x"] = S["xr"]
            elif S["phase"] == 0:
                S["phase"], S["x"] = 1, S["xr"]
            else:
                S["phase"] = 2
                S["x"] = shrink_draw(c)
        elif ok:
            u[c], theta[c], logl[c] = point(c), th, y
            counts[c, 0] += 1
            if counts[c, 0] == int(slices):
                S["done"] = True
            else:
                begin(c)
        else:
            S["nc"] += 1
            counts[c, 2] += 1
            if S["x"] < 0.0:
                S["xl"] = S["x"]
            elif S["x"] > 0.0:
                S["xr"] = S["x"]
            if S["nc"] == max_contract:
                S["done"] = True
                return
            S["i"] += 1
            S["x"] = shrink_draw(c)

    def next_point(c):
        # next proposal inside the cube (None when the chain has ended); outside points cost no call
        while not st[c]["done"]:
            p = point(c)
            edge = float(np.min(np.minimum(p, 1.0 - p)))
            margins.append(abs(edge))
            if edge > 0.0:
                return p
            advance(c, False)
        return None

    pending = {}
    for c in range(k):
        if not st[c]["done"]:
            begin(c)
            p = next_point(c)
            if p is not None:
                pending[c] = p
    while pending:
        idx = sorted(pending)
        th = np.atleast_2d(transform(np.array([pending[c] for c in idx])))
        y = np.asarray(loglike(th), dtype=np.float64).reshape(-1)
        margins.append(float(np.min(np.abs(y - lmin))))
        nxt = {}
        for j, c in enumerate(idx):
            counts[c, 3] += 1
            advance(c, bool(y[j] > lmin), th[j], y[j])
            p = next_point(c)
            if p is not None:
                nxt[c] = p
        pending = nxt
    return u, theta, logl, counts, min(margins)
