"""Inputs at the numerical edges of both methods, shared by the extended-precision reference's self-tests
(tests/test_hp_reference.py) and the GPU tests (tests/test_gpu_numerical_edges.py).

A case is (matrix variant, x, G or w0, theta).  The matrix variants are the synthetic problem's yTilde / YTilde and
edits of it:
  base      the synthetic problem (oracle.synthetic_problem)
  rowoff    every row shifted by ~1e3 x its spread (YTilde shifted alike): avg_i and y_ij - avg_i cancel
  top@P     column P (first / mid / last) made the unique argmax of x = v . y for the forces direction v
  tie       the argmax column copied to several places that straddle CTA and rank borders: exact ties at the max
"""
import zlib

import numpy as np

from oracle.oracle import synthetic_problem

PLACES = ("first", "mid", "last")

LOGW_REGIMES = (["benign"] + ["conc700_" + p for p in PLACES] + ["conc3000_" + p for p in PLACES]
                + ["theta1e-8", "theta1e8", "theta0", "gauge1e3", "gauge-1e4", "gauge1e5", "rowoff", "ties"])
FORCES_REGIMES = (["benign"] + ["x300_" + p for p in PLACES] + ["x3000_" + p for p in PLACES]
                  + ["w0zero30", "w0run", "w0zero_argmax", "w0subnormal", "theta1e-8", "theta1e8", "theta0",
                     "rowoff", "ties"])


def place(P, N):
    """first: column 0 (first tile, CTA 0, rank 0); last: N - 1 (ragged last tile); mid: a column that CTA 0 and
    rank 0 do not own (rank 1 of 2 or 3 ranks)"""
    return {"first": 0, "mid": N // 2 + 1 if N > 2 else N - 1, "last": N - 1}[P]


def tie_columns(N):
    return sorted({0, max(N // 3 - 1, 0), N // 3, N // 2, (2 * N) // 3, N - 1})


def _direction(M, N):
    return np.random.default_rng(7 * M + N).standard_normal(M)


_MATS = {}


def matrix(variant, M, N):
    """(yTilde (M, N), YTilde (M,)) of a variant (cached; callers must not modify them)"""
    key = (variant, M, N)
    if key in _MATS:
        return _MATS[key]
    P = synthetic_problem(M, N, seed=1000 + M + N)
    y, Y = P["yTilde"].copy(), P["YTilde"].ravel().copy()
    if variant == "rowoff":
        off = 1e3 * y.std(axis=1) * (1.0 + np.random.default_rng(M).random(M))
        y += off[:, None]
        Y += off
    elif variant.startswith("top@") or variant == "tie":
        v = _direction(M, N)
        js = int(np.argmax(v @ y))
        col = y[:, js] + 0.25 * np.sign(v)
        cols = tie_columns(N) if variant == "tie" else [place(variant[4:], N)]
        for j in cols:
            y[:, j] = col
    elif variant != "base":
        raise ValueError(variant)
    _MATS[key] = (np.ascontiguousarray(y), Y)
    return _MATS[key]


def _w0(rng, N):
    w0 = rng.random(N) + 0.1
    return w0 / w0.sum()


def _forces_span(y, M, N, span):
    """the forces s v whose x = f . y spans `span`"""
    v = _direction(M, N)
    xv = v @ y
    return v * (span / (xv.max() - xv.min())) if N > 1 else v * (span / max(abs(xv[0]), 1e-300))


def case(method, regime, M, N):
    """(variant, x, G or w0, theta) of a regime; method 0 log-weights, 1 forces"""
    rng = np.random.default_rng([method, zlib.crc32(regime.encode()), M, N])
    theta = 3.7
    if regime.startswith("theta"):
        theta = float(regime[5:])
    variant = "base"
    if method == 0:
        G = 0.2 * rng.standard_normal(N)
        g = G + 0.1 * rng.standard_normal(N)
        if regime.startswith("conc"):
            span, p = regime[4:].split("_")
            j = place(p, N)
            if span == "700":            # weights from 1e-304 to 1
                g = -700.0 * rng.random(N)
            else:                        # one structure and its neighbours carry all the weight: every other CTA slice /
                g = -750.0 - 2250.0 * rng.random(N)   # chunk / shard has exp(m_c - m) < 1e-325, i.e. 0
                near = slice(max(j - 16, 0), min(j + 17, N))
                g[near] = -700.0 * rng.random(g[near].size)
            g[j] = 0.0
        elif regime.startswith("gauge"):
            c = float(regime[5:])
            g, G = g + c, G + c
        elif regime == "rowoff":
            variant = "rowoff"
        elif regime == "ties":
            variant = "tie"
            g = -700.0 * rng.random(N)
            g[tie_columns(N)] = 0.0
        return variant, g, G, theta
    w0 = _w0(rng, N)
    span = 30.0
    if regime.startswith("x"):
        s, p = regime[1:].split("_")
        variant, span = "top@" + p, float(s)
    elif regime == "benign" or regime.startswith("theta"):
        span = None
    elif regime == "w0zero30":
        w0[rng.random(N) < 0.3] = 0.0
    elif regime == "w0run":
        # a run covering whole CTA slices / team slabs and rank 1's shard of 3
        lo, hi = N // 3, (2 * N) // 3
        hi = min(N - 1, max(hi, lo + 2048))
        w0[lo:hi] = 0.0
    elif regime in ("w0zero_argmax", "w0subnormal"):
        variant, span = "top@mid", 300.0
    elif regime == "rowoff":
        variant, span = "rowoff", None
    elif regime == "ties":
        variant, span = "tie", 300.0
    y, _ = matrix(variant, M, N)
    f = 1e-3 * rng.standard_normal(M) if span is None else _forces_span(y, M, N, span)
    j = place("mid", N)
    if regime == "w0zero_argmax":
        w0[j] = 0.0
    elif regime == "w0subnormal" and N > 1:
        # w0_j = 1e-310 on the argmax, and x_j - x_next such that w0_next e^{x_next - x_j} = 1e-304: w_j ~ 1e-6
        # although w0_j is subnormal, with a normal sum sum_k w0_k e^{x_k - x_j} (1 / sum stays finite; at w_j ~ 1 the
        # sum would be subnormal and its reciprocal overflow -- in the reference as in every kernel)
        x = f @ y
        k = int(np.argsort(x)[-2])
        w0[j] = 1e-310
        f = f * ((np.log(w0[k]) - np.log(1e-304)) / (x[j] - x[k]))
    if not w0.any():
        w0[0] = 1.0
    return variant, f, w0, theta
