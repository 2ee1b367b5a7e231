"""Uncertainty of reweighted averages and the choice of theta: bootstrap and cross-validation over observables.

Both need hundreds of minimisations of problems that share yTilde and differ only in the observed data YTilde,
in per-observable weights of chi^2, or in the reference weights w0.  They run as batches of up to 32 problems on
Problem.batch_minimize (the theta scan's lockstep L-BFGS; yTilde is streamed once per pass for the whole batch).

Resampling happens on the host with numpy.random.default_rng(seed): a seed reproduces every replicate.  Both helpers
use the method whose data is set on the problem (set_logw or set_forces) and its YTilde / w0.
"""
import numpy as np

from .problem import FORCES, LBFGS_OK

BATCH = 32
RESAMPLE = ("observables", "noise", "structures")
NOT_RUN = -2001   # code of a replicate that was not minimised: every structure it drew has w0_j = 0


def _method(problem):
    if problem.method is None:
        raise RuntimeError("bioen_b200.replicates: call set_logw or set_forces on the problem first")
    return problem.method


def _start_points(problem, R, x0):
    """x0 as given to the helpers: None (zeros), one start point (n,) for all replicates, or one per replicate (R, n)"""
    n = problem.m if problem.method == FORCES else problem.n
    x = np.zeros(n) if x0 is None else np.asarray(x0, dtype=np.float64)
    if x.shape not in ((n,), (R, n)):
        raise ValueError("x0 must have shape (%d,) or (%d, %d), got %s" % (n, R, n, x.shape))
    return x


def _run_batches(problem, R, theta_of, planes_of, x0, cfg, runnable=None):
    """Minimise R problems in chunks of BATCH.  theta_of(ids) / planes_of(ids) give the thetas and the dict of
    per-problem arrays of the replicates `ids`.  Replicates outside `runnable` are not minimised: code NOT_RUN and NaN
    results.  Returns x, fmin, codes, averages, chi2, kl with NaN statistics where the code is not a success."""
    M = problem.m
    x0 = _start_points(problem, R, x0)
    out = dict(x=np.full((R, x0.shape[-1]), np.nan), fmin=np.full(R, np.nan), codes=np.full(R, NOT_RUN),
               averages=np.empty((R, M)), chi2=np.empty(R), kl=np.empty(R))
    ids_all = np.arange(R) if runnable is None else np.flatnonzero(runnable)
    for c in range(0, ids_all.size, BATCH):
        ids = ids_all[c:c + BATCH]
        X, fmin, codes, info = problem.batch_minimize(theta_of(ids), x0=x0[ids] if x0.ndim == 2 else x0,
                                                      **planes_of(ids), **cfg)
        out["x"][ids], out["fmin"][ids], out["codes"][ids] = X, fmin, codes
        out["averages"][ids], out["chi2"][ids], out["kl"][ids] = info["averages"], info["chi2"], info["kl"]
    failed = ~np.isin(out["codes"], LBFGS_OK)
    out["averages"][failed] = np.nan
    out["chi2"][failed] = np.nan
    out["kl"][failed] = np.nan
    return out


def bootstrap(problem, n_replicates, resample, theta, seed=0, x0=None, **lbfgs_cfg):
    """R = n_replicates minimisations at one theta, each on resampled data:

    resample="observables"  multinomial counts over the M observables become the chi^2 weights (row_weights)
    resample="noise"        YTilde + eps with eps ~ N(0, 1) per observable (YTilde = YObs / sigma, so eps is a fresh
                            draw of the experimental error)
    resample="structures"   w0 * counts over the N structures, rescaled to the sum of w0 (forces method only)

    x0: one start point (n,) for every replicate or one per replicate (R, n); default zeros.

    Returns a dict: averages (R, M) = yTilde . w at each replicate's optimum, chi2, kl, fmin, codes (R,), x (R, n) and
    the resampling input of every replicate: counts (R, M) or (R, N) int32, or noise (R, M).  A replicate whose
    liblbfgs code is not 0, 1 or 2 keeps its code, fmin and x and gets NaN averages, chi2 and kl; it raises nothing.
    A structure replicate that drew only structures with w0_j = 0 has no reference weights; it is not minimised and
    gets code NOT_RUN and NaN results."""
    method = _method(problem)
    if resample not in RESAMPLE:
        raise ValueError("resample must be one of %s, got %r" % (RESAMPLE, resample))
    if resample == "structures" and method != FORCES:
        raise ValueError("resample='structures' needs the forces method: a structure drawn zero times has w0_j = 0, "
                         "which the log-weights parametrisation (G_j = log w0_j) cannot represent")
    R = int(n_replicates)
    if R != n_replicates or R < 1:
        raise ValueError("n_replicates must be a positive integer")
    theta = float(theta)
    if not np.isfinite(theta) or theta < 0:
        raise ValueError("theta must be finite and >= 0")
    M, N = problem.m, problem.n
    _start_points(problem, R, x0)
    rng = np.random.default_rng(seed)
    res = {}
    runnable = None
    if resample == "observables":
        counts = rng.multinomial(M, np.full(M, 1.0 / M), size=R).astype(np.int32)
        res["counts"] = counts
        planes = lambda ids: dict(row_weights=counts[ids].astype(np.float64))
    elif resample == "noise":
        noise = rng.standard_normal((R, M))
        res["noise"] = noise
        Y = np.asarray(problem.YTilde, dtype=np.float64).ravel()
        planes = lambda ids: dict(YTilde=Y + noise[ids])
    else:
        counts = np.empty((R, N), dtype=np.int32)
        for r in range(R):
            counts[r] = rng.multinomial(N, np.full(N, 1.0 / N))
        res["counts"] = counts
        w0 = np.asarray(problem.w0, dtype=np.float64).ravel()
        runnable = (counts @ (w0 > 0)) > 0

        def planes(ids):
            w = w0 * counts[ids]
            return dict(w0=w * (w0.sum() / w.sum(axis=1, keepdims=True)))
    res.update(_run_batches(problem, R, lambda ids: np.full(ids.size, theta), planes, x0, lbfgs_cfg, runnable))
    return res


def fold_assignment(M, folds, rng):
    """A random partition of the M observables into `folds` groups of sizes differing by at most one: fold[i]."""
    fold = np.empty(M, dtype=np.int64)
    fold[rng.permutation(M)] = np.arange(M) % folds
    return fold


def cross_validate(problem, thetas, folds=5, seed=0, x0=None, **lbfgs_cfg):
    """K-fold cross-validation over observables for every theta: each (theta, fold) pair is one minimisation with
    chi^2 weight 0 on the fold's observables and 1 elsewhere.  Returns a dict with held_out_chi2 (T, F) =
    1/2 sum over the fold of (avg_i - YTilde_i)^2 at the fold's optimum, the training chi2, kl, fmin and codes (T, F),
    averages (T, F, M), fold (M,) = the fold of each observable, and thetas.  Pairs whose liblbfgs code is not
    0, 1 or 2 get NaN statistics.  x0: one start point (n,) for every pair or one per pair (T * F, n), pair
    (t, f) at row t * folds + f; default zeros."""
    method = _method(problem)  # noqa: F841  (raises when no data is set)
    thetas = np.asarray(thetas, dtype=np.float64).ravel()
    if thetas.size < 1 or not np.all(np.isfinite(thetas)) or np.any(thetas < 0):
        raise ValueError("thetas must be a non-empty list of finite values >= 0")
    M = problem.m
    F = int(folds)
    if F != folds or not 2 <= F <= M:
        raise ValueError("folds must be an integer in 2..M (M = %d)" % M)
    rng = np.random.default_rng(seed)
    fold = fold_assignment(M, F, rng)
    T = thetas.size
    th = np.repeat(thetas, F)                              # problem p = (t, f) with p = t * F + f
    fo = np.tile(np.arange(F), T)
    weights = (fold[None, :] != fo[:, None]).astype(np.float64)
    out = _run_batches(problem, T * F, lambda ids: th[ids], lambda ids: dict(row_weights=weights[ids]), x0, lbfgs_cfg)
    Y = np.asarray(problem.YTilde, dtype=np.float64).ravel()
    held = 0.5 * np.sum((1.0 - weights) * (out["averages"] - Y) ** 2, axis=1)
    return dict(held_out_chi2=held.reshape(T, F), chi2=out["chi2"].reshape(T, F), kl=out["kl"].reshape(T, F),
                fmin=out["fmin"].reshape(T, F), codes=out["codes"].reshape(T, F),
                averages=out["averages"].reshape(T, F, M), fold=fold, thetas=thetas)
