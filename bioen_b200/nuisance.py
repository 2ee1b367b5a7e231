"""Nuisance-parameter refits on the resident matrix (SURVEY.md section 8 f3).

Between two weight optimisations the reference refits the DEER modulation depths and the scattering scale factor
against the current weights and rebuilds the simulated-data matrix on the host, entry by entry in a Python double
loop (bioen/analyze/observables/observables.py: get_proc_sim 110-143, moddepth_fit 146-171, coeff_fit 174-188,
update_sim 191-216, update_sim_init 219-229; driven by bioen/analyze/procedure.py:62-83).  Both parameters act
AFFINELY on the rows of yTilde:

    DEER label (rows of one spin-label pair)   yTilde_ij = (1 - m + m s_ij) / err_i  =  (m) * b_ij + (1 - m) / err_i
    scattering                                 yTilde_ij = c s_ij / err_i            =  (c) * b_ij
    generic / CD                               yTilde_ij = s_ij / err_i              =      b_ij          (no parameter)

with the parameter-free base b_ij = s_ij / err_i.  So with yTilde resident in HBM

  * the chi^2 of ANY trial value of a parameter needs the base averages  (b . w)_i  only: ONE row pass on the device
    (Problem.average) serves the whole least-squares fit of all blocks, every trial after that is O(rows) on the host;
  * committing the refitted values is the in-place row-affine transform Problem.affine_rows (one read + one write
    pass on the device) instead of a rebuild on the host and a new upload;
  * a theta series whose problems carry DIFFERENT values (theta_series) needs no commit at all: problem k's matrix
    a_k * yTilde + b_k is two per-problem row planes of the batched engine (Problem.batch_minimize), and up to 32
    theta values share every pass over the unchanged resident matrix.

The fit itself is the reference's: scipy.optimize.leastsq on the scalar chi^2 of the block (observables.py:207,
212), same start values, same "initial-optimization" defaults (0.15 / 0.0002).
"""
import numpy as np
from scipy.optimize import leastsq

from . import _lib
from .problem import LBFGS_OK
from .replicates import BATCH, NOT_RUN, _start_points

DEER, SCATTERING, FIXED = "deer", "scattering", "fixed"
INITIAL = "initial-optimization"
INITIAL_VALUES = {DEER: 0.15, SCATTERING: 0.0002}          # observables.py:224, 228


class Block:
    """Rows [start, stop) of yTilde that share one nuisance parameter.

    kind      'deer' (modulation depth m), 'scattering' (scale factor c) or 'fixed'
    err       (rows,) experimental errors
    exp_fit   (rows,) experimental values the PARAMETER is fitted against (DEER: the background-corrected raw trace,
              exp_tmp[:, 1], observables.py:161; scattering: I(q), :179) -- not necessarily the values the weights are
              optimised against (DEER: the polynomial fit, exp_tmp[:, 2], :340)
    value     current parameter (float), or 'initial-optimization'
    """

    def __init__(self, kind, start, stop, err=None, exp_fit=None, value=None, name=None):
        if kind not in (DEER, SCATTERING, FIXED):
            raise ValueError("unknown block kind %r" % (kind,))
        self.kind, self.start, self.stop = kind, int(start), int(stop)
        n = self.stop - self.start
        self.err = np.ones(n) if err is None else _lib.vec(err)
        self.exp_fit = None if exp_fit is None else _lib.vec(exp_fit)
        if kind != FIXED and (self.exp_fit is None or self.exp_fit.size != n or self.err.size != n):
            raise ValueError("err and exp_fit must have one entry per row of the block")
        self.value = value
        self.name = name or "%s[%d:%d]" % (kind, self.start, self.stop)

    # row-affine map base -> yTilde for a parameter value:  yTilde = scale * base + offset
    def scale_offset(self, value):
        n = self.stop - self.start
        if self.kind == DEER:
            return np.full(n, float(value)), (1.0 - float(value)) / self.err
        if self.kind == SCATTERING:
            return np.full(n, float(value)), np.zeros(n)
        return np.ones(n), np.zeros(n)

    def chi2(self, value, base_avg, sum_w):
        """0.5 * || yTilde(value) . w - exp_fit / err ||^2 over the rows of the block -- what moddepth_fit / coeff_fit
        return (observables.py:171, 188), from the base averages (b . w)_i."""
        s, o = self.scale_offset(np.ravel(value)[0])
        r = s * base_avg + o * sum_w - self.exp_fit / self.err
        return 0.5 * float(r @ r)


def base_matrix(raw_rows, err):
    """b = s / err[:, None] for raw simulated data s (rows x models): the parameter-free matrix to keep resident."""
    return np.asarray(raw_rows, dtype=np.float64) / _lib.vec(err)[:, None]


def proc_sim(base, blocks):
    """yTilde for the blocks' current values from the base matrix on the HOST (NumPy twin of get_proc_sim,
    observables.py:110-143; used to build the first upload and by the tests)."""
    out = np.array(base, dtype=np.float64, copy=True)
    for b in blocks:
        if b.kind == FIXED:
            continue
        s, o = b.scale_offset(_start_value(b))
        out[b.start:b.stop] = s[:, None] * out[b.start:b.stop] + o[:, None]
    return out


def _start_value(block):
    if isinstance(block.value, str):
        if block.value != INITIAL:
            raise ValueError("block value must be a number or %r" % INITIAL)
        return INITIAL_VALUES[block.kind]
    return float(block.value)


def _transform(blocks, values, m):
    """Row-wise (scale, offset) of the map base -> yTilde when block b has the value values[b.name] (default: its
    current value); rows outside the blocks and FIXED blocks keep the identity."""
    scale, offset = np.ones(m), np.zeros(m)
    for b in blocks:
        if b.kind != FIXED:
            scale[b.start:b.stop], offset[b.start:b.stop] = b.scale_offset(values.get(b.name, b.value))
    return scale, offset


def _fit(blocks, base_avg, sum_w, starts):
    """Least-squares refit of every parameter block against the base averages (observables.py:203-213), block b from
    starts[b.name].  Returns {name: value}."""
    out = {}
    for b in blocks:
        if b.kind == FIXED:
            continue
        sl = base_avg[b.start:b.stop]
        opt, _ = leastsq(lambda v: b.chi2(v, sl, sum_w), starts[b.name])
        out[b.name] = float(np.ravel(opt)[0])
    return out


class NuisanceRefit:
    """Refit loop state for one resident problem.

    `problem` (bioen_b200.Problem or dist.ShardedProblem) must hold yTilde built with the blocks' CURRENT values
    (e.g. uploaded from proc_sim(base, blocks)); rows outside all blocks are left alone.  `update(w)` mirrors
    Observables.update_sim (observables.py:191-216): refit every block against the weights w, then commit.
    """

    def __init__(self, problem, blocks):
        self.problem = problem
        self.blocks = list(blocks)
        self.m = problem.m
        for b in self.blocks:
            if not (0 <= b.start <= b.stop <= self.m):
                raise ValueError("block %s outside the matrix" % b.name)
            if b.kind != FIXED:
                b.value = _start_value(b)
        # resident matrix = _scale * base + _offset (row-wise)
        self._scale, self._offset = _transform(self.blocks, {}, self.m)

    def relative(self, values):
        """(a, c, scale, offset): the matrix of the blocks at `values` ({name: value}; blocks not named keep their
        current value) is a * resident + c = scale * base + offset, row-wise."""
        s, o = _transform(self.blocks, values, self.m)
        a = s / self._scale
        return a, o - self._offset * a, s, o

    def base_from_averages(self, avg, sum_w):
        """(b . w)_i from the averages avg = yTilde . w of the resident matrix and sum(w)."""
        return (avg - self._offset * sum_w) / self._scale

    def base_averages(self, w):
        """(b . w)_i and sum(w): one row pass over the resident matrix, mapped back through the current transform."""
        w = _lib.vec(w)
        sw = float(w.sum())
        return self.base_from_averages(self.problem.average(w), sw), sw

    def chi2(self, block, value, w=None, base_avg=None, sum_w=None):
        """chi^2 of one block for a trial value (= Observables.moddepth_fit / coeff_fit)."""
        if base_avg is None:
            base_avg, sum_w = self.base_averages(w)
        return block.chi2(value, base_avg[block.start:block.stop], sum_w)

    def fit(self, w):
        """Least-squares refit of every block against w (observables.py:203-213).  Returns {name: value}; nothing
        is committed."""
        base_avg, sw = self.base_averages(w)
        return _fit(self.blocks, base_avg, sw, {b.name: b.value for b in self.blocks})

    def commit(self, values):
        """Make the resident matrix the one of the given values: one in-place row-affine pass on the device."""
        new = {}
        for b in self.blocks:
            if b.kind == FIXED or b.name not in values:
                continue
            new[b.name] = float(values[b.name])
            if new[b.name] == 0.0:
                raise ValueError("a zero %s parameter makes the block's rows independent of the simulated data; the "
                                 "resident matrix cannot be transformed back from that" % b.kind)
        a, c, new_s, new_o = self.relative(new)      # new = a * old + c
        for b in self.blocks:
            if b.name in new:
                b.value = new[b.name]
        if np.any(a != 1.0) or np.any(c != 0.0):
            self.problem.affine_rows(a, c)
        self._scale, self._offset = new_s, new_o

    def update(self, w):
        """Observables.update_sim: refit, then rebuild (here: transform in place).  Returns {name: value}."""
        values = self.fit(w)
        self.commit(values)
        return values


def theta_series(problem, blocks, thetas, iterations, values=None, x0=None, **lbfgs_cfg):
    """The reference's theta series with nuisance-parameter refits (bioen/analyze/procedure.py:40-83) for every theta
    at once, in batches of up to 32 problems on ONE resident matrix that is never modified.

    `problem` holds yTilde built with the blocks' CURRENT values, as for NuisanceRefit, and its set_logw / set_forces
    data (YTilde, G or w0; the method of the minimisations).  Problem t runs at thetas[t] with its own block values,
    starting from values[name] (a scalar or one value per theta; default: the block's current value).  Each of the
    `iterations` rounds
      1. minimises every problem from x0 (as batch_minimize: (n,) or one row per theta; default zeros -- the
         reference restarts every find_optimum from the same log-weights) on the matrix of its own values, given to
         the batched engine as the row-affine planes relative to the resident matrix;
      2. recovers the base averages (b . w)_i from the resident averages batch_minimize returns;
      3. refits every block by least squares from the problem's current value (Observables.update_sim).
    The reference refits against its weights with exact zeros replaced by 1e-150; the device weights sum to 1, and the
    replacement changes neither that sum nor any average above ~1e-134 * sum_j |y_ij| in double precision, so the
    refit uses the averages as returned and sum(w) = 1.  A problem whose liblbfgs code is not 0, 1 or 2 keeps that
    round's x, fmin and code and stops there: NaN values afterwards, code NOT_RUN and NaN x / fmin in later rounds.

    Returns dict(x (iterations, T, n), fmin (iterations, T), codes (iterations, T), values {name: (iterations + 1, T)}
    with the start values in row 0 and the refit of round i in row i + 1, thetas (T,))."""
    thetas = _lib.vec(thetas)
    T = thetas.size
    if T < 1 or not np.all(np.isfinite(thetas)) or np.any(thetas < 0):
        raise ValueError("thetas must be a non-empty list of finite values >= 0")
    iterations = int(iterations)
    if iterations < 1:
        raise ValueError("iterations must be >= 1")
    if problem.method is None:
        raise RuntimeError("theta_series: call set_logw or set_forces on the problem first")
    x0 = _start_points(problem, T, x0)
    resident = NuisanceRefit(problem, blocks)          # bookkeeping of the resident matrix; nothing is committed
    fitted = [b for b in resident.blocks if b.kind != FIXED]
    if np.any(resident._scale == 0.0):
        raise ValueError("a block's current value is zero: the base averages cannot be recovered from the resident "
                         "matrix")
    given = {} if values is None else dict(values)
    unknown = set(given) - {b.name for b in fitted}
    if unknown:
        raise ValueError("values for unknown blocks: %s" % sorted(unknown))
    hist = {}
    for b in fitted:
        v = np.asarray(given.get(b.name, b.value), dtype=np.float64)
        if v.shape not in ((), (T,)) or not np.all(np.isfinite(v)):
            raise ValueError("values[%r] must be a finite scalar or have one entry per theta" % b.name)
        hist[b.name] = np.full((iterations + 1, T), np.nan)
        hist[b.name][0] = v
    out = dict(x=np.full((iterations, T, x0.shape[-1]), np.nan), fmin=np.full((iterations, T), np.nan),
               codes=np.full((iterations, T), NOT_RUN), values=hist, thetas=thetas)
    for lo in range(0, T, BATCH):
        alive = np.arange(lo, min(T, lo + BATCH))
        for it in range(iterations):
            if alive.size == 0:
                break
            planes = [resident.relative({name: h[it, t] for name, h in hist.items()})[:2] for t in alive]
            X, fmin, codes, info = problem.batch_minimize(thetas[alive], x0=x0[alive] if x0.ndim == 2 else x0,
                                                          row_scale=np.stack([p[0] for p in planes]),
                                                          row_offset=np.stack([p[1] for p in planes]), **lbfgs_cfg)
            out["x"][it, alive], out["fmin"][it, alive], out["codes"][it, alive] = X, fmin, codes
            ok = np.isin(codes, LBFGS_OK)
            for q in np.flatnonzero(ok):
                t = alive[q]
                base = resident.base_from_averages(info["averages"][q], 1.0)
                for name, v in _fit(fitted, base, 1.0, {name: h[it, t] for name, h in hist.items()}).items():
                    hist[name][it + 1, t] = v
            alive = alive[ok]
    return out
