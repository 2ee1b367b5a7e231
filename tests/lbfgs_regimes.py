"""L-BFGS histories for the direction-update tests (tests/hp_twoloop.py is their reference).

state(regime, n, end_old, bound) is the input of one update: x, xp, g, gp (n), a ring S, Y (m x n) whose `bound - 1`
older pairs sit in the slots before end_old, and ys_ring (m) holding those pairs' y.s rounded to fp64 (what the
device's ring would hold).  Slots that no pair occupies hold finite junk, so an implementation that reads them shows.

Regimes:
  benign          y = A s with A SPD diagonal, cond 10
  ys_decades      the pairs' curvature y.s spans 1e-12 .. 1e12
  near_orth       one pair with y nearly orthogonal to s (ys / (|y| |s|) ~ 1e-10): ys formed by cancellation
  ys_negative     the new pair has ys < 0 (Armijo backtracking allows it; liblbfgs does not guard)
  range150        components spanning 1e-150 .. 1e150 in x, s, y and g (products stay below 1e306)
  zero_block      a block of structures that do not move (s = 0 there in every pair)
  zero_pair       the new pair is zero (x = xp, g = gp): ys = yy = 0 and the direction is NaN
  g_last          g nonzero only in the last (ragged) element
  subnormal       a block of subnormal components in x, xp, s, y and g
"""
import numpy as np

M = 6
REGIMES = ["benign", "ys_decades", "near_orth", "ys_negative", "range150", "zero_block", "zero_pair", "g_last",
           "subnormal"]
# the (end_old, bound) a minimisation reaches: before the ring wraps end_old = bound - 1, afterwards bound = 6
REACHABLE = [(b - 1, b) for b in range(1, M)] + [(e, M) for e in range(M)]
ALL_STATES = [(e, b) for b in range(1, M + 1) for e in range(M)]


def _exact_dot(a, b):
    return float(np.sum(a.astype(np.longdouble) * b.astype(np.longdouble)))


def state(regime, n, end_old, bound, seed=0):
    rng = np.random.default_rng([n, end_old, bound, REGIMES.index(regime), seed])
    sig = np.ones(n)
    gsig = np.ones(n)
    if regime == "range150":
        sig = 10.0 ** rng.uniform(-150.0, 150.0, n)
        gsig = sig
    lo, hi = n // 4, max(n // 2, n // 4 + 1) if n > 1 else 0
    if regime == "subnormal":
        sig[lo:hi] = 1e-310
        gsig[lo:hi] = 1e-310
    a = 1.0 + 9.0 * rng.random(n)                       # eigenvalues of A: cond <= 10
    ages = list(range(bound))                           # age 0: the new pair, slot end_old
    scale = {age: 1.0 for age in ages}
    if regime == "ys_decades":
        for age, e in zip(ages, [6.0, -6.0, 3.0, -3.0, 1.5, -1.5]):
            scale[age] = 10.0 ** e

    def pair(age):
        s = rng.standard_normal(n) * sig * scale[age]
        if regime == "zero_block":
            s[lo:hi] = 0.0
        y = a * s
        if regime == "near_orth" and age == min(1, bound - 1) and n > 1:
            # remove y's component along s, then put back 1e-10 |y| |s| of it
            z = rng.standard_normal(n) * sig * scale[age]
            y = z - (np.dot(z, s) / np.dot(s, s)) * s
            y = y + 1e-10 * (np.linalg.norm(y) / np.linalg.norm(s)) * s
        if regime == "ys_negative" and age == 0:
            y = -y
        if regime == "zero_block":
            y[lo:hi] = rng.standard_normal(hi - lo)       # a structure that does not move may still see g change
        return s, y

    S = rng.standard_normal((M, n)) * 1e3               # junk in slots no pair occupies
    Y = rng.standard_normal((M, n)) * 1e3
    ys_ring = np.full(M, 7.0)
    for age in ages[1:]:
        slot = (end_old - age) % M
        S[slot], Y[slot] = pair(age)
        ys_ring[slot] = _exact_dot(S[slot], Y[slot])
    s_new, y_new = pair(0)
    xp = rng.standard_normal(n) * sig
    g = rng.standard_normal(n) * gsig
    if regime == "g_last":
        g[:-1] = 0.0
    if regime == "zero_pair":
        x, gp = xp.copy(), g.copy()
    else:
        x = xp + s_new
        gp = g - y_new
    if regime == "zero_block":
        x[lo:hi] = xp[lo:hi]
    return dict(x=x, xp=xp, g=g, gp=gp, S=S, Y=Y, ys_ring=ys_ring, end_old=end_old, bound=bound)
