"""CPU: the extended-precision two-loop reference (tests/hp_twoloop.py) that tests/test_gpu_lbfgs_update.py judges the
L-BFGS update engines by.  It must agree with the fp64 oracle's two-loop recursion on benign histories, with mpmath at
50 digits on tiny problems (ys < 0 and near-orthogonal pairs included), and its rule must be sharp: directions that
are wrong the way a subtly broken update would be wrong (ring order, gamma, beta's denominator, a dropped pair, the
ring end not advanced, a flipped sign, a batch problem reading its neighbour's ring) must miss it by 1e3 x the
largest constant a test may use."""
import numpy as np
import pytest

import hp_reference as H
import hp_twoloop as T
import lbfgs_regimes as R

pytestmark = pytest.mark.skipif(not H.available(), reason="np.longdouble is not the x86-64 80-bit format")

# numpy's fp64 dot products sum in blocks of 8 with pairwise accumulation; over the benign histories below the oracle's
# recursion stays within 4 u * scale
C_ORACLE = 16
C_MAX = 64              # the largest constant a test may use with this reference
MUTANTS = ["order", "gamma_oldest", "beta_slot", "bound_minus_1", "end_not_advanced", "sign"]


def _update(st, **kw):
    return T.update(st["x"], st["xp"], st["g"], st["gp"], st["S"], st["Y"], st["ys_ring"], st["end_old"],
                    st["bound"], **kw)


@pytest.mark.parametrize("n", [1, 5, 257, 4003])
def test_agrees_with_oracle_two_loop(n):
    from oracle import oracle as O
    for end_old, bound in R.REACHABLE:
        st = R.state("benign", n, end_old, bound)
        ref = _update(st)
        s, y = ref["s"], ref["y"]
        ys, yy = float(np.dot(y, s)), float(np.dot(y, y))
        ys_arr = st["ys_ring"].copy()
        ys_arr[end_old] = ys
        d = O.lbfgs_two_loop(st["g"], ref["S"], ref["Y"], ys_arr, (end_old + 1) % T.M, bound, ys, yy)
        r = T.ratio(d, ref["d"], ref["s_d"])
        assert r <= C_ORACLE, (end_old, bound, r)
        assert T.ratio(ys, ref["ys"], ref["s_ys"]) <= C_ORACLE and T.ratio(yy, ref["yy"], ref["s_yy"]) <= C_ORACLE


def _mp_update(st):
    """the same recursion in mpmath at 50 digits, on the fp64 pair s = fl(x - xp), y = fl(g - gp)"""
    import mpmath as mp
    mp.mp.dps = 50
    v = lambda a: [mp.mpf(float(t)) for t in np.ravel(a)]
    dot = lambda a, b: mp.fsum(p * q for p, q in zip(a, b))
    end_old, bound = st["end_old"], st["bound"]
    S = [v(r) for r in st["S"]]
    Y = [v(r) for r in st["Y"]]
    S[end_old] = v(st["x"] - st["xp"])
    Y[end_old] = v(st["g"] - st["gp"])
    ring = v(st["ys_ring"])
    ys, yy = dot(Y[end_old], S[end_old]), dot(Y[end_old], Y[end_old])
    ring[end_old] = ys
    g = v(st["g"])
    d = [-t for t in g]
    js = T.newest_first((end_old + 1) % T.M, bound)
    alpha, araw = {}, {}
    for j in js:
        araw[j] = dot(S[j], d)
        alpha[j] = araw[j] / ring[j]
        d = [p - alpha[j] * q for p, q in zip(d, Y[j])]
    d = [p * ys / yy for p in d]
    for j in js[::-1]:
        beta = dot(Y[j], d) / ring[j]
        d = [p + (alpha[j] - beta) * q for p, q in zip(d, S[j])]
    return dict(d=d, dg=[dot(g, d)], ys=[ys], yy=[yy], alpha=araw)


def _mp_ld(vals):
    import mpmath as mp
    out = []
    for t in vals:
        hi = float(t)
        out.append(H.LD(hi) + H.LD(float(t - mp.mpf(hi))))
    return np.array(out, dtype=H.LD)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("regime", ["benign", "ys_negative", "near_orth", "ys_decades", "range150", "g_last"])
def test_agrees_with_mpmath(regime, n):
    for end_old, bound in [(0, 1), (2, 3), (4, 6), (1, 6)]:
        st = R.state(regime, n, end_old, bound)
        ref = _update(st)
        mpv = _mp_update(st)
        for k in ("d", "dg", "ys", "yy"):
            err = np.abs(np.atleast_1d(ref[k]).astype(H.LD) - _mp_ld(mpv[k]))
            assert np.all(err <= 1e-17 * np.atleast_1d(ref["s_" + k]).astype(H.LD)), (k, end_old, bound)
        for j, a in mpv["alpha"].items():
            assert abs(ref["alpha"][j] - _mp_ld([a])[0]) <= 1e-17 * ref["s_alpha"][j], ("alpha", j)


def test_non_finite_where_a_pair_did_not_move():
    """a zero new pair: ys = yy = 0, gamma = 0/0, so d and g.d are NaN in every component; the newest raw s.d is 0"""
    st = R.state("zero_pair", 33, 2, 6)
    ref = _update(st)
    assert float(ref["ys"]) == 0.0 and float(ref["yy"]) == 0.0
    assert not np.any(np.isfinite(ref["d"])) and not np.isfinite(ref["dg"])
    assert ref["alpha"][2] == 0
    assert T.ratio(np.full(33, np.nan), ref["d"], ref["s_d"]) == 0.0
    assert T.ratio(np.ones(33), ref["d"], ref["s_d"]) == float("inf")


@pytest.mark.parametrize("n", [5, 257, 4003])
def test_gram_reference_agrees_with_the_vector_recursion(n):
    """the coefficient-space restatement computes the same direction (both in extended precision)"""
    for regime in ("benign", "ys_decades", "ys_negative", "near_orth"):
        for end_old, bound in R.REACHABLE:
            st = R.state(regime, n, end_old, bound)
            ref = _update(st)
            gr = T.gram(st["g"], ref["S"], ref["Y"], end_old, bound, st["ys_ring"])
            assert T.ratio(np.asarray(gr["d"], dtype=np.float64), ref["d"], ref["s_d"]) <= 1.0, (regime, end_old)
            assert T.ratio(float(gr["dg"]), ref["dg"], ref["s_dg"]) <= 1.0


def _miss(mut, ref):
    return max(T.ratio(np.asarray(mut["d"], dtype=np.float64), ref["d"], ref["s_d"]),
               T.ratio(float(mut["dg"]), ref["dg"], ref["s_dg"]))


@pytest.mark.parametrize("mutant", MUTANTS + ["batch_neighbour"])
def test_mutants_violate_the_rule(mutant):
    """each mutant, rounded to fp64, misses C_MAX u scale by 1e3 x on at least one regime (and the correct update,
    rounded to fp64, passes everywhere)"""
    need = 1e3 * C_MAX
    worst = {}
    for regime in R.REGIMES:
        if regime == "zero_pair":
            continue
        st = R.state(regime, 257, 3, 6)
        ref = _update(st)
        assert _miss(dict(d=ref["d"], dg=ref["dg"]), ref) <= 1.0, regime
        if mutant == "batch_neighbour":
            # problem q reads problem q - 1's ring slots (its own new pair is where the pair kernel wrote it)
            nb = R.state(regime, 257, 3, 6, seed=1)
            S, Y, ring = nb["S"].copy(), nb["Y"].copy(), nb["ys_ring"].copy()
            S[3], Y[3] = ref["s"], ref["y"]
            ring_ld = ring.astype(T.LD)
            ring_ld[3] = ref["ys"]
            mut = T.two_loop(st["g"], S, Y, ring_ld, np.zeros(T.M, dtype=T.LD), 4, 6, ref["ys"], ref["s_ys"],
                             ref["yy"], ref["s_yy"])
        else:
            mut = _update(st, mutant=mutant)
        worst[regime] = _miss(mut, ref)
    assert max(worst.values()) >= need, {k: "%.3g" % v for k, v in worst.items()}
