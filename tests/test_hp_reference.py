"""CPU: the extended-precision reference (tests/hp_reference.py) that tests/test_gpu_numerical_edges.py judges the
kernels by.  It must agree with the fp64 oracle wherever the oracle is defined, with mpmath at 50 digits, and it must
be sharp: fp64 answers that are wrong the way a subtly broken kernel would be wrong (a structure dropped, one CTA's
slice scaled by exp(1e-6), the w0 guard skipped, the maximum taken over the wrong set) must miss the acceptance rule
by orders of magnitude at the shapes the GPU tests use."""
import numpy as np
import pytest

import edge_regimes as R
import hp_reference as H
from conftest import FORCES_FIXTURES, LOGW_FIXTURES, load_golden

pytestmark = pytest.mark.skipif(not H.available(), reason="np.longdouble is not the x86-64 80-bit format")

# The fp64 oracle sums sequentially (errors ~ sqrt(N) u, up to N u); over the fixtures and the synthetic regimes below
# it stays within 80 u * scale (largest seen: 72, forces at theta = 1e8, 5 x 80001).  The kernels' blocked sums stay
# within 2 u * scale (tests/test_gpu_numerical_edges.py, C = 16 there).
C = 256
C_MAX = 1024            # the largest constant a test may use with this reference
SHAPES = [(28, 50001), (300, 4003), (1000, 777), (5, 80001), (3, 5)]


def _oracle_eval(oracle, method, x, a, y, Y, theta):
    with np.errstate(all="ignore"):
        if method == 0:
            f, g = oracle.logw_fg(x, a, y, Y.reshape(1, -1), theta)
            w, _ = oracle.logw_weights(x)
        else:
            f, g = oracle.forces_fg(x, a, y, Y.reshape(1, -1), theta)
            w = oracle.forces_weights(x, a, y)
    return np.array([f]), g, w


def _ref(method, x, a, y, Y, theta, **kw):
    return (H.logw if method == 0 else H.forces)(x, a, y, Y, theta, **kw)


@pytest.mark.parametrize("name", LOGW_FIXTURES + FORCES_FIXTURES)
def test_agrees_with_oracle_on_golden_fixtures(oracle, name):
    d = load_golden(name)
    method = 0 if d["kind"] == "logw" else 1
    a = d["G"] if method == 0 else d["w0"]
    Y = np.asarray(d["YTilde"]).ravel()
    for x in ((d["GInit"] if method == 0 else d["forces_init"]), d["probe"]):
        ref = _ref(method, x, a, d["yTilde"], Y, d["theta"])
        f, g, w = _oracle_eval(oracle, method, x, a, d["yTilde"], Y, d["theta"])
        r = H.ratios(ref, f=f, grad=g, w=w)
        assert max(r.values()) <= C, r


@pytest.mark.parametrize("M,N", SHAPES)
@pytest.mark.parametrize("method", [0, 1])
def test_agrees_with_oracle_where_the_oracle_is_defined(oracle, method, M, N):
    """every regime the fp64 oracle can evaluate: all but the gauge offsets (its softmax overflows at g ~ 1e3)"""
    for regime in (R.LOGW_REGIMES if method == 0 else R.FORCES_REGIMES):
        if regime.startswith("gauge"):
            continue
        variant, x, a, theta = R.case(method, regime, M, N)
        y, Y = R.matrix(variant, M, N)
        ref = _ref(method, x, a, y, Y, theta)
        f, g, w = _oracle_eval(oracle, method, x, a, y, Y, theta)
        r = H.ratios(ref, f=f, grad=g, w=w)
        assert max(r.values()) <= C, (regime, r)


def _mp_eval(method, x, a, y, Y, theta, c=None):
    """the same semantics in mpmath at 50 digits (tiny problems)"""
    import mpmath as mp
    mp.mp.dps = 50
    M, N = y.shape
    yv = [[mp.mpf(float(y[i, j])) for j in range(N)] for i in range(M)]
    Yv = [mp.mpf(float(v)) for v in np.ravel(Y)]
    cv = [mp.mpf(1)] * M if c is None else [mp.mpf(float(v)) for v in c]
    th = mp.mpf(float(theta))
    if method == 0:
        g = [mp.mpf(float(v)) for v in np.ravel(x)]
        G = [mp.mpf(float(v)) for v in np.ravel(a)]
        e = [mp.exp(v) for v in g]
        s = mp.fsum(e)
        w = [v / s for v in e]
        s0 = mp.fsum(mp.exp(v) for v in G)
        prior = th * (mp.fsum((g[j] - G[j]) * w[j] for j in range(N)) - mp.log(s) + mp.log(s0))
    else:
        f = [mp.mpf(float(v)) for v in np.ravel(x)]
        w0 = [mp.mpf(float(v)) for v in np.ravel(a)]
        xs = [mp.fsum(f[i] * yv[i][j] for i in range(M)) for j in range(N)]
        u = [w0[j] * mp.exp(xs[j]) for j in range(N)]
        s = mp.fsum(u)
        w = [v / s for v in u]
        ok = [float(w[j]) >= H.TINY and float(a[j]) >= H.TINY for j in range(N)]
        lr = [mp.log(w[j]) - mp.log(w0[j]) if ok[j] else mp.mpf(0) for j in range(N)]
        prior = th * mp.fsum(w[j] * lr[j] for j in range(N))
    avg = [mp.fsum(yv[i][j] * w[j] for j in range(N)) for i in range(M)]
    r = [avg[i] - Yv[i] for i in range(M)]
    chi2 = mp.fsum(cv[i] * r[i] ** 2 for i in range(M)) / 2
    if method == 0:
        gbar = mp.fsum(g[j] * w[j] for j in range(N))
        Gbar = mp.fsum(G[j] * w[j] for j in range(N))
        grad = [w[j] * th * (g[j] - gbar - G[j] + Gbar)
                + w[j] * mp.fsum(cv[i] * r[i] * (yv[i][j] - avg[i]) for i in range(M)) for j in range(N)]
    else:
        t = [mp.fsum(yv[i][j] * cv[i] * r[i] for i in range(M)) for j in range(N)]
        E = [(th * (1 + lr[j]) + t[j]) * w[j] for j in range(N)]
        grad = [mp.fsum((yv[i][j] - avg[i]) * E[j] for j in range(N)) for i in range(M)]
    return dict(f=[prior + chi2], grad=grad, w=w, avg=avg)


def _tiny_inputs(method, kind, M, N, rng):
    y = rng.standard_normal((M, N)) * 2.0 + 1.0
    Y = rng.standard_normal(M)
    if method == 0:
        G = 0.3 * rng.standard_normal(N)
        g = G + 0.1 * rng.standard_normal(N)
        if kind == "concentrated":
            g = -700.0 * rng.random(N)
            g[N // 2] = 0.0
        return g, G, y, Y
    w0 = rng.random(N) + 0.1
    w0 /= w0.sum()
    f = 0.3 * rng.standard_normal(M)
    if kind == "concentrated":
        f *= 300.0 / np.ptp(f @ y)
    elif kind == "zero_w0":
        w0[::3] = 0.0
    elif kind == "subnormal_w0":
        x = f @ y
        j, k = np.argsort(x)[-1], np.argsort(x)[-2]
        w0[j] = 1e-310
        f *= (np.log(w0[k]) - np.log(1e-304)) / (x[j] - x[k])
    return f, w0, y, Y


@pytest.mark.parametrize("M,N", [(3, 7), (5, 33)])
@pytest.mark.parametrize("method,kind", [(0, "benign"), (0, "concentrated"), (1, "benign"), (1, "concentrated"),
                                         (1, "zero_w0"), (1, "subnormal_w0")])
def test_agrees_with_mpmath(method, kind, M, N):
    rng = np.random.default_rng([M, N, method, len(kind)])
    x, a, y, Y = _tiny_inputs(method, kind, M, N, rng)
    c = rng.random(M) * 2.0
    for cc in (None, c):
        ref = _ref(method, x, a, y, Y, 2.5, c=cc)
        mpv = _mp_eval(method, x, a, y, Y, 2.5, c=cc)
        for k in ("f", "grad", "w", "avg"):
            err = np.abs(np.asarray(ref[k], dtype=H.LD).ravel() - _mp_ld(mpv[k]))
            assert np.all(err <= 1e-17 * np.asarray(ref["s_" + k], dtype=H.LD).ravel() + 1e-320), (k, cc is None)


def _mp_ld(vals):
    """mpmath numbers -> longdouble, correct to the longdouble's precision (hi + lo parts)"""
    import mpmath as mp
    out = []
    for v in vals:
        hi = float(v)
        lo = float(v - mp.mpf(hi))
        out.append(H.LD(hi) + H.LD(lo))
    return np.array(out, dtype=H.LD)


def _cta_cols(N):
    """a CTA-sized slice that CTA 0 does not own: the slice kernel's column block 1 (N / 148 columns wide)"""
    nc = max(8, -(-N // 148))
    return slice(min(nc, N - 1), min(2 * nc, N))


def _violation(ref, **got):
    return max(H.ratios(ref, **got).values())


@pytest.mark.parametrize("M,N", [s for s in SHAPES if s[1] > 5])
@pytest.mark.parametrize("method", [0, 1])
def test_mutants_violate_the_rule(method, M, N):
    """each mutant is an fp64 rounding of what a broken kernel would compute exactly; a correct kernel's error is at
    most C_MAX u scale.  The mutants' weights must miss by 100 x that at least, and their gradients must miss the rule
    too (the gradient's scale carries the cancellation in sum_i r_i (y_ij - avg_i), so a 1e-6 change in one slice's
    weights shows in it at 1e3..1e5 x u scale; the componentwise weights are the sharp check)."""
    need = 100 * C_MAX
    f64 = lambda v: np.asarray(v, dtype=np.float64)
    regimes = ("benign", "conc700_last", "conc3000_last") if method == 0 else ("benign", "x300_last", "w0zero30")
    for regime in regimes:
        variant, x, a, theta = R.case(method, regime, M, N)
        y, Y = R.matrix(variant, M, N)
        ref = _ref(method, x, a, y, Y, theta)
        # structure N - 1 dropped (a lost ragged last tile)
        if method == 0:
            mut = H.logw(x[:-1], a[:-1], y[:, :-1], Y, theta)
            g_mut, w_mut = np.append(f64(mut["grad"]), 0.0), np.append(f64(mut["w"]), 0.0)
        else:
            a2 = a.copy()
            a2[-1] = 0.0
            mut = H.forces(x, a2, y, Y, theta)
            g_mut, w_mut = f64(mut["grad"]), f64(mut["w"])
        if ref["w"][-1] > 1e-300:     # (a structure of weight 0 is dropped at no cost)
            assert _violation(ref, w=w_mut) > need and _violation(ref, grad=g_mut) > C_MAX, (regime, "drop N-1")
        # one CTA-sized slice of e_j scaled by exp(1e-6) (only visible where the slice carries weight)
        cols = _cta_cols(N)
        if np.max(ref["w"][cols]) < 1e-300:
            continue
        if method == 0:
            x2 = x.copy()
            x2[cols] += 1e-6
            mut = H.logw(x2, a, y, Y, theta)
        else:
            a2 = a.copy()
            a2[cols] *= np.exp(1e-6)
            mut = H.forces(x, a2, y, Y, theta)
        assert _violation(ref, w=f64(mut["w"])) > need, (regime, "scaled slice")
        if regime == "benign":      # elsewhere the slice's weights may be far below the gradient's rounding
            assert _violation(ref, grad=f64(mut["grad"])) > C_MAX, (regime, "scaled slice")
    # the maximum over the wrong set: CTA 0's columns only, while the argmax lies elsewhere, > 709 above them (forces:
    # x3000 stretched to a span of 12000), so the stabilised exponentials overflow
    regime = "conc3000_mid" if method == 0 else "x3000_mid"
    variant, x, a, theta = R.case(method, regime, M, N)
    if method == 1:
        x = 4.0 * x
    y, Y = R.matrix(variant, M, N)
    ref = _ref(method, x, a, y, Y, theta)
    z = x if method == 0 else x @ y
    with np.errstate(all="ignore"):
        e = np.exp(z - z[:_cta_cols(N).start].max()) * (1.0 if method == 0 else a)
        w_mut = e / e.sum()
    assert _violation(ref, w=w_mut) > need
    # the w0 guard skipped: a subnormal w0 on the structure of largest x
    if method == 1:
        variant, x, a, theta = R.case(1, "w0subnormal", M, N)
        y, Y = R.matrix(variant, M, N)
        ref = H.forces(x, a, y, Y, theta)
        mut = H.forces(x, a, y, Y, theta, guard_w0=False)
        assert _violation(ref, f=np.array([float(mut["f"])])) > need
