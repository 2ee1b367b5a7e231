"""GPU: batched replicates -- K <= 32 problems on one resident yTilde with per-problem YTilde, observable weights
(chi^2 = 1/2 sum_i c_i r_i^2) and, for the forces method, reference weights w0 -- and the bootstrap /
cross-validation helpers built on them.

For the log-weights method the equivalent explicit problem of observable weights c is the one whose rows of yTilde and
YTilde are scaled by sqrt(c): the weights do not depend on yTilde, and its chi^2 and gradient are those of the weighted
problem.  The forces method's weights are w ~ w0 exp(f . y), so scaling rows would change the parametrisation; there
the reference is the oracle's own f and gradient with the back-projected residual replaced by c r
(_forces_fg_weighted), and end points are compared with the oracle's liblbfgs restatement run on it.
Per-evaluation parity is 1e-11, as for every evaluation path of the library; end points follow the rules of the
theta-scan tests."""
import numpy as np
import pytest

from conftest import load_golden, grad_err, rel

pytestmark = pytest.mark.gpu

LOGW, FORCES = 0, 1
TOL = 1e-11
LS_NOISE = {-998, -1001, -1000, -999, -996}   # line-search verdicts at rounding level (test_gpu_minimizers.py)


def _w0(rng, N, zeros=False):
    w0 = rng.random(N) + 0.2
    if zeros:
        w0[rng.random(N) < 0.3] = 0.0
    return w0 / w0.sum()


def _planes(rng, K, M, N, forces):
    """K problems of mixed kinds: integer multinomial counts (with zero rows), real weights with zero rows, noise
    replicates, and for forces resampled w0 with zeros."""
    C = np.ones((K, M))
    for k in range(K):
        if k % 3 == 0:
            C[k] = rng.multinomial(M, np.full(M, 1.0 / M))
        elif k % 3 == 1:
            C[k] = rng.random(M) * 2.0
            C[k, rng.random(M) < 0.25] = 0.0
    noise = rng.standard_normal((K, M))
    w0 = None
    if forces:
        w0 = np.stack([_w0(rng, N, zeros=(k % 2 == 0)) for k in range(K)])
    return C, noise, w0


def _explicit(oracle, P, YTk, c):
    """(yTilde, YTilde) of the explicit problem with observable weights c"""
    s = np.sqrt(c)
    return P["yTilde"] * s[:, None], YTk * s


def _forces_fg_weighted(oracle, x, w0, yT, Y, c, theta):
    """forces f and gradient with chi^2 = 1/2 sum_i c_i r_i^2: the oracle's gradient with YTilde replaced by avg - c r
    (its residual is then c r, which is what the gradient back-projects), and its objective with 1/2 sum (c r)^2
    swapped for 1/2 sum c r^2"""
    avg = oracle.average(yT, oracle.forces_weights(x, w0, yT))
    r = avg - Y
    f, g = oracle.forces_fg(x, w0, yT, avg - c * r, theta)
    return f - 0.5 * np.dot(c * r, c * r) + 0.5 * np.dot(c * r, r), g


def _weights_np(oracle, forces, x, G_or_w0, yT):
    if forces:
        return oracle.forces_weights_np(x, G_or_w0, yT)
    e = np.exp(x - x.max())
    return e / e.sum()


def _kl_np(w, ref):
    ok = (w >= np.finfo(float).tiny) & (ref >= np.finfo(float).tiny)
    return float(np.sum(w[ok] * np.log(w[ok] / ref[ok])))


def _check_eval(oracle, p, P, forces, G, K, seed):
    M, N = P["yTilde"].shape
    rng = np.random.default_rng(seed)
    C, noise, W0 = _planes(rng, K, M, N, forces)
    YT = P["YTilde"].ravel() + noise
    thetas = np.geomspace(100.0, 0.5, K)
    X = (1e-3 * rng.standard_normal((K, M))) if forces else (G + 0.1 * rng.standard_normal((K, N)))
    f, g, info = p.batch_evaluate(X, thetas, YTilde=YT, row_weights=C, w0=W0)
    f2, g2, info2 = p.batch_evaluate(X, thetas, YTilde=YT, row_weights=C, w0=W0, gradient=False)
    assert g2 is None and np.array_equal(f, f2) and np.array_equal(info["averages"], info2["averages"])
    for k in range(K):
        if forces:
            fo, go = _forces_fg_weighted(oracle, X[k], W0[k], P["yTilde"], YT[k], C[k], thetas[k])
        else:
            yT, Yk = _explicit(oracle, P, YT[k], C[k])
            fo, go = oracle.logw_fg(X[k], G, yT, Yk, thetas[k])
        assert rel(f[k], fo) < TOL, (k, f[k], fo)
        assert grad_err(g[k], go) < TOL, (k, grad_err(g[k], go))
        w = _weights_np(oracle, forces, X[k], W0[k] if forces else None, P["yTilde"])
        avg = P["yTilde"] @ w
        assert np.max(np.abs(info["averages"][k] - avg)) <= 1e-12 * np.max(np.abs(avg))
        chi2 = 0.5 * np.sum(C[k] * (avg - YT[k]) ** 2)
        assert rel(info["chi2"][k], chi2) < 1e-12, (k, info["chi2"][k], chi2)
        ref = W0[k] if forces else _weights_np(oracle, False, G, None, None)
        kl = _kl_np(w, ref)
        assert abs(info["kl"][k] - kl) <= 1e-12 * max(1.0, abs(kl)), (k, info["kl"][k], kl)
        assert rel(f[k], thetas[k] * info["kl"][k] + info["chi2"][k]) < 1e-13


@pytest.mark.parametrize("M,N,K", [(7, 33, 1), (37, 5001, 8), (300, 1000, 9), (1000, 777, 32), (257, 4099, 24)])
@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_batch_evaluate_matches_oracle(oracle, M, N, K, method):
    import bioen_b200
    P = oracle.synthetic_problem(M, N, seed=M + N + K)
    G = 0.1 * np.random.default_rng(K).standard_normal(N)
    with bioen_b200.Problem(P["yTilde"]) as p:
        if method == FORCES:
            p.set_forces(_w0(np.random.default_rng(1), N), P["YTilde"], 1.0)
        else:
            p.set_logw(G, P["YTilde"], 1.0)
        _check_eval(oracle, p, P, method == FORCES, G, K, seed=M * N)


@pytest.mark.parametrize("name", ["data_potra_part_2_logw_M205xN10", "data_forces_M64xN64"])
def test_batch_evaluate_matches_oracle_reference_fixture(oracle, name):
    import bioen_b200
    d = load_golden(name)
    P = dict(yTilde=np.ascontiguousarray(d["yTilde"]), YTilde=np.asarray(d["YTilde"]).ravel())
    forces = d["kind"] != "logw"
    G = None if forces else np.asarray(d["G"]).ravel()
    with bioen_b200.Problem(P["yTilde"]) as p:
        if forces:
            p.set_forces(d["w0"], P["YTilde"], d["theta"])
        else:
            p.set_logw(G, P["YTilde"], d["theta"])
        _check_eval(oracle, p, P, forces, G, 11, seed=5)


@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_trivial_planes_reproduce_theta_scan_bit_for_bit(oracle, method):
    import bioen_b200
    M, N = (100, 20000) if method == LOGW else (300, 4000)
    P = oracle.synthetic_problem(M, N, seed=M + N)
    thetas = np.array([1000.0, 300.0, 100.0, 30.0, 10.0, 3.0, 1.0, 0.3, 100.0, 10.0, 55.0])
    K = thetas.size
    w0 = _w0(np.random.default_rng(7), N)
    with bioen_b200.Problem(P["yTilde"]) as p:
        if method == LOGW:
            p.set_logw(P["G"], P["YTilde"], 1.0)
        else:
            p.set_forces(w0, P["YTilde"], 1.0)
        planes = dict(YTilde=np.tile(P["YTilde"].ravel(), (K, 1)), row_weights=np.ones((K, M)))
        if method == FORCES:
            planes["w0"] = np.tile(w0, (K, 1))
        for ls in (2, 0):
            X, fmin, codes, info = p.theta_scan(thetas, method=method, linesearch=ls)
            Xb, fb, cb, ib = p.batch_minimize(thetas, linesearch=ls, **planes)
            assert np.array_equal(X, Xb) and np.array_equal(fmin, fb) and np.array_equal(codes, cb)
            assert np.array_equal(info["iterations"], ib["iterations"])
            assert np.array_equal(info["evaluations"], ib["evaluations"])
            # identical inputs give identical planes
            assert np.array_equal(Xb[2], Xb[8]) and fb[4] == fb[9]


def _single(oracle, P, method, G, kind, c, Yk, w0k, theta, ls):
    """One replicate alone: opt_lbfgs on its explicit problem, or for forces with observable weights the oracle's
    liblbfgs on the weighted f and gradient.  Returns (fmin, code, iterations)."""
    import bioen_b200
    if method == FORCES and kind == "observables":
        r = oracle.lbfgs(lambda v: _forces_fg_weighted(oracle, v, w0k, P["yTilde"], Yk, c, theta),
                         np.zeros(P["yTilde"].shape[0]), linesearch=ls)
        return r["fx"], r["code"], r["iterations"]
    yT, Y = _explicit(oracle, P, Yk, c)
    with bioen_b200.Problem(yT) as q:
        if method == FORCES:
            q.set_forces(w0k, Y, theta)
            x, f, code, info = q.opt_lbfgs(np.zeros(yT.shape[0]), linesearch=ls)
        else:
            q.set_logw(G, Y, theta)
            x, f, code, info = q.opt_lbfgs(G, linesearch=ls)
        return f, code, info["iterations"]


@pytest.mark.parametrize("method,M,N,kinds", [(LOGW, 37, 5001, ("observables", "noise")),
                                              (FORCES, 28, 5001, ("observables", "noise", "structures")),
                                              (FORCES, 300, 1000, ("observables", "structures"))])
def test_batch_minimize_matches_single_runs(oracle, method, M, N, kinds):
    import bioen_b200
    P = oracle.synthetic_problem(M, N, seed=3 * M + N)
    rng = np.random.default_rng(M)
    G = np.zeros(N)
    w0 = _w0(rng, N)
    Y0 = P["YTilde"].ravel()
    theta = 10.0
    K = 12
    with bioen_b200.Problem(P["yTilde"]) as p:
        if method == FORCES:
            p.set_forces(w0, Y0, theta)
        else:
            p.set_logw(G, Y0, theta)
        for kind in kinds:
            C, Y, W = np.ones((K, M)), np.tile(Y0, (K, 1)), np.tile(w0, (K, 1))
            if kind == "observables":
                C = rng.multinomial(M, np.full(M, 1.0 / M), size=K).astype(float)
                planes = dict(row_weights=C)
            elif kind == "noise":
                Y = Y0 + rng.standard_normal((K, M))
                planes = dict(YTilde=Y)
            else:
                W = w0 * rng.multinomial(N, np.full(N, 1.0 / N), size=K)
                W /= W.sum(axis=1, keepdims=True)
                planes = dict(w0=W)
            for ls in (2, 0):
                X, fmin, codes, info = p.batch_minimize(theta, linesearch=ls, **planes)
                for q in (0, K // 2, K - 1):
                    f1, c1, it1 = _single(oracle, P, method, G, kind, C[q], Y[q], W[q], theta, ls)
                    its = max(it1, int(info["iterations"][q]))
                    tol = 1e-8 if its < 50 else 1e-6 if its < 150 else 1e-4 if its < 500 else 1e-3
                    if method == LOGW:
                        assert codes[q] == c1, (kind, ls, q, codes[q], c1)
                    elif codes[q] not in LS_NOISE and c1 not in LS_NOISE:
                        assert codes[q] == c1, (kind, ls, q, codes[q], c1)
                    assert rel(fmin[q], f1) < tol, (kind, ls, q, fmin[q], f1, its)
                    if codes[q] in (0, 1, 2):     # the report is taken at the returned point
                        assert rel(theta * info["kl"][q] + info["chi2"][q], fmin[q]) < 1e-12


def test_batch_inputs_are_checked(oracle):
    import bioen_b200
    M, N = 20, 300
    P = oracle.synthetic_problem(M, N, seed=11)
    with bioen_b200.Problem(P["yTilde"]) as p:
        with pytest.raises(RuntimeError, match="set_logw or set_forces"):
            p.batch_minimize([1.0, 2.0])
        p.set_logw(P["G"], P["YTilde"], 1.0)
        with pytest.raises(RuntimeError, match="need the forces method"):
            p.batch_minimize([1.0, 2.0], w0=np.full((2, N), 1.0 / N))
        with pytest.raises(ValueError, match="1..32"):
            p.batch_minimize(np.ones(33))
        with pytest.raises(ValueError, match="shape"):
            p.batch_minimize([1.0, 2.0], row_weights=np.ones((2, M + 1)))
        with pytest.raises(ValueError, match="disagree"):
            p.batch_minimize([1.0, 2.0, 3.0], YTilde=np.zeros((2, M)))
        with pytest.raises(ValueError, match="shape"):
            p.batch_evaluate(np.zeros((2, N - 1)), [1.0, 2.0])
        p.set_forces(np.full(N, 1.0 / N), P["YTilde"], 1.0)
        for bad in (-1.0, np.nan, np.inf):
            c = np.ones((3, M))
            c[1, 4] = bad
            with pytest.raises(RuntimeError, match="row weights must be finite and >= 0"):
                p.batch_minimize([1.0, 2.0, 3.0], row_weights=c)
        Y = np.zeros((2, M))
        Y[0, 3] = np.nan
        with pytest.raises(RuntimeError, match="YTilde must be finite"):
            p.batch_evaluate(np.zeros((2, M)), 1.0, YTilde=Y)
        W = np.full((2, N), 1.0 / N)
        W[1] = 0.0
        with pytest.raises(RuntimeError, match="positive sum"):
            p.batch_minimize(1.0, w0=W)
        W[1] = 1.0 / N
        W[0, 7] = -1e-3
        with pytest.raises(RuntimeError, match="w0 must be finite and >= 0"):
            p.batch_minimize(1.0, w0=W)
        # a refused batch leaves the context usable
        X, fmin, codes, info = p.batch_minimize([1.0, 2.0], max_iterations=3)
        assert np.all(np.isfinite(fmin)) and info["averages"].shape == (2, M)
        # refused L-BFGS parameters: codes say so, the report is NaN
        X, fmin, codes, info = p.batch_minimize([1.0, 2.0], delta=-1.0)
        assert list(codes) == [-1015] * 2 and np.all(np.isnan(info["chi2"]))
    # structure-major-only mode keeps the theta scan's error
    P = oracle.synthetic_problem(256, 1000, seed=2)
    with bioen_b200.Problem(P["yTilde"], structure_major_only=True) as p:
        p.set_forces(np.full(1000, 1e-3), P["YTilde"], 1.0)
        with pytest.raises(RuntimeError, match="row-major"):
            p.batch_minimize([1.0, 2.0], row_weights=np.ones((2, 256)))
        with pytest.raises(RuntimeError, match="row-major"):
            p.batch_evaluate(np.zeros((2, 256)), 1.0)


@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_bootstrap_reproducible_and_equal_to_direct_batches(oracle, method):
    import bioen_b200
    from bioen_b200 import replicates
    M, N = 37, 5001
    P = oracle.synthetic_problem(M, N, seed=17)
    kinds = ("observables", "noise") + (("structures",) if method == FORCES else ())
    with bioen_b200.Problem(P["yTilde"]) as p:
        if method == FORCES:
            p.set_forces(_w0(np.random.default_rng(3), N), P["YTilde"], 1.0)
        else:
            p.set_logw(P["G"], P["YTilde"], 1.0)
        if method == LOGW:
            with pytest.raises(ValueError, match="forces method"):
                replicates.bootstrap(p, 40, "structures", 10.0)
        for kind in kinds:
            a = replicates.bootstrap(p, 40, kind, 10.0, seed=1, max_iterations=200)
            b = replicates.bootstrap(p, 40, kind, 10.0, seed=1, max_iterations=200)
            for key in ("averages", "fmin", "codes", "chi2", "kl", "x"):
                assert np.array_equal(a[key], b[key], equal_nan=True), (kind, key)
            assert np.all(np.isin(a["codes"], (0, 1, 2, -997) + tuple(LS_NOISE)))
            # the second chunk (replicates 32..39) again, from its recorded inputs
            if kind == "observables":
                planes = dict(row_weights=a["counts"][32:].astype(float))
            elif kind == "noise":
                planes = dict(YTilde=p.YTilde + a["noise"][32:])
            else:
                w = p.w0 * a["counts"][32:]
                planes = dict(w0=w * (p.w0.sum() / w.sum(axis=1, keepdims=True)))
            X, fmin, codes, info = p.batch_minimize(10.0, max_iterations=200, **planes)
            ok = np.isin(codes, (0, 1, 2))
            assert np.array_equal(X, a["x"][32:]) and np.array_equal(fmin, a["fmin"][32:])
            assert np.array_equal(codes, a["codes"][32:])
            assert np.array_equal(info["averages"][ok], a["averages"][32:][ok])
            assert np.array_equal(info["chi2"][ok], a["chi2"][32:][ok])


def test_cross_validate_held_out_chi2(oracle):
    import bioen_b200
    from bioen_b200 import replicates
    M, N = 40, 3001
    P = oracle.synthetic_problem(M, N, seed=23)
    thetas = np.geomspace(1000.0, 1.0, 7)
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_forces(_w0(np.random.default_rng(4), N), P["YTilde"], 1.0)
        out = replicates.cross_validate(p, thetas, folds=5, seed=2)
        assert out["held_out_chi2"].shape == (7, 5)
        Y = p.YTilde
        for t in range(7):
            for f in range(5):
                if out["codes"][t, f] not in (0, 1, 2):
                    assert np.isnan(out["held_out_chi2"][t, f])
                    continue
                fold = out["fold"] == f
                want = 0.5 * np.sum((out["averages"][t, f, fold] - Y[fold]) ** 2)
                assert rel(out["held_out_chi2"][t, f], want) < 1e-14
                train = 0.5 * np.sum((out["averages"][t, f, ~fold] - Y[~fold]) ** 2)
                assert rel(out["chi2"][t, f], train) < 1e-12
        again = replicates.cross_validate(p, thetas, folds=5, seed=2)
        assert np.array_equal(out["held_out_chi2"], again["held_out_chi2"], equal_nan=True)
