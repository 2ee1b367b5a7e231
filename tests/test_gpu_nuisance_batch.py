"""GPU: per-problem row-affine transforms in the batched engine (row_scale a_k, row_offset b_k: problem k is the one
of the matrix a_k[:, None] * yTilde + b_k[:, None]) and the batched theta series with nuisance-parameter refits built
on them (nuisance.theta_series).

References: the oracle on the explicit transformed matrix for evaluations; opt_lbfgs on a Problem holding that matrix
for minimisations; the reference's own weights <-> nuisance workflow (tests/golden/nuisance_*.npz, recorded by
make_nuisance_golden.py) and the sequential per-theta NuisanceRefit loop for the series."""
import numpy as np
import pytest

from conftest import grad_err, load_golden, rel
from test_gpu_replicates import LS_NOISE, _explicit, _forces_fg_weighted, _kl_np, _planes, _w0, _weights_np

pytestmark = pytest.mark.gpu

LOGW, FORCES = 0, 1
TOL = 1e-11


def _affine(rng, K, M):
    """scales with negative and zero entries, offsets of either sign"""
    A = rng.uniform(-1.5, 2.5, (K, M))
    A[rng.random((K, M)) < 0.1] = 0.0
    A[0] = 1.0
    return A, rng.standard_normal((K, M))


def _tol(its):
    return 1e-8 if its < 50 else 1e-6 if its < 150 else 1e-4 if its < 500 else 1e-3


@pytest.mark.parametrize("M,N,K", [(7, 33, 1), (37, 5001, 8), (300, 1000, 9), (1000, 777, 32), (257, 4099, 24)])
@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_affine_batch_evaluate_matches_oracle(oracle, M, N, K, method):
    import bioen_b200
    forces = method == FORCES
    P = oracle.synthetic_problem(M, N, seed=M + N + K)
    G = 0.1 * np.random.default_rng(K).standard_normal(N)
    rng = np.random.default_rng(M * N + 1)
    C, noise, W0 = _planes(rng, K, M, N, forces)
    A, B = _affine(rng, K, M)
    YT = P["YTilde"].ravel() + noise
    thetas = np.geomspace(100.0, 0.5, K)
    X = (1e-3 * rng.standard_normal((K, M))) if forces else (G + 0.1 * rng.standard_normal((K, N)))
    with bioen_b200.Problem(P["yTilde"]) as p:
        if forces:
            p.set_forces(_w0(np.random.default_rng(1), N), P["YTilde"], 1.0)
        else:
            p.set_logw(G, P["YTilde"], 1.0)
        planes = dict(YTilde=YT, row_weights=C, w0=W0, row_scale=A, row_offset=B)
        f, g, info = p.batch_evaluate(X, thetas, **planes)
        f2, g2, info2 = p.batch_evaluate(X, thetas, gradient=False, **planes)
        assert g2 is None and np.array_equal(f, f2) and np.array_equal(info["averages"], info2["averages"])
        for k in range(K):
            yk = A[k][:, None] * P["yTilde"] + B[k][:, None]
            if forces:
                fo, go = _forces_fg_weighted(oracle, X[k], W0[k], yk, YT[k], C[k], thetas[k])
            else:
                yT, Yk = _explicit(oracle, dict(yTilde=yk), YT[k], C[k])
                fo, go = oracle.logw_fg(X[k], G, yT, Yk, thetas[k])
            assert rel(f[k], fo) < TOL, (k, f[k], fo)
            assert grad_err(g[k], go) < TOL, (k, grad_err(g[k], go))
            w = _weights_np(oracle, forces, X[k], W0[k] if forces else None, yk)
            avg = P["yTilde"] @ w                      # the averages output is that of the RESIDENT matrix
            assert np.max(np.abs(info["averages"][k] - avg)) <= 1e-12 * np.max(np.abs(avg))
            chi2 = 0.5 * np.sum(C[k] * (A[k] * avg + B[k] - YT[k]) ** 2)
            assert rel(info["chi2"][k], chi2) < 1e-12, (k, info["chi2"][k], chi2)
            ref = W0[k] if forces else _weights_np(oracle, False, G, None, None)
            kl = _kl_np(w, ref)
            assert abs(info["kl"][k] - kl) <= 1e-12 * max(1.0, abs(kl)), (k, info["kl"][k], kl)
            assert rel(f[k], thetas[k] * info["kl"][k] + info["chi2"][k]) < 1e-13


@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_identity_planes_are_bit_identical(oracle, method):
    import bioen_b200
    M, N = (100, 20000) if method == LOGW else (300, 4000)
    P = oracle.synthetic_problem(M, N, seed=M + N)
    thetas = np.array([1000.0, 300.0, 100.0, 30.0, 10.0, 3.0, 1.0, 0.3, 100.0, 10.0, 55.0])
    K = thetas.size
    with bioen_b200.Problem(P["yTilde"]) as p:
        if method == LOGW:
            p.set_logw(P["G"], P["YTilde"], 1.0)
        else:
            p.set_forces(_w0(np.random.default_rng(7), N), P["YTilde"], 1.0)
        C = np.random.default_rng(3).random((K, M)) + 0.5
        for ls in (2, 0):
            X, fmin, codes, info = p.theta_scan(thetas, method=method, linesearch=ls)
            for extra in ({}, dict(row_weights=C)):
                Xa, fa, ca, ia = p.batch_minimize(thetas, linesearch=ls, **extra)
                Xb, fb, cb, ib = p.batch_minimize(thetas, linesearch=ls, row_scale=np.ones((K, M)),
                                                  row_offset=np.zeros((K, M)), **extra)
                for key in ("iterations", "evaluations"):
                    assert np.array_equal(ia[key], ib[key])
                for key in ("averages", "chi2", "kl"):
                    assert np.array_equal(ia[key], ib[key], equal_nan=True)
                assert np.array_equal(Xa, Xb) and np.array_equal(fa, fb) and np.array_equal(ca, cb)
                if not extra:
                    assert np.array_equal(X, Xb) and np.array_equal(fmin, fb) and np.array_equal(codes, cb)
                    assert np.array_equal(info["iterations"], ib["iterations"])
            # one plane given alone: the other half is the identity
            Xs, fs, cs, _ = p.batch_minimize(thetas, linesearch=ls, row_scale=np.ones(M))
            Xo, fo, co, _ = p.batch_minimize(thetas, linesearch=ls, row_offset=np.zeros(M))
            assert np.array_equal(Xs, X) and np.array_equal(Xo, X) and np.array_equal(fs, fmin)
            assert np.array_equal(fo, fmin)


@pytest.mark.parametrize("method,M,N", [(LOGW, 37, 5001), (FORCES, 28, 5001), (FORCES, 300, 1000)])
def test_affine_batch_minimize_matches_single_runs(oracle, method, M, N):
    import bioen_b200
    P = oracle.synthetic_problem(M, N, seed=3 * M + N + 1)
    rng = np.random.default_rng(M + 1)
    G = np.zeros(N)
    w0 = _w0(rng, N)
    Y0 = P["YTilde"].ravel()
    theta = 10.0
    K = 12
    A = rng.uniform(0.5, 1.5, (K, M))
    A[:, rng.random(M) < 0.1] *= -1.0
    A[1, :3] = 0.0
    B = 0.5 * rng.standard_normal((K, M))
    with bioen_b200.Problem(P["yTilde"]) as p:
        if method == FORCES:
            p.set_forces(w0, Y0, theta)
        else:
            p.set_logw(G, Y0, theta)
        for ls in (2, 0):
            X, fmin, codes, info = p.batch_minimize(theta, linesearch=ls, row_scale=A, row_offset=B)
            for q in (0, 1, K // 2, K - 1):
                with bioen_b200.Problem(A[q][:, None] * P["yTilde"] + B[q][:, None]) as s:
                    if method == FORCES:
                        s.set_forces(w0, Y0, theta)
                        x1, f1, c1, i1 = s.opt_lbfgs(np.zeros(M), linesearch=ls)
                    else:
                        s.set_logw(G, Y0, theta)
                        x1, f1, c1, i1 = s.opt_lbfgs(G, linesearch=ls)
                its = max(i1["iterations"], int(info["iterations"][q]))
                if method == LOGW:
                    assert codes[q] == c1, (ls, q, codes[q], c1)
                elif codes[q] not in LS_NOISE and c1 not in LS_NOISE:
                    assert codes[q] == c1, (ls, q, codes[q], c1)
                assert rel(fmin[q], f1) < _tol(its), (ls, q, fmin[q], f1, its)
                if codes[q] in (0, 1, 2):
                    assert rel(theta * info["kl"][q] + info["chi2"][q], fmin[q]) < 1e-12


def _golden_cfg():
    return dict(epsilon=1e-7, delta=1e-10, max_iterations=20000)


@pytest.mark.parametrize("kind", ["deer", "scattering"])
def test_theta_series_matches_the_reference_workflow(kind):
    """Two problems of the reference's recorded workflow (make_nuisance_golden.py: workflow) in one batch: problem 0
    at the first theta from the value update_sim_init gave, problem 1 at the second theta from the value the
    reference carried over from the first one.  Both restart every minimisation from G, as the reference does."""
    import bioen_b200
    from bioen_b200 import nuisance as NU
    d = load_golden("nuisance_" + kind)
    rows, n = d["raw"].shape
    its = int(d["wf_iterations"])
    blocks = [NU.Block(kind, 0, rows, err=d["err"], exp_fit=d["exp_fit"], value=float(d["wf_values"][0]), name=kind)]
    base = NU.base_matrix(d["raw"], d["err"])
    G = np.zeros(n)                                   # getGs of the uniform w0
    with bioen_b200.Problem(NU.proc_sim(base, blocks)) as P:
        y0 = P.download()
        P.set_logw(G, d["YTilde"].ravel(), 1.0)
        out = NU.theta_series(P, blocks, d["wf_thetas"], its, values={kind: [d["wf_values"][0], d["wf_values"][its]]},
                              x0=G, **_golden_cfg())
        assert np.array_equal(P.download(), y0)
        for t in range(2):
            for it in range(its):
                k = t * its + it
                assert out["codes"][it, t] in (0, 1, 2)
                assert rel(out["fmin"][it, t], d["wf_fmin"][k]) < 1e-7, (t, it, out["fmin"][it, t], d["wf_fmin"][k])
                w, _ = P.weights(out["x"][it, t])
                assert np.max(np.abs(w - d["wf_weights"][k])) < 1e-5, (t, it)
                v = out["values"][kind][it + 1, t]
                assert abs(v / d["wf_values"][k + 1] - 1.0) < 1e-5, (t, it, v, d["wf_values"][k + 1])


def _synthetic_blocks(NU, N, seed):
    """300 rows: two DEER blocks, one scattering block, fixed rows; data made from known weights and values"""
    rng = np.random.default_rng(seed)
    spec = [(NU.DEER, 0, 90, 0.35), (NU.DEER, 90, 170, 0.5), (NU.SCATTERING, 170, 260, 3e-4), (NU.FIXED, 260, 300, None)]
    M = spec[-1][2]
    raw = np.empty((M, N))
    err = np.empty(M)
    for kind, a, b, _ in spec:
        if kind == NU.DEER:
            t = np.linspace(0.0, 3.0, b - a)[:, None]
            raw[a:b] = np.exp(-t * rng.uniform(0.5, 3.0, N)[None, :])
            err[a:b] = 0.2
        elif kind == NU.SCATTERING:
            q = np.linspace(0.01, 0.5, b - a)[:, None]
            raw[a:b] = 3000.0 * np.exp(-(q * rng.uniform(5.0, 15.0, N)[None, :]) ** 2 / 3.0)
            err[a:b] = 0.2
        else:
            raw[a:b] = rng.standard_normal((b - a, N))
            err[a:b] = 0.5
    base = NU.base_matrix(raw, err)
    wtrue = rng.random(N) ** 4
    wtrue /= wtrue.sum()
    blocks_true = [NU.Block(k, a, b, err=err[a:b], exp_fit=np.ones(b - a), value=v) for k, a, b, v in spec]
    ytrue = NU.proc_sim(base, blocks_true) @ wtrue
    obs = ytrue + rng.standard_normal(M)
    blocks = [NU.Block(k, a, b, err=err[a:b], exp_fit=None if k == NU.FIXED else obs[a:b] * err[a:b],
                       value=None if v is None else 1.2 * v, name="b%d" % q) for q, (k, a, b, v) in enumerate(spec)]
    return base, blocks, obs


@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_theta_series_matches_the_sequential_refit_loop(method):
    import bioen_b200
    from bioen_b200 import nuisance as NU
    M, N = 300, 4000
    base, blocks, Y = _synthetic_blocks(NU, N, seed=5)
    thetas = np.geomspace(1000.0, 10.0, 20)      # converged minimisations (at most ~120 iterations on the oracle)
    its = 3
    start = {"b0": np.linspace(0.3, 0.45, 20), "b2": 2.5e-4}
    G = np.zeros(N)
    w0 = np.full(N, 1.0 / N)
    x0 = np.zeros(M if method == FORCES else N)
    cfg = _golden_cfg()

    def set_data(q, theta):
        if method == FORCES:
            q.set_forces(w0, Y, theta)
        else:
            q.set_logw(G, Y, theta)

    compared = 0
    y_res = NU.proc_sim(base, blocks)
    with bioen_b200.Problem(y_res) as p:
        set_data(p, 1.0)
        out = NU.theta_series(p, blocks, thetas, its, values=start, x0=x0, **cfg)
        assert np.array_equal(p.download(), y_res)
    for t, theta in enumerate(thetas):
        bl = [NU.Block(b.kind, b.start, b.stop, err=b.err, exp_fit=b.exp_fit,
                       value=None if b.kind == NU.FIXED else out["values"][b.name][0, t], name=b.name) for b in blocks]
        with bioen_b200.Problem(NU.proc_sim(base, bl)) as q:
            set_data(q, theta)
            refit = NU.NuisanceRefit(q, bl)
            for it in range(its):
                x, fmin, code, info = q.opt_lbfgs(x0, **cfg)
                if out["codes"][it, t] not in (0, 1, 2) or code not in (0, 1, 2):
                    # both runs end the same way, or a line search that ends at rounding level ends one of them
                    if code != out["codes"][it, t]:
                        for c in (code, out["codes"][it, t]):
                            assert c in (0, 1, 2) or c in LS_NOISE, (t, it, code, out["codes"][it, t])
                    break
                compared += 1
                assert rel(out["fmin"][it, t], fmin) < _tol(info["iterations"]), (t, it, out["fmin"][it, t], fmin)
                w, _ = q.weights(x)
                w[w == 0.0] = 1e-150
                vals = refit.update(w)
                for name, v in vals.items():
                    got = out["values"][name][it + 1, t]
                    assert abs(got / v - 1.0) < 1e-5, (t, it, name, got, v)
    assert compared >= its * thetas.size // 2, compared


def test_plane_refusals(oracle):
    import bioen_b200
    from bioen_b200 import dist as D
    M, N = 20, 300
    P = oracle.synthetic_problem(M, N, seed=11)
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_logw(P["G"], P["YTilde"], 1.0)
        for bad in (np.nan, np.inf, -np.inf):
            a = np.ones((3, M))
            a[2, 5] = bad
            with pytest.raises(RuntimeError, match="row_scale must be finite"):
                p.batch_minimize([1.0, 2.0, 3.0], row_scale=a)
            with pytest.raises(RuntimeError, match="row_offset must be finite"):
                p.batch_evaluate(np.zeros((3, N)), 1.0, row_offset=a - 1.0)
        with pytest.raises(ValueError, match="shape"):
            p.batch_minimize([1.0, 2.0], row_scale=np.ones((2, M + 1)))
        with pytest.raises(ValueError, match="shape"):
            p.batch_evaluate(np.zeros((2, N)), 1.0, row_offset=np.zeros(M - 1))
        with pytest.raises(ValueError, match="disagree"):
            p.batch_minimize([1.0, 2.0], row_scale=np.ones((3, M)))
        # zero scales are allowed; a refused batch leaves the context usable
        X, fmin, codes, info = p.batch_minimize([1.0, 2.0], row_scale=np.zeros(M), max_iterations=3)
        assert np.all(np.isfinite(fmin))
    with D.LocalGroup(P["yTilde"], 2) as grp:
        def run(r, q, lo, hi):
            q.set_logw(np.zeros(hi - lo), P["YTilde"], 1.0)
            with pytest.raises(RuntimeError, match="sharded"):
                q.batch_minimize([1.0, 2.0], row_scale=np.ones((2, M)), row_offset=np.zeros((2, M)))
            return True
        assert all(grp.call(run))
    P = oracle.synthetic_problem(256, 1000, seed=2)
    with bioen_b200.Problem(P["yTilde"], structure_major_only=True) as p:
        p.set_forces(np.full(1000, 1e-3), P["YTilde"], 1.0)
        with pytest.raises(RuntimeError, match="row-major"):
            p.batch_minimize([1.0, 2.0], row_scale=np.ones((2, 256)))
        with pytest.raises(RuntimeError, match="row-major"):
            p.batch_evaluate(np.zeros((2, 256)), 1.0, row_offset=np.zeros(256))
