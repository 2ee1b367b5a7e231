"""GPU: the device-resident minimisers against the reference's end points (golden, produced by the unmodified
reference C code + liblbfgs + GSL) and against the oracle's restatement run on identical inputs.

Tolerances (north_star): same final objective to 1e-8 relative, converged weights within 1e-6 max-abs.
"""
import numpy as np
import pytest

from conftest import FORCES_FIXTURES, LOGW_FIXTURES, load_golden, rel, select_eval_path

pytestmark = pytest.mark.gpu

F_TOL = 1e-8
W_TOL = 1e-6
GSL_ALGS = ["conjugate_fr", "conjugate_pr", "bfgs2", "bfgs", "steepest_descent"]


def _softmax(g):
    e = np.exp(g - g.max())
    return e / e.sum()


def _setup(p, d):
    if d["kind"] == "logw":
        p.set_logw(d["G"], d["YTilde"], d["theta"])
        return d["GInit"].ravel()
    p.set_forces(d["w0"], d["YTilde"], d["theta"])
    return d["forces_init"].ravel()


def _bound(d, key):
    """1e-8, widened to 30x the reference's OWN end-point noise for this problem/minimiser where that is larger
    (|fmin - fmin_alt| between its reproducible and its fast OpenMP mode, stored by make_golden.py): long,
    chaotic trajectories (steepest descent hitting max_iterations, Fletcher-Reeves on ill-conditioned data) do
    not reproduce to 1e-8 between two runs of the reference itself."""
    noise = abs(d[key + "_fmin_alt"] - d[key + "_fmin"]) / abs(d[key + "_fmin"])
    return max(F_TOL, 30.0 * noise) if np.isfinite(noise) else None


@pytest.mark.parametrize("name", LOGW_FIXTURES + FORCES_FIXTURES)
@pytest.mark.parametrize("ls", [0, 1, 2, 3])
@pytest.mark.parametrize("persistent", [0, 1, 2])
def test_lbfgs_matches_reference_endpoint(name, ls, persistent):
    import bioen_b200
    d = load_golden(name)
    key = "lbfgs%d" % ls
    with bioen_b200.Problem(d["yTilde"]) as p:
        select_eval_path(p, persistent)
        x0 = _setup(p, d)
        x, fmin, code, info = p.opt_lbfgs(x0, linesearch=ls)
        assert code == d[key + "_code"], (code, info)
        assert rel(fmin, d[key + "_fmin"]) < _bound(d, key), (rel(fmin, d[key + "_fmin"]), _bound(d, key))
        if code in (0, 1, 2):
            # fmin must be the objective at the returned point (test_find_opt_analytical_grad_logw.py:162-188);
            # after a failed line search liblbfgs returns the reverted x with the last trial's f (lbfgs.c:475-481)
            assert rel(p.objective(x), fmin) < 5e-13
            if d["kind"] == "logw":
                assert np.max(np.abs(_softmax(x) - _softmax(d[key + "_x"]))) < W_TOL
            else:
                w, _ = p.weights(x)
                wr, _ = p.weights(d[key + "_x"])
                assert np.max(np.abs(w - wr)) < W_TOL


# End points that the stored mode-to-mode noise of the reference under-estimates.  Fletcher-Reeves on
# data_potra_part_1 (808 x 80, ill-conditioned) passes BioEn's max|g| < 1e-3 stop test in two different places,
# 8.3e-5 apart in f: the CPU oracle alone shows it (C evaluator 4042.786885 after 644 iterations, NumPy evaluator
# 4043.121431 after 293, start point perturbed by 1e-15: 4043.121738 after 317, by 1e-14: GSL code 27).  The
# reference's two OpenMP modes happen to land on the same side; the persistent kernel's rounding lands on the other.
SENSITIVE_END_POINTS = {("conjugate_fr", "data_potra_part_1_logw_M808xN80"): 3e-4}


@pytest.mark.parametrize("name", ["data_16x15", "data_deer_test_logw_M808xN10", "data_potra_part_2_logw_M205xN10",
                                  "data_potra_part_1_logw_M808xN80", "data_forces_M64xN64",
                                  "data_deer_test_forces_M808xN10"])
@pytest.mark.parametrize("alg", GSL_ALGS)
@pytest.mark.parametrize("persistent", [0, 1, 2])
def test_gsl_matches_reference_endpoint(name, alg, persistent):
    """Both evaluation paths (stand-alone kernels / persistent kernel: different partial-sum cuts, i.e. different
    rounding) against the reference's end point."""
    import bioen_b200
    from bioen_b200.optimize.ext import c_bioen
    d = load_golden(name)
    key = "gsl_" + alg
    with bioen_b200.Problem(d["yTilde"]) as p:
        select_eval_path(p, persistent)
        x0 = _setup(p, d)
        x, fmin, code, info = p.opt_gsl(x0, algorithm=c_bioen.get_gsl_method(alg))
        assert code == d[key + "_code"], (code, info)
        bound = max(_bound(d, key), SENSITIVE_END_POINTS.get((alg, name), 0.0))
        assert rel(fmin, d[key + "_fmin"]) < bound, (rel(fmin, d[key + "_fmin"]), bound)
        assert rel(p.objective(x), fmin) < 5e-13


def test_gsl_chaotic_fixture_stays_within_reference_tolerance():
    """data_potra_part_2_logw_M808xN10 (808 x 100; excluded from the reference's own test list): |grad|_inf
    jumps by 4 orders of magnitude between consecutive bfgs2 iterations near the end, the reference's two
    OpenMP modes end with different GSL codes (conjugate_fr: 0 vs 27) and its vector_bfgs end point is NaN.
    Checked at the reference's own 10 % bar only."""
    import bioen_b200
    from bioen_b200.optimize.ext import c_bioen
    d = load_golden("data_potra_part_2_logw_M808xN10")
    with bioen_b200.Problem(d["yTilde"]) as p:
        x0 = _setup(p, d)
        for alg in ("conjugate_pr", "bfgs2"):
            x, fmin, code, info = p.opt_gsl(x0, algorithm=c_bioen.get_gsl_method(alg))
            assert code in (0, -2, 27)
            assert rel(fmin, d["gsl_%s_fmin" % alg]) < 1e-6
            assert rel(fmin, d["ref_scalar"]) < 1e-1


def test_lbfgs_synthetic_vs_oracle_and_reference(oracle):
    """SURVEY 8d synthetic problem: same stop code, evaluation count and end point as liblbfgs."""
    import bioen_b200
    d = load_golden("synthetic_M100xN20000")
    P = oracle.synthetic_problem(int(d["M"]), int(d["N"]), seed=int(d["seed"]))
    theta = d["theta"]
    with bioen_b200.Problem(P["yTilde"]) as p:
        for ls in (0, 2):
            p.set_logw(P["G"], P["YTilde"], theta)
            x, fmin, code, info = p.opt_lbfgs(P["GInit"], linesearch=ls)
            assert code == d["logw_lbfgs%d_code" % ls]
            assert rel(fmin, d["logw_lbfgs%d_fmin" % ls]) < F_TOL
            assert np.max(np.abs(_softmax(x) - _softmax(d["logw_lbfgs%d_x" % ls]))) < W_TOL
            r = oracle.lbfgs(lambda v: oracle.logw_fg(v, P["G"], P["yTilde"], P["YTilde"], theta), P["GInit"],
                             linesearch=ls)
            assert r["code"] == code and rel(fmin, r["fx"]) < F_TOL
            assert abs(r["iterations"] - info["iterations"]) <= 2
            p.set_forces(P["w0"], P["YTilde"], theta)
            x, fmin, code, info = p.opt_lbfgs(P["forces_init"], linesearch=ls)
            assert code == d["forces_lbfgs%d_code" % ls]
            assert rel(fmin, d["forces_lbfgs%d_fmin" % ls]) < F_TOL
        p.set_logw(P["G"], P["YTilde"], theta)
        x, fmin, code, info = p.opt_gsl(P["GInit"])
        assert code == d["logw_gsl_bfgs2_code"] and rel(fmin, d["logw_gsl_bfgs2_fmin"]) < F_TOL
        p.set_forces(P["w0"], P["YTilde"], theta)
        x, fmin, code, info = p.opt_gsl(P["forces_init"])
        assert code == d["forces_gsl_bfgs2_code"] and rel(fmin, d["forces_gsl_bfgs2_fmin"]) < F_TOL


def test_lbfgs_parameter_validation_codes():
    """lbfgs.c:286-364: each invalid parameter maps to its own negative code, before any evaluation."""
    import bioen_b200
    d = load_golden("data_16x15")
    with bioen_b200.Problem(d["yTilde"]) as p:
        x0 = _setup(p, d)
        for kw, code in ((dict(epsilon=-1.0), -1017), (dict(past=-1), -1016), (dict(delta=-1.0), -1015),
                         (dict(ftol=-1.0), -1011), (dict(wolfe=1.5), -1010), (dict(gtol=-0.1), -1009),
                         (dict(max_linesearch=0), -1007), (dict(linesearch=7), -1014)):
            assert p.opt_lbfgs(x0, **kw)[2] == code, kw
        # max_iterations reached: -997, and x / fmin of the last iterate are kept
        x, fmin, code, info = p.opt_lbfgs(x0, max_iterations=2)
        assert code == -997 and info["iterations"] == 2 and fmin < p.objective(x0)
        # already minimised start point
        xo = p.opt_lbfgs(x0, epsilon=1e-9, delta=0.0, past=0)[0]
        assert p.opt_lbfgs(xo, epsilon=1e-3)[2] == 2


def test_part1_drivers_and_error_convention():
    """c_bioen mirror: success returns (x, fmin); failures raise RuntimeError with 'return code'
    (test_error_opt_logw.py / test_error_opt_forces.py)."""
    from bioen_b200 import optimize
    from bioen_b200.optimize.ext import c_bioen
    d = load_golden("data_16x15")
    cfg = optimize.minimize.Parameters("lbfgs")
    cfg["verbose"] = False
    cfg["cache_ytilde_transposed"] = False
    x, fmin = c_bioen.bioen_opt_lbfgs_logw(d["GInit"].ravel(), d["G"], d["yTilde"], d["YTilde"], d["theta"], cfg)
    assert rel(fmin, d["lbfgs2_fmin"]) < F_TOL and x.shape == (16,)
    cfg["params"]["delta"] = -1
    with pytest.raises(RuntimeError, match="return code"):
        c_bioen.bioen_opt_lbfgs_logw(d["GInit"].ravel(), d["G"], d["yTilde"], d["YTilde"], d["theta"], cfg)
    cfg = optimize.minimize.Parameters("gsl")
    cfg["verbose"] = False
    cfg["cache_ytilde_transposed"] = False
    x, fmin = c_bioen.bioen_opt_bfgs_logw(d["GInit"].ravel(), d["G"], d["yTilde"], d["YTilde"], d["theta"], cfg)
    assert rel(fmin, d["gsl_bfgs2_fmin"]) < F_TOL
    cfg["algorithm"] = "TEST_INVALID"
    with pytest.raises(RuntimeError, match="return code"):
        c_bioen.bioen_opt_bfgs_logw(d["GInit"].ravel(), d["G"], d["yTilde"], d["YTilde"], d["theta"], cfg)
    d = load_golden("data_forces_M64xN64")
    cfg = optimize.minimize.Parameters("lbfgs")
    cfg["verbose"] = False
    cfg["cache_ytilde_transposed"] = False
    x, fmin = c_bioen.bioen_opt_lbfgs_forces(d["forces_init"].ravel(), d["w0"], d["yTilde"], d["YTilde"],
                                             d["theta"], cfg)
    assert rel(fmin, d["lbfgs2_fmin"]) < F_TOL and x.shape == (64,)
    cfg["params"]["delta"] = -1
    with pytest.raises(RuntimeError, match="return code"):
        c_bioen.bioen_opt_lbfgs_forces(d["forces_init"].ravel(), d["w0"], d["yTilde"], d["YTilde"], d["theta"], cfg)
    cfg = optimize.minimize.Parameters("gsl")
    cfg["verbose"] = False
    cfg["cache_ytilde_transposed"] = False
    x, fmin = c_bioen.bioen_opt_bfgs_forces(d["forces_init"].ravel(), d["w0"], d["yTilde"], d["YTilde"],
                                            d["theta"], cfg)
    assert rel(fmin, d["gsl_bfgs2_fmin"]) < F_TOL


# ---- theta scan: K problems minimised together (batched fp64 tensor-core evaluations, lockstep L-BFGS) -----------
def test_theta_scan_matches_single_problem_runs(oracle):
    import bioen_b200
    P = oracle.synthetic_problem(100, 20000, seed=12345)
    thetas = np.array([1000.0, 300.0, 100.0, 30.0, 10.0, 3.0, 1.0, 0.3, 100.0, 10.0, 55.0])   # K = 11 (padded to 16)
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_logw(P["G"], P["YTilde"], 1.0)
        for ls in (2, 0):
            X, fmin, codes, info = p.theta_scan(thetas, linesearch=ls)
            assert X.shape == (thetas.size, 20000)
            for q, th in enumerate(thetas):
                p.set_theta(th)
                x1, f1, c1, i1 = p.opt_lbfgs(P["GInit"], linesearch=ls)
                tol = 1e-8 if i1["iterations"] < 150 else 1e-4      # long delta-stopped runs are chaotic
                assert codes[q] == c1, (th, ls, codes[q], c1)
                assert rel(fmin[q], f1) < tol, (th, ls, fmin[q], f1, info["iterations"][q], i1)
                if i1["iterations"] < 150:
                    assert abs(int(info["iterations"][q]) - i1["iterations"]) <= 2
                assert rel(p.objective(X[q]), fmin[q]) < 5e-13
                if i1["iterations"] < 150:
                    assert np.max(np.abs(_softmax(X[q]) - _softmax(x1))) < W_TOL
            # identical thetas give identical results (planes do not interact)
            assert fmin[2] == fmin[8] and np.array_equal(X[2], X[8])
            assert fmin[4] == fmin[9] and np.array_equal(X[4], X[9])


def test_theta_scan_against_reference_golden(oracle):
    """theta = 10 plane of a scan reproduces the reference's liblbfgs end point stored in the golden file."""
    import bioen_b200
    d = load_golden("synthetic_M100xN20000")
    P = oracle.synthetic_problem(int(d["M"]), int(d["N"]), seed=int(d["seed"]))
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_logw(P["G"], P["YTilde"], d["theta"])
        for ls in (0, 2):
            X, fmin, codes, info = p.theta_scan([d["theta"], 2 * d["theta"]], linesearch=ls)
            assert codes[0] == d["logw_lbfgs%d_code" % ls]
            assert rel(fmin[0], d["logw_lbfgs%d_fmin" % ls]) < F_TOL
            assert np.max(np.abs(_softmax(X[0]) - _softmax(d["logw_lbfgs%d_x" % ls]))) < W_TOL


@pytest.mark.parametrize("M,N,K", [(7, 33, 1), (37, 5001, 8), (300, 1000, 9), (1000, 777, 32), (257, 4099, 24)])
def test_theta_scan_ragged_shapes(oracle, M, N, K):
    import bioen_b200
    P = oracle.synthetic_problem(M, N, seed=M + N + K)
    rng = np.random.default_rng(K)
    G = 0.1 * rng.standard_normal(N)
    thetas = np.geomspace(100.0, 1.0, K)
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_logw(G, P["YTilde"], 1.0)
        X, fmin, codes, info = p.theta_scan(thetas, x0=G, max_iterations=15)
        for q in (0, K // 2, K - 1):
            p.set_theta(thetas[q])
            x1, f1, c1, i1 = p.opt_lbfgs(G, max_iterations=15)
            assert codes[q] == c1 and rel(fmin[q], f1) < 1e-9, (q, codes[q], c1, fmin[q], f1)
            fo, _ = oracle.logw_fg(X[q], G, P["yTilde"], P["YTilde"], thetas[q])
            assert rel(fo, fmin[q]) < 1e-11 or codes[q] < 0


def test_increasing_gradient_keeps_the_last_accepted_objective(oracle):
    """A search that ends in LBFGSERR_INCREASEGRADIENT (the new direction is not a descent direction) returns before
    its first trial in liblbfgs: x is the last accepted point and fmin its objective.  The minimisers enqueue that
    trial before the slope is known; its objective must not become fmin.  Backtracking (linesearch 1) on this seeded
    problem ends so at theta = 0.01 (7 iterations) and theta = 1."""
    import bioen_b200
    P = oracle.synthetic_problem(8, 40, seed=5)
    thetas = [0.01, 1.0]
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_logw(P["G"], P["YTilde"], 1.0)
        X, fmin, codes, info = p.theta_scan(thetas, x0=P["GInit"], linesearch=1)
        for q, th in enumerate(thetas):
            ref = oracle.lbfgs(lambda x: oracle.logw_fg(x, P["G"], P["yTilde"], P["YTilde"], th), P["GInit"],
                               linesearch=1)
            assert ref["code"] == -994
            p.set_theta(th)
            x1, f1, c1, _ = p.opt_lbfgs(P["GInit"], linesearch=1)
            for x, f, code in ((X[q], fmin[q], codes[q]), (x1, f1, c1)):
                assert code == -994, (th, code)
                assert rel(f, ref["fx"]) < 1e-11, (th, f, ref["fx"])
                assert rel(f, p.objective(x)) < 1e-11, (th, f, p.objective(x))


def test_theta_scan_errors_and_chunking(oracle):
    import bioen_b200
    from bioen_b200 import optimize
    P = oracle.synthetic_problem(20, 600, seed=3)
    with bioen_b200.Problem(P["yTilde"]) as p:
        with pytest.raises(RuntimeError, match="log-weights data not set"):
            p.theta_scan([1.0, 2.0])
        p.set_logw(P["G"], P["YTilde"], 1.0)
        with pytest.raises(RuntimeError, match="1..32"):
            p.theta_scan(np.ones(33))
        # invalid liblbfgs parameters: every problem reports the parameter code, nothing is evaluated
        X, fmin, codes, info = p.theta_scan([1.0, 2.0, 3.0], delta=-1.0)
        assert list(codes) == [-1015] * 3 and info["rounds"] == 0
        # a start point that already satisfies the convergence test
        xo, fo, co, _ = p.opt_lbfgs(P["GInit"], epsilon=1e-10, delta=0.0, past=0)
        X, fmin, codes, info = p.theta_scan([1.0], x0=xo, epsilon=1e-3)
        assert codes[0] == 2 and rel(fmin[0], fo) < 1e-12
    # more theta values than one batch holds: find_optimum_series chunks by 32
    cfg = optimize.minimize.Parameters("lbfgs")
    cfg["verbose"] = False
    thetas = np.geomspace(100.0, 1.0, 35)
    out = optimize.log_weights.find_optimum_series(P["GInit"], P["G"], P["y"], P["yTilde"], P["YTilde"], thetas, cfg)
    assert len(out) == 35
    f_final = np.array([o[4] for o in out])
    assert np.all(np.diff(f_final) < 1e-9)          # the optimum decreases with theta
    for q in (2, 33):       # one plane of each chunk against the oracle's liblbfgs restatement
        r = oracle.lbfgs(lambda v: oracle.logw_fg(v, P["G"], P["yTilde"], P["YTilde"], thetas[q]), P["GInit"])
        assert rel(out[q][4], r["fx"]) < (1e-8 if r["iterations"] < 150 else 1e-4), (q, out[q][4], r["fx"])


@pytest.mark.parametrize("M,N,K", [(28, 5001, 7), (300, 4000, 16), (1000, 3001, 32), (5, 17, 3)])
def test_theta_scan_forces_matches_single_runs(oracle, M, N, K):
    """Batched forces scan (four tensor-core GEMMs per evaluation) against the single-problem device L-BFGS and
    the oracle's liblbfgs restatement on identical inputs."""
    import bioen_b200
    from bioen_b200.problem import FORCES
    P = oracle.synthetic_problem(M, N, seed=M + N)
    rng = np.random.default_rng(K)
    w0 = rng.random(N) + 0.2
    w0 /= w0.sum()
    thetas = np.geomspace(300.0, 3.0, K)
    with bioen_b200.Problem(P["yTilde"]) as p:
        p.set_forces(w0, P["YTilde"], 1.0)
        for ls in (2, 0):
            X, fmin, codes, info = p.theta_scan(thetas, method=FORCES, linesearch=ls)
            assert X.shape == (K, M)
            for q in sorted({0, K // 2, K - 1}):
                p.set_theta(thetas[q])
                x1, f1, c1, i1 = p.opt_lbfgs(np.zeros(M), linesearch=ls)
                # Runs that end on liblbfgs' progress rule ((f[k-10] - f[k]) / f[k] < delta = 1e-6) stop somewhere on
                # a slow tail, and WHERE depends on the last bits of the trajectory: measured on the 1000 x 3001
                # problem at theta = 3, the batched scan stops after 876 iterations at 380.0918, the single run
                # after 646 at 380.1745 (2.2e-4 apart, both code 1) -- the tail still gains ~1e-6 per 10 iterations.
                its = max(i1["iterations"], int(info["iterations"][q]))
                tol = 1e-8 if its < 50 else 1e-6 if its < 150 else 1e-4 if its < 500 else 1e-3
                # At large theta the forces problem converges to rounding level, where liblbfgs' line search
                # fails or succeeds on the last bits of f (-998 / -1001 vs 0; the reference behaves the same,
                # SURVEY.md section 7): then only the end point is compared.
                ls_noise = {-998, -1001, -1000, -999, -996}
                if codes[q] not in ls_noise and c1 not in ls_noise:
                    assert codes[q] == c1, (q, ls, codes[q], c1)
                assert rel(fmin[q], f1) < tol, (q, ls, fmin[q], f1, info["iterations"][q], i1)
                if codes[q] >= 0:
                    fo, _ = oracle.forces_fg(X[q], w0, P["yTilde"], P["YTilde"], thetas[q])
                    assert rel(fo, fmin[q]) < 1e-11
            r = oracle.lbfgs(lambda v: oracle.forces_fg(v, w0, P["yTilde"], P["YTilde"], thetas[K - 1]), np.zeros(M),
                             linesearch=ls)
            assert rel(fmin[K - 1], r["fx"]) < (1e-8 if r["iterations"] < 150 else 1e-4)


def test_minimiser_bit_reproducibility():
    """The reference's test_{logw,forces}_reproducibility.py: GSL bfgs2 repeated many times must give the same
    fmin and x to the last bit (its slow/reproducible OpenMP mode).  Device reductions are fixed-order, so the
    same holds here for every minimiser."""
    import bioen_b200
    for name in ("data_potra_part_2_logw_M205xN10", "data_forces_M64xN64"):
        d = load_golden(name)
        with bioen_b200.Problem(d["yTilde"]) as p:
            x0 = _setup(p, d)
            x_ref, f_ref, c_ref, _ = p.opt_gsl(x0)
            xl_ref, fl_ref, cl_ref, _ = p.opt_lbfgs(x0)
            for _ in range(40):
                x, f, c, _ = p.opt_gsl(x0)
                assert f == f_ref and c == c_ref and np.array_equal(x, x_ref)
                x, f, c, _ = p.opt_lbfgs(x0)
                assert f == fl_ref and c == cl_ref and np.array_equal(x, xl_ref)


def test_lazy_gradient_is_bit_identical(oracle):
    """BIOEN_B200_OPT_LAZY_GRADIENT: the minimisers skip (backtracking trials that fail the sufficient-decrease
    test) or defer (GSL's f-then-df on one point) the gradient half of an evaluation.  liblbfgs / GSL never read
    what is skipped, so end point, objective, code and evaluation counts must not move by a bit."""
    import bioen_b200
    skipped, continued = 0, [0] * 5
    for (M, N, theta) in ((100, 20000, 10.0), (50, 20000, 1.0), (300, 3001, 3.0)):
        P = oracle.synthetic_problem(M, N, seed=12345)
        with bioen_b200.Problem(P["yTilde"]) as p:
            p.set_option(8, 0)     # (the L-BFGS driver does not split evaluations on the slice kernel: nothing to gain there)
            for method, setter, x0 in (("logw", lambda: p.set_logw(P["G"], P["YTilde"], theta), P["GInit"]),
                                       ("forces", lambda: p.set_forces(P["w0"], P["YTilde"], theta),
                                        P["forces_init"])):
                setter()
                for ls in (1, 2, 3):
                    p.set_option(3, 1)
                    x1, f1, c1, i1 = p.opt_lbfgs(x0, linesearch=ls, max_iterations=60)
                    p.set_option(3, 0)
                    x0_, f0, c0, i0 = p.opt_lbfgs(x0, linesearch=ls, max_iterations=60)
                    assert c1 == c0 and f1 == f0 and np.array_equal(x1, x0_), (method, M, N, ls)
                    assert i1["iterations"] == i0["iterations"] and i1["evaluations"] == i0["evaluations"]
                    assert i0["gradients_skipped"] == 0
                    skipped += i1["gradients_skipped"]
                for alg in range(5):     # conjugate_fr, conjugate_pr, bfgs2, bfgs, steepest_descent
                    p.set_option(3, 1)
                    x1, f1, c1, i1 = p.opt_gsl(x0, algorithm=alg, max_iterations=25)
                    p.set_option(3, 0)
                    x0_, f0, c0, i0 = p.opt_gsl(x0, algorithm=alg, max_iterations=25)
                    assert c1 == c0 and f1 == f0 and np.array_equal(x1, x0_), (method, M, N, "gsl", alg)
                    assert i1["gradient_evaluations"] == i0["gradient_evaluations"]
                    assert i1["f_only_evaluations"] == i0["f_only_evaluations"] and i0["gradient_half_only"] == 0
                    continued[alg] += i1["gradient_half_only"]
                p.set_option(3, 1)
    # the short cuts were actually taken (steepest descent only when one of its steps was rejected)
    assert skipped > 0 and all(c > 0 for c in continued[:4]), (skipped, continued)


def test_small_update_kernel_and_speculative_trial(oracle):
    """BIOEN_B200_OPT_LBFGS_SMALL (9): the (s, y) pair and the two-loop recursion as ONE single-CTA kernel for
    n <= 1024 -- bit-identical to the 15-kernel path up to 256 variables (one block there as well), same end point
    beyond.  BIOEN_B200_OPT_LBFGS_SPECULATIVE (10): the first trial of a line search enqueued before the initial
    slope is fetched -- must not move a bit or an evaluation count, for any n."""
    import bioen_b200
    OPT_SMALL, OPT_SPEC = 9, 10
    cases = []
    d = load_golden("data_forces_M64xN64")
    cases.append(("forces 64", d["yTilde"], lambda p: p.set_forces(d["w0"], d["YTilde"], d["theta"]),
                  d["forces_init"].ravel(), True))
    d2 = load_golden("data_potra_part_1_logw_M808xN80")
    cases.append(("logw 80", d2["yTilde"], lambda p: p.set_logw(d2["G"], d2["YTilde"], d2["theta"]),
                  d2["GInit"].ravel(), True))
    d3 = load_golden("data_deer_test_forces_M808xN10")
    cases.append(("forces 808", d3["yTilde"], lambda p: p.set_forces(d3["w0"], d3["YTilde"], d3["theta"]),
                  d3["forces_init"].ravel(), False))
    P = oracle.synthetic_problem(1000, 777, seed=5)
    cases.append(("forces 1000", P["yTilde"], lambda p: p.set_forces(P["w0"], P["YTilde"], 10.0),
                  P["forces_init"], False))
    P2 = oracle.synthetic_problem(28, 5001, seed=6)
    cases.append(("logw 5001 (speculative only)", P2["yTilde"], lambda p: p.set_logw(P2["G"], P2["YTilde"], 10.0),
                  P2["GInit"], True))
    for name, yT, setter, x0, bitwise in cases:
        with bioen_b200.Problem(yT) as p:
            setter(p)
            for ls in (0, 2):
                res = {}
                for small, spec in ((0, 0), (0, 1), (1, 0), (1, 1)):
                    p.set_option(OPT_SMALL, small)
                    p.set_option(OPT_SPEC, spec)
                    k0 = p.kernels_launched()
                    res[small, spec] = p.opt_lbfgs(x0, linesearch=ls, max_iterations=50) + (p.kernels_launched() - k0,)
                for small in (0, 1):      # speculative trial: identical bits and counts
                    a, b = res[small, 0], res[small, 1]
                    assert a[2] == b[2] and a[1] == b[1] and np.array_equal(a[0], b[0]), (name, ls, small)
                    assert a[3] == b[3], (name, ls, small)
                a, b = res[0, 1], res[1, 1]
                if x0.size <= 1024:
                    assert b[4] < a[4], (name, "fewer launches", a[4], b[4])
                if bitwise:
                    assert a[2] == b[2] and a[1] == b[1] and np.array_equal(a[0], b[0]), (name, ls)
                else:
                    assert a[2] == b[2] and rel(b[1], a[1]) < 1e-8, (name, ls, a[1], b[1], a[2], b[2])


def test_zero_copy_scalar_fetch_is_transparent(oracle):
    """BIOEN_B200_OPT_FETCH_ZEROCOPY (12): the scalar file reaches the host through a one-warp kernel's stores into
    page-locked memory instead of a copy-engine transfer.  Same values: every minimiser result is bit-identical."""
    import bioen_b200
    P = oracle.synthetic_problem(40, 6001, seed=3)
    with bioen_b200.Problem(P["yTilde"]) as p:
        for setter, x0 in ((lambda: p.set_logw(P["G"], P["YTilde"], 5.0), P["GInit"]),
                           (lambda: p.set_forces(P["w0"], P["YTilde"], 5.0), P["forces_init"])):
            setter()
            out = []
            for zc in (1, 0, 1):
                p.set_option(12, zc)
                a = p.opt_lbfgs(x0, max_iterations=30)
                b = p.opt_gsl(x0, max_iterations=10)
                f, g = p.objective_and_gradient(np.asarray(x0).ravel() + 0.01)
                out.append((a, b, f, g))
            for o in out[1:]:
                assert o[0][1] == out[0][0][1] and o[0][2] == out[0][0][2] and np.array_equal(o[0][0], out[0][0][0])
                assert o[1][1] == out[0][1][1] and o[1][2] == out[0][1][2] and np.array_equal(o[1][0], out[0][1][0])
                assert o[2] == out[0][2] and np.array_equal(o[3], out[0][3])


def test_reused_context_starts_with_default_options():
    """The options of bioen_b200_set_option live in one record of the context.  A small context is kept for reuse
    when its Problem closes and handed to the next Problem of the same shape: that one must start with every option
    at its default again (bioen_b200_query 10: bitmask of the options that differ from their defaults)."""
    import bioen_b200
    non_default = {1: 0, 3: 0, 4: 0, 5: 0, 6: 1, 8: 0, 9: 0, 10: 0, 12: 0}
    d = load_golden("data_forces_M64xN64")
    with bioen_b200.Problem(d["yTilde"]) as p:
        assert p.query(10) == 0
        for option, value in non_default.items():
            p.set_option(option, value)
        assert p.query(10) == sum(1 << option for option in non_default)
        device = p.device
    with bioen_b200.Problem(d["yTilde"], device=device) as q:
        assert q.query(10) == 0
