"""GPU: every evaluation path against the extended-precision reference (tests/hp_reference.py) at the numerical edges.

The parity tests elsewhere compare with the fp64 oracle to 1e-11 on near-uniform weights, where no stabilising
maximum, rescale or guard is ever exercised.  Here each path -- the stand-alone kernels (narrow, and wide enough for
the column pass's gradient epilogue), the persistent kernel, the shared-memory slice kernel, the fused two-pass forces
kernels, structure-major-only mode, fp32 storage, the batched planes and the N-sharded path -- is run on the regimes of
tests/edge_regimes.py (concentrated weights with the argmax in the first tile, the ragged last tile or a slice / rank
other than the first; forces spanning hundreds to thousands; zero, contiguous-zero and subnormal prior weights;
theta = 0, 1e-8, 1e8; gauge offsets; large row offsets; exact ties), and every output -- f of the combined and of the
objective-only launch, each gradient component of the combined launch and of the gradient continuation, each weight
-- must satisfy  |gpu - ref| <= C u scale (+ a few 2^-1074 for weights and gradients that may be subnormal).

Every case asserts that the intended path ran (query counters and the pass kernel's name), not a fallback.
"""
import os
from collections import OrderedDict

import numpy as np
import pytest

import edge_regimes as R
import hp_reference as H

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not H.available(), reason="np.longdouble is not the x86-64 80-bit format")]

os.environ.setdefault("BIOEN_B200_P2P_TIMEOUT_S", "30")   # a rank that never arrives poisons the result after 30 s

# One constant for every path and regime.  The benign regime (the inputs of the parity tests) sets the baseline: its
# largest ratio |gpu - ref| / (u scale) is printed by test_zz_report, and C must be at least 4x that.  Measured on a
# B200: benign 0.69 (stand-alone kernels and slice kernel), edge regimes 1.89 at most (fp32 storage); every path's
# kernels reduce in a fixed order, so the ratios do not change from run to run.  C = 16 is 23x the benign and 8x the
# largest edge ratio; the mutants of tests/test_hp_reference.py miss by more than 1024 (gradients) and 102400 (weights).
C = 16
LOGW, FORCES = 0, 1
OPT_FUSED, OPT_PERSISTENT, OPT_FP32, OPT_SLICE = 1, 5, 7, 8

PATHS = OrderedDict([
    # path: (shapes, methods).  5 x 80001 is wide (>= 4 x 148 column blocks, odd N) -> stream_colgrad_kernel
    ("standalone", ([(5, 80001), (1000, 777), (3, 5)], (LOGW, FORCES))),
    ("persistent", ([(28, 50001), (300, 4003)], (LOGW, FORCES))),
    ("slice", ([(28, 50001), (1000, 777), (3, 5)], (LOGW, FORCES))),
    ("fused", ([(300, 4003), (1000, 777)], (FORCES,))),
    ("structure_major_only", ([(300, 4003)], (FORCES,))),
    ("fp32", ([(28, 50001), (5, 80001)], (LOGW, FORCES))),
    ("sharded2", ([(28, 50001)], (LOGW, FORCES))),
    ("sharded3", ([(300, 4003), (1000, 777)], (LOGW, FORCES))),
])


def _cases():
    out = []
    for path, (shapes, methods) in PATHS.items():
        for M, N in shapes:
            for method in methods:
                for regime in (R.LOGW_REGIMES if method == LOGW else R.FORCES_REGIMES):
                    out.append(pytest.param(path, M, N, method, regime,
                                            id="%s-%dx%d-%s-%s" % (path, M, N, ("logw", "forces")[method], regime)))
    return out


WORST = {}            # (path, benign?) -> largest ratio seen
_REFS = {}


def _record(path, regime, r):
    key = (path, regime == "benign")
    WORST[key] = max(WORST.get(key, 0.0), max(r.values()))


def _reference(method, regime, M, N, fp32=False, c=None, x=None, a=None, theta=None, variant=None):
    if x is None:
        variant, x, a, theta = R.case(method, regime, M, N)
    key = (method, regime, M, N, fp32, variant) if c is None else None
    if key is not None and key in _REFS:
        return _REFS[key]
    y, Y = R.matrix(variant, M, N)
    if fp32:
        y = y.astype(np.float32).astype(np.float64)
    ref = (H.logw if method == LOGW else H.forces)(x, a, y, Y, theta, c=c)
    if key is not None:
        _REFS[key] = ref
    return ref


class _Cache:
    """the last few device problems, keyed by (path, shape, matrix variant); older ones are closed"""
    def __init__(self, size=4):
        self.size, self.items = size, OrderedDict()

    def get(self, key, make):
        if key in self.items:
            self.items.move_to_end(key)
            return self.items[key]
        while len(self.items) >= self.size:
            self.items.popitem(last=False)[1].close()
        self.items[key] = make()
        return self.items[key]

    def close(self):
        while self.items:
            self.items.popitem()[1].close()


@pytest.fixture(scope="module")
def cache():
    c = _Cache()
    yield c
    c.close()


def _make(path, y, world=1):
    import bioen_b200
    from bioen_b200 import dist as D
    if world > 1:
        return D.LocalGroup(y, world)
    p = bioen_b200.Problem(y, structure_major_only=(path == "structure_major_only"))
    if path == "standalone" or path == "fp32":
        p.set_option(OPT_PERSISTENT, 0)
        p.set_option(OPT_FUSED, 0)
    elif path == "persistent":
        p.set_option(OPT_PERSISTENT, 1)
        p.set_option(OPT_SLICE, 0)
        p.set_option(OPT_FUSED, 0)
    elif path == "slice":
        p.set_option(OPT_PERSISTENT, 1)
        p.set_option(OPT_SLICE, 1)
    elif path == "fused":
        p.set_option(OPT_PERSISTENT, 0)
        p.set_option(OPT_FUSED, 1)
    if path == "fp32":
        p.set_option(OPT_FP32, 1)
    return p


def _assert_path(p, path, method, n5, n6):
    """the path that evaluated is the one the case names (n5 / n6: one-launch / slice launches before the case)"""
    d5, d6 = p.query(5) - n5, p.query(6) - n6
    name = p.pass_kernel_name(method)
    if path in ("standalone", "fp32"):
        assert p.query(3) == 0 and p.query(7) == 0 and d5 == 0 and name == "stream_pass_kernel", (path, name)
        assert method == LOGW or p.query(0) == 0
        assert p.query(4) == (4 if path == "fp32" else 8)
    elif path == "persistent":
        assert p.query(3) == 1 and p.query(7) == 0 and d5 > 0 and d6 == 0 and name == "persistent_eval_kernel"
    elif path == "slice":
        assert p.query(7) == 1 and d6 > 0 and d6 == d5 and name == "slice_eval_kernel"
    elif path in ("fused", "structure_major_only"):
        assert p.query(0) == 1 and p.query(3) == 0 and p.query(7) == 0 and d5 == 0 and name == "fused_team_pass"
        assert p.query(9) == (1 if path == "structure_major_only" else 0)


def _run_single(p, path, method, x, a, Y, theta):
    n5, n6 = p.query(5), p.query(6)
    if method == LOGW:
        p.set_logw(a, Y, theta)
    else:
        p.set_forces(a, Y, theta)
    f, g = p.objective_and_gradient(x)
    fo = p.objective(x)
    g2 = p.gradient(x)                    # the gradient half of the point just probed
    w, _ = p.weights(x)
    _assert_path(p, path, method, n5, n6)
    return dict(f=[f, fo], grad=[g, g2], w=[w])


def _run_sharded(grp, method, x, a, Y, theta):
    assert grp.call(lambda r, p, lo, hi: p.comm_mode()) == ["p2p"] * grp.world
    xs = (lambda lo, hi: x[lo:hi]) if method == LOGW else (lambda lo, hi: x)
    if method == LOGW:
        grp.call(lambda r, p, lo, hi: p.set_logw(a[lo:hi], Y, theta))
    else:
        grp.call(lambda r, p, lo, hi: p.set_forces(a[lo:hi], Y, theta))
    assert all(e > 0 for e in grp.call(lambda r, p, lo, hi: p.exchanges_per_eval()))
    res = grp.call(lambda r, p, lo, hi: p.objective_and_gradient(xs(lo, hi)))
    split = grp.call(lambda r, p, lo, hi: (p.objective(xs(lo, hi)), p.gradient(xs(lo, hi))))
    ws = grp.call(lambda r, p, lo, hi: p.weights(xs(lo, hi))[0])
    fs = [f for f, _ in res] + [f for f, _ in split]
    assert all(f == fs[0] or not np.isfinite(fs[0]) for f in fs[:grp.world]), fs   # every rank gets the same f
    if method == LOGW:
        grads = [grp.gather([g for _, g in res]), grp.gather([g for _, g in split])]
    else:
        grads = [g for _, g in res] + [g for _, g in split]
    return dict(f=fs, grad=grads, w=[grp.gather(ws)])


def _check(path, regime, ref, got):
    r = {}
    for k, vals in got.items():
        for v in vals:
            r[k] = max(r.get(k, 0.0), H.ratio(np.atleast_1d(v), np.atleast_1d(ref[k]), np.atleast_1d(ref["s_" + k]),
                                              H.FLOORS.get(k, 0.0)))
    _record(path, regime, r)
    assert max(r.values()) <= C, (path, regime, {k: "%.3g" % v for k, v in r.items()})
    if regime.startswith("gauge"):
        # f does not depend on a common offset of g and G, and the gradient sums to 0
        for g in got["grad"]:
            assert abs(np.sum(g)) <= C * H.U * float(np.sum(ref["s_grad"])), (path, regime, np.sum(g))


@pytest.mark.parametrize("path,M,N,method,regime", _cases())
def test_path_at_edge(cache, path, M, N, method, regime):
    variant, x, a, theta = R.case(method, regime, M, N)
    y, Y = R.matrix(variant, M, N)
    world = int(path[-1]) if path.startswith("sharded") else 1
    obj = cache.get((path, M, N, variant), lambda: _make(path, y, world))
    if world > 1:
        got = _run_sharded(obj, method, x, a, Y, theta)
    else:
        got = _run_single(obj, path, method, x, a, Y, theta)
    _check(path, regime, _reference(method, regime, M, N, fp32=(path == "fp32")), got)


def _row_weights(rng, K, M):
    Cw = np.ones((K, M))
    for k in range(K):
        if k % 3 == 1:
            Cw[k] = rng.multinomial(M, np.full(M, 1.0 / M))
        elif k % 3 == 2:
            Cw[k] = 2.0 * rng.random(M)
            Cw[k, rng.random(M) < 0.25] = 0.0
    return Cw


@pytest.mark.parametrize("M,N", [(300, 4003), (1000, 777)])
@pytest.mark.parametrize("method", [LOGW, FORCES])
def test_batch_evaluate_at_edges(method, M, N):
    """The batched planes (batch_evaluate, the theta scan's engine): one batch holds every regime of the method, one
    per plane, with per-plane theta, w0 (forces) and observable weights; f, each gradient component, averages, chi^2
    and KL of every plane under the same rule.  Log-weights planes share G, so the gauge planes are plain offsets of
    g there; the forces planes run on the matrix whose argmax column lies in the middle."""
    import bioen_b200
    regimes = R.LOGW_REGIMES if method == LOGW else R.FORCES_REGIMES
    variant = "base" if method == LOGW else "top@mid"
    y, Y = R.matrix(variant, M, N)
    cases = [R.case(method, reg, M, N) for reg in regimes]
    K = len(cases)
    X = np.stack([c[1] for c in cases])
    thetas = np.array([c[3] for c in cases])
    Cw = _row_weights(np.random.default_rng(M + N + method), K, M)
    G = cases[0][2] if method == LOGW else None
    W0 = np.stack([c[2] for c in cases]) if method == FORCES else None
    with bioen_b200.Problem(y) as p:
        if method == LOGW:
            p.set_logw(G, Y, 1.0)
        else:
            p.set_forces(W0[0], Y, 1.0)
        f, g, info = p.batch_evaluate(X, thetas, row_weights=Cw, w0=W0)
        fo, _, info_o = p.batch_evaluate(X, thetas, row_weights=Cw, w0=W0, gradient=False)
    for k, reg in enumerate(regimes):
        ref = _reference(method, reg, M, N, c=Cw[k], x=X[k], a=G if method == LOGW else W0[k], theta=thetas[k],
                         variant=variant)
        got = dict(f=[f[k], fo[k]], grad=[g[k]], avg=[info["averages"][k], info_o["averages"][k]],
                   chi2=[info["chi2"][k]], kl=[info["kl"][k]])
        _check("batch", reg, ref, got)


def test_zz_report():
    """the largest |gpu - ref| / (u scale) per path, benign regime and edge regimes (run with -s to see it)"""
    print("\nlargest |gpu - ref| / (u * scale), C = %d" % C)
    for path in list(PATHS) + ["batch"]:
        b, e = WORST.get((path, True)), WORST.get((path, False))
        if b is not None or e is not None:
            print("  %-22s benign %8.3g   edge regimes %8.3g" % (path, b or 0.0, e or 0.0))
    benign = [v for (path, is_b), v in WORST.items() if is_b]
    if benign:
        assert C >= 4 * max(benign), "C must be at least 4x the largest benign ratio"
