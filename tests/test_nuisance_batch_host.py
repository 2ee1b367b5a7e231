"""CPU: the host side of the batched theta series with nuisance-parameter refits (nuisance.theta_series): the
per-problem row-affine planes it hands to the batched engine, the base averages it recovers from the resident
averages, its history and its chunking into batches of 32.  The device is replaced by a NumPy stand-in whose
batch_minimize records the planes it is given; tests/test_gpu_nuisance_batch.py runs the series on the GPU."""
import numpy as np
import pytest

from conftest import load_golden


def _multi_blocks(NU, rng, m_rows=(40, 30, 25, 10, 15)):
    """two DEER blocks, one scattering block, fixed rows and rows outside every block"""
    r = np.cumsum((0,) + m_rows)
    blk = []
    for q, (kind, v) in enumerate(((NU.DEER, 0.3), (NU.DEER, 0.45), (NU.SCATTERING, 2e-4), (NU.FIXED, None))):
        n = r[q + 1] - r[q]
        blk.append(NU.Block(kind, r[q], r[q + 1], err=rng.random(n) + 0.5,
                            exp_fit=None if kind == NU.FIXED else rng.random(n), value=v, name="b%d" % q))
    return blk, int(r[-1])


def _at(NU, blocks, vals):
    """copies of the blocks at the given values"""
    return [NU.Block(b.kind, b.start, b.stop, err=b.err, exp_fit=b.exp_fit, value=vals.get(b.name, b.value),
                     name=b.name) for b in blocks]


class BatchHost:
    """Problem's attributes and batch_minimize as theta_series uses them.  Each problem's 'minimisation' returns
    weights fixed by its theta; the averages are those of the resident matrix, as on the device."""

    def __init__(self, yTilde, fail=()):
        self.y = np.array(yTilde, dtype=np.float64)
        self.m, self.n = self.y.shape
        self.method = 0
        self.calls = []
        self.fail = set(fail)

    def average(self, w):
        return self.y @ np.asarray(w, dtype=np.float64).ravel()

    def weights(self, theta):
        w = 1.0 + np.cos(np.arange(self.n) * (1.0 + theta))
        return w / w.sum()

    def batch_minimize(self, thetas, x0=None, row_scale=None, row_offset=None, **cfg):
        thetas = np.asarray(thetas)
        self.calls.append(dict(thetas=thetas.copy(), a=row_scale.copy(), b=row_offset.copy(), cfg=cfg))
        W = np.stack([self.weights(t) for t in thetas])
        codes = np.array([-998 if float(t) in self.fail else 0 for t in thetas])
        return (np.log(W), thetas * 0.5, codes, dict(averages=W @ self.y.T))


def test_planes_compose_the_resident_transform_with_each_problems_values():
    from bioen_b200 import nuisance as NU
    rng = np.random.default_rng(1)
    blocks, M = _multi_blocks(NU, rng)
    base = rng.random((M, 23)) + 0.1
    resident = NU.proc_sim(base, blocks)
    ref = NU.NuisanceRefit(BatchHost(resident), blocks)
    for _ in range(5):
        vals = {"b0": rng.random(), "b1": rng.random(), "b2": 1e-4 * rng.random()}
        a, c, s, o = ref.relative(vals)
        want = NU.proc_sim(base, _at(NU, blocks, vals))
        got = a[:, None] * resident + c[:, None]
        assert np.max(np.abs(got - want) / np.abs(want)) < 1e-14
        assert np.max(np.abs(s[:, None] * base + o[:, None] - want) / np.abs(want)) < 1e-14
    # the resident values themselves give the identity exactly
    a, c, _, _ = ref.relative({})
    assert np.array_equal(a, np.ones(M)) and np.array_equal(c, np.zeros(M))
    # base averages from resident averages
    w = rng.random(23)
    w /= w.sum()
    assert np.max(np.abs(ref.base_from_averages(resident @ w, w.sum()) - base @ w) / (base @ w)) < 1e-13


def test_history_shapes_chunking_and_failures():
    from bioen_b200 import nuisance as NU
    from bioen_b200.replicates import NOT_RUN
    rng = np.random.default_rng(2)
    blocks, M = _multi_blocks(NU, rng)
    base = rng.random((M, 17)) + 0.1
    thetas = np.linspace(0.5, 20.0, 40)
    prob = BatchHost(NU.proc_sim(base, blocks), fail={float(thetas[3]), float(thetas[35])})
    start = {"b0": np.linspace(0.2, 0.6, 40), "b2": 3e-4}
    out = NU.theta_series(prob, blocks, thetas, 3, values=start, max_iterations=50)
    assert out["x"].shape == (3, 40, 17) and out["fmin"].shape == (3, 40) and out["codes"].shape == (3, 40)
    assert set(out["values"]) == {"b0", "b1", "b2"}
    assert all(v.shape == (4, 40) for v in out["values"].values())
    assert np.array_equal(out["values"]["b0"][0], start["b0"])
    assert np.all(out["values"]["b1"][0] == 0.45) and np.all(out["values"]["b2"][0] == 3e-4)
    # chunks of 32 and 8; the failed problems leave the batch after their first round
    assert [c["thetas"].size for c in prob.calls] == [32, 31, 31, 8, 7, 7]
    assert all(c["cfg"] == dict(max_iterations=50) for c in prob.calls)
    for t in (3, 35):
        assert out["codes"][0, t] == -998 and np.all(out["codes"][1:, t] == NOT_RUN)
        assert np.isfinite(out["fmin"][0, t]) and np.all(np.isnan(out["fmin"][1:, t]))
        assert np.all(np.isnan(out["x"][1:, t]))
        assert all(np.all(np.isnan(v[1:, t])) for v in out["values"].values())
    ok = np.ones(40, bool)
    ok[[3, 35]] = False
    assert np.all(out["codes"][:, ok] == 0) and all(np.all(np.isfinite(v[:, ok])) for v in out["values"].values())
    # every round's planes are the transform of the values that round started from, and each refit is the
    # NuisanceRefit one against the problem's weights
    first = prob.calls[0]
    for q in (0, 17, 31):
        vals = {name: h[0, q] for name, h in out["values"].items()}
        a, c, _, _ = NU.NuisanceRefit(BatchHost(prob.y), blocks).relative(vals)
        assert np.array_equal(first["a"][q], a) and np.array_equal(first["b"][q], c)
    for q in (0, 39):
        prob_k = BatchHost(prob.y)
        for it in range(3):
            vals = {name: h[it, q] for name, h in out["values"].items()}
            bl = _at(NU, blocks, vals)
            nr = NU.NuisanceRefit(BatchHost(NU.proc_sim(base, bl)), bl)
            fitted = nr.fit(prob_k.weights(thetas[q]))
            for name, v in fitted.items():
                assert abs(v / out["values"][name][it + 1, q] - 1.0) < 1e-8, (q, it, name)


def test_the_resident_matrix_is_not_touched_and_inputs_are_checked():
    from bioen_b200 import nuisance as NU
    d = load_golden("nuisance_deer")
    blocks = [NU.Block("deer", 0, d["raw"].shape[0], err=d["err"], exp_fit=d["exp_fit"], value=0.3, name="deer")]
    y0 = NU.proc_sim(NU.base_matrix(d["raw"], d["err"]), blocks)
    prob = BatchHost(y0)
    prob.affine_rows = None          # a call would fail
    out = NU.theta_series(prob, blocks, [10.0, 1.0], 2, values={"deer": [0.3, 0.42]})
    assert np.array_equal(prob.y, y0) and out["values"]["deer"].shape == (3, 2)
    with pytest.raises(ValueError, match="unknown blocks"):
        NU.theta_series(prob, blocks, [1.0], 1, values={"nope": 1.0})
    with pytest.raises(ValueError, match="one entry per theta"):
        NU.theta_series(prob, blocks, [1.0, 2.0], 1, values={"deer": [0.1, 0.2, 0.3]})
    with pytest.raises(ValueError, match="iterations"):
        NU.theta_series(prob, blocks, [1.0], 0)
    with pytest.raises(ValueError, match="x0"):
        NU.theta_series(prob, blocks, [1.0], 1, x0=np.zeros(3))
