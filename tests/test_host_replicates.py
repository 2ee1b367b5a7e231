"""CPU: the host side of bioen_b200.replicates -- resampling, fold generation, chunking and argument checks -- on a
stand-in problem that records the batches it is asked to minimise instead of running them on a device."""
import numpy as np
import pytest

from bioen_b200 import replicates
from bioen_b200.problem import FORCES, LOGW


class RecordingProblem:
    """The attributes and the batch_minimize signature replicates.py uses; returns the inputs it was given so that
    tests can see them, and counts its calls."""

    def __init__(self, m, n, method, fail=()):
        self.m, self.n, self.method = m, n, method
        rng = np.random.default_rng(m * n)
        self.YTilde = rng.standard_normal(m)
        self.w0 = None
        if method == FORCES:
            self.w0 = rng.random(n) + 0.1
            self.w0 /= self.w0.sum()
        self.calls = []
        self.fail = set(fail)     # global replicate indices that report a failed line search

    def batch_minimize(self, thetas, x0=None, YTilde=None, row_weights=None, w0=None, **cfg):
        thetas = np.asarray(thetas, dtype=float)
        K = thetas.size
        r0 = sum(len(c["thetas"]) for c in self.calls)
        self.calls.append(dict(thetas=thetas, x0=x0, YTilde=YTilde, row_weights=row_weights, w0=w0, cfg=cfg))
        n = self.m if self.method == FORCES else self.n
        codes = np.array([-1001 if r0 + k in self.fail else 0 for k in range(K)])
        avg = np.tile(np.arange(self.m, dtype=float), (K, 1)) + np.arange(K)[:, None]
        return (np.zeros((K, n)), thetas.copy(), codes,
                dict(averages=avg, chi2=np.arange(K, dtype=float), kl=np.ones(K)))


class NoDevice(RecordingProblem):
    def batch_minimize(self, *a, **k):
        raise AssertionError("argument checks must come before any device call")


@pytest.mark.parametrize("resample,method", [("observables", LOGW), ("noise", LOGW), ("observables", FORCES),
                                             ("noise", FORCES), ("structures", FORCES)])
def test_bootstrap_is_deterministic_and_chunked(resample, method):
    p1, p2, p3 = (RecordingProblem(37, 101, method) for _ in range(3))
    a = replicates.bootstrap(p1, 70, resample, 10.0, seed=5, max_iterations=7)
    b = replicates.bootstrap(p2, 70, resample, 10.0, seed=5, max_iterations=7)
    c = replicates.bootstrap(p3, 70, resample, 10.0, seed=6, max_iterations=7)
    key = "noise" if resample == "noise" else "counts"
    assert np.array_equal(a[key], b[key]) and not np.array_equal(a[key], c[key])
    assert [len(cl["thetas"]) for cl in p1.calls] == [32, 32, 6]
    assert all(cl["cfg"] == dict(max_iterations=7) for cl in p1.calls)
    assert all(np.all(cl["thetas"] == 10.0) for cl in p1.calls)
    for k1, k2 in zip(p1.calls, p2.calls):
        for name in ("YTilde", "row_weights", "w0"):
            assert (k1[name] is None) == (k2[name] is None)
            if k1[name] is not None:
                assert np.array_equal(k1[name], k2[name])
    assert a["averages"].shape == (70, 37) and a["fmin"].shape == (70,) and a["codes"].shape == (70,)


def test_observable_counts_sum_to_M_and_become_row_weights():
    p = RecordingProblem(37, 101, LOGW)
    out = replicates.bootstrap(p, 40, "observables", 1.0, seed=1)
    assert out["counts"].shape == (40, 37)
    assert np.all(out["counts"].sum(axis=1) == 37) and np.all(out["counts"] >= 0)
    rw = np.concatenate([c["row_weights"] for c in p.calls])
    assert np.array_equal(rw, out["counts"].astype(float))
    assert all(c["YTilde"] is None and c["w0"] is None for c in p.calls)


def test_structure_counts_sum_to_N_and_scale_w0():
    p = RecordingProblem(12, 101, FORCES)
    out = replicates.bootstrap(p, 40, "structures", 1.0, seed=2)
    assert out["counts"].shape == (40, 101) and np.all(out["counts"].sum(axis=1) == 101)
    w0 = np.concatenate([c["w0"] for c in p.calls])
    assert np.all(w0[out["counts"] == 0] == 0.0)
    np.testing.assert_allclose(w0.sum(axis=1), p.w0.sum(), rtol=1e-14)
    for r in range(40):       # w0_r is proportional to w0 * counts_r
        on = out["counts"][r] > 0
        q = w0[r, on] / (p.w0[on] * out["counts"][r, on])
        np.testing.assert_allclose(q, q[0], rtol=1e-14)


def test_noise_has_the_requested_shape_and_shifts_YTilde():
    p = RecordingProblem(37, 101, FORCES)
    out = replicates.bootstrap(p, 33, "noise", 1.0, seed=3)
    assert out["noise"].shape == (33, 37)
    Y = np.concatenate([c["YTilde"] for c in p.calls])
    np.testing.assert_array_equal(Y, p.YTilde + out["noise"])
    assert abs(out["noise"].mean()) < 0.1 and abs(out["noise"].std() - 1.0) < 0.1


def test_failed_replicates_get_nan_statistics_and_keep_their_code():
    p = RecordingProblem(20, 50, LOGW, fail={3, 35})
    out = replicates.bootstrap(p, 40, "observables", 1.0)
    assert out["codes"][3] == -1001 and out["codes"][35] == -1001
    for r in (3, 35):
        assert np.all(np.isnan(out["averages"][r])) and np.isnan(out["chi2"][r]) and np.isnan(out["kl"][r])
    ok = np.setdiff1d(np.arange(40), [3, 35])
    assert np.all(np.isfinite(out["averages"][ok])) and np.all(np.isfinite(out["chi2"][ok]))


def test_folds_partition_the_observables():
    for M, F in ((37, 5), (10, 10), (101, 3)):
        f1 = replicates.fold_assignment(M, F, np.random.default_rng(4))
        f2 = replicates.fold_assignment(M, F, np.random.default_rng(4))
        assert np.array_equal(f1, f2)
        assert f1.shape == (M,) and set(f1) == set(range(F))
        sizes = np.bincount(f1, minlength=F)
        assert sizes.sum() == M and sizes.max() - sizes.min() <= 1


def test_cross_validate_problems_and_held_out_chi2():
    p = RecordingProblem(23, 60, FORCES, fail={7})
    thetas = [100.0, 10.0, 1.0, 0.1, 0.01, 3.0, 30.0]
    out = replicates.cross_validate(p, thetas, folds=5, seed=9)
    again = replicates.cross_validate(RecordingProblem(23, 60, FORCES, fail={7}), thetas, folds=5, seed=9)
    assert np.array_equal(out["fold"], again["fold"])
    assert [len(c["thetas"]) for c in p.calls] == [32, 3]
    th = np.concatenate([c["thetas"] for c in p.calls])
    rw = np.concatenate([c["row_weights"] for c in p.calls])
    assert np.array_equal(th, np.repeat(thetas, 5))
    for q in range(35):
        f = q % 5
        assert np.array_equal(rw[q], (out["fold"] != f).astype(float))
    assert out["held_out_chi2"].shape == (7, 5) and out["codes"].shape == (7, 5)
    for t in range(7):
        for f in range(5):
            if t * 5 + f == 7:
                assert np.isnan(out["held_out_chi2"][t, f]) and out["codes"][t, f] == -1001
                continue
            fold = out["fold"] == f
            want = 0.5 * np.sum((out["averages"][t, f, fold] - p.YTilde[fold]) ** 2)
            assert out["held_out_chi2"][t, f] == pytest.approx(want, rel=1e-14)


def test_arguments_are_checked_before_any_device_call():
    lw, fo = NoDevice(20, 50, LOGW), NoDevice(20, 50, FORCES)
    with pytest.raises(ValueError, match="forces method"):
        replicates.bootstrap(lw, 4, "structures", 1.0)
    with pytest.raises(ValueError, match="resample"):
        replicates.bootstrap(fo, 4, "rows", 1.0)
    for bad in (0, -3, 2.5):
        with pytest.raises(ValueError, match="n_replicates"):
            replicates.bootstrap(fo, bad, "noise", 1.0)
    for bad in (np.nan, -1.0, np.inf):
        with pytest.raises(ValueError, match="theta"):
            replicates.bootstrap(fo, 4, "noise", bad)
    for bad in (1, 21, 2.5):
        with pytest.raises(ValueError, match="folds"):
            replicates.cross_validate(fo, [1.0], folds=bad)
    for bad in ([], [np.nan], [-1.0, 2.0]):
        with pytest.raises(ValueError, match="thetas"):
            replicates.cross_validate(fo, bad)
    unset = NoDevice(20, 50, LOGW)
    unset.method = None
    with pytest.raises(RuntimeError, match="set_logw or set_forces"):
        replicates.bootstrap(unset, 4, "noise", 1.0)
    with pytest.raises(RuntimeError, match="set_logw or set_forces"):
        replicates.cross_validate(unset, [1.0])


def test_structure_draws_without_reference_weight_are_not_run():
    p = RecordingProblem(6, 5, FORCES)
    p.w0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0])       # only structure 0 carries weight
    out = replicates.bootstrap(p, 40, "structures", 1.0, seed=4)
    empty = out["counts"][:, 0] == 0
    assert empty.any() and not empty.all()
    assert np.all(out["codes"][empty] == replicates.NOT_RUN)
    assert np.all(np.isnan(out["fmin"][empty])) and np.all(np.isnan(out["averages"][empty]))
    assert np.all(out["codes"][~empty] == 0)
    sent = np.concatenate([c["w0"] for c in p.calls])
    assert sent.shape[0] == np.count_nonzero(~empty) and np.all(sent.sum(axis=1) > 0)


def test_per_replicate_start_points_follow_their_chunk():
    p = RecordingProblem(8, 30, LOGW)
    X0 = np.arange(40 * 30, dtype=float).reshape(40, 30)
    replicates.bootstrap(p, 40, "noise", 1.0, x0=X0)
    assert np.array_equal(np.concatenate([c["x0"] for c in p.calls]), X0)
    with pytest.raises(ValueError, match="x0"):
        replicates.bootstrap(NoDevice(8, 30, LOGW), 40, "noise", 1.0, x0=np.zeros((39, 30)))
    with pytest.raises(ValueError, match="x0"):
        replicates.cross_validate(NoDevice(8, 30, LOGW), [1.0], folds=2, x0=np.zeros(29))
