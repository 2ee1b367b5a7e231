"""CPU: the product's liblbfgs line-search state machine (csrc/lbfgs.cuh LineSearchState -- the code the device
L-BFGS and the theta scan run on the host side) against the oracle's restatement of lbfgs.c:645-1001, on 1-D
functions, through the host-only C hook bioen_b200_selftest_linesearch.  No GPU involved."""
import ctypes as C
import math

import numpy as np
import pytest

from bioen_b200 import _lib

PHI = {
    "quadratic": (lambda t: (t - 1.3) ** 2 + 0.5, lambda t: 2 * (t - 1.3)),
    "quartic": (lambda t: (t - 2.0) ** 4 - 3 * t + 7.0, lambda t: 4 * (t - 2.0) ** 3 - 3),
    "exp": (lambda t: math.exp(0.7 * t) - 2.5 * t, lambda t: 0.7 * math.exp(0.7 * t) - 2.5),
    "more_thuente_1": (lambda t: -t / (t * t + 2.0), lambda t: (t * t - 2.0) / (t * t + 2.0) ** 2),
    "wiggly": (lambda t: 0.1 * math.sin(9 * t) + (t - 0.8) ** 2, lambda t: 0.9 * math.cos(9 * t) + 2 * (t - 0.8)),
}


def _oracle_search(oracle, name, ls, stp0, over):
    phi, dphi = PHI[name]
    p = dict(oracle.LBFGS_BIOEN_DEFAULTS)
    p.update(over)
    p["linesearch"] = ls

    def evaluate(x, g):
        g[0] = dphi(float(x[0]))
        return phi(float(x[0]))

    x, g, xp, s = np.zeros(1), np.array([dphi(0.0)]), np.zeros(1), np.ones(1)
    fn = oracle._ls_morethuente if ls == 0 else oracle._ls_backtracking
    code, f, stp = fn(evaluate, x, phi(0.0), g, s, stp0, xp, p)
    return code, f, stp


def _product_search(name, ls, stp0, over):
    phi, dphi = PHI[name]
    lib = _lib.load()
    cfg = _lib.lbfgs_config_params(linesearch=ls, max_iterations=0, delta=1e-6, epsilon=1e-6,
                                   ftol=over.get("ftol", 1e-5), gtol=over.get("gtol", 0.9),
                                   wolfe=over.get("wolfe", 0.9), past=10,
                                   max_linesearch=over.get("max_linesearch", 100))
    CB = C.CFUNCTYPE(None, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double))

    def cb(t, f, dg):
        f[0] = phi(t)
        dg[0] = dphi(t)

    stp, f, n = C.c_double(), C.c_double(), C.c_int()
    code = lib.bioen_b200_selftest_linesearch(cfg, phi(0.0), dphi(0.0), stp0, CB(cb), C.byref(stp), C.byref(f),
                                              C.byref(n))
    return code, f.value, stp.value, n.value


@pytest.mark.parametrize("name", sorted(PHI))
@pytest.mark.parametrize("ls", [0, 1, 2, 3])
@pytest.mark.parametrize("stp0", [1e-3, 1.0, 25.0])
def test_linesearch_matches_liblbfgs_restatement(oracle, name, ls, stp0):
    for over in ({}, {"ftol": 1e-4, "gtol": 0.1, "wolfe": 0.5}, {"max_linesearch": 3}):
        try:
            co, fo, so = _oracle_search(oracle, name, ls, stp0, over)
        except ValueError:
            continue      # the Python restatement's math.sqrt raises where C yields NaN: nothing to compare against
        cp, fp, sp, n = _product_search(name, ls, stp0, over)
        assert cp == co, (name, ls, stp0, over, cp, co)
        assert fp == fo and sp == so, (name, ls, stp0, over, (fp, sp), (fo, so))
        if cp > 0:
            assert n == cp


def test_linesearch_rejects_ascent_direction_and_bad_step():
    lib = _lib.load()
    cfg = _lib.lbfgs_config_params(linesearch=2, max_iterations=0, delta=0, epsilon=0, ftol=1e-5, gtol=0.9,
                                   wolfe=0.9, past=0, max_linesearch=10)
    CB = C.CFUNCTYPE(None, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double))
    cb = CB(lambda t, f, dg: None)
    assert lib.bioen_b200_selftest_linesearch(cfg, 1.0, +0.5, 1.0, cb, None, None, None) == -994   # INCREASEGRADIENT
    assert lib.bioen_b200_selftest_linesearch(cfg, 1.0, -0.5, 0.0, cb, None, None, None) == -995   # INVALIDPARAMETERS


def test_fletcher_interpolation_matches_gsl_restatement(oracle):
    """gsl_min.cuh fletcher::interpolate (the bracketing / sectioning step of vector_bfgs2's line search) against
    the oracle's restatement of linear_minimize.c, including the NaN-derivative (quadratic) branch."""
    lib = _lib.load()
    rng = np.random.default_rng(11)
    for _ in range(400):
        a, b = sorted(rng.uniform(-2, 5, 2))
        fa, fb = rng.uniform(-3, 3, 2)
        fpa = rng.uniform(-4, 0.5)
        fpb = rng.uniform(-4, 4) if rng.random() < 0.7 else float("nan")
        lo, hi = sorted(rng.uniform(a - 1, b + 2, 2))
        for order in (2, 3):
            want = oracle._interpolate(a, fa, fpa, b, fb, fpb, lo, hi, order)
            got = lib.bioen_b200_selftest_interpolate(a, fa, fpa, b, fb, fpb, lo, hi, order)
            assert got == want or (math.isnan(got) and math.isnan(want)), (a, fa, fpa, b, fb, fpb, lo, hi, order)


def _run_two_loop_schedule(steps, g, S, Y, sc):
    """Execute the steps of bioen_b200_selftest_twoloop_schedule in NumPy with the oracle's operations: each dot product
    is np.dot(v, d), each quotient a separate division, each axpy d + coef*u."""
    ring = {1: S, 2: Y}
    d = None
    for init, u_kind, u_slot, v_kind, v_slot, c_num, c_den, csign, c2_num, scale, out in steps:
        if init:
            d = -g
        if u_kind:
            coef = float(csign) * (sc[c_num] / sc[c_den])
            if c2_num >= 0:
                coef = coef - sc[c2_num] / sc[c_den]
            d = d + coef * ring[u_kind][u_slot]
        if scale:
            d = d * (sc[16] / sc[17])
        if v_kind:
            sc[out] = float(np.dot(g if v_kind == 3 else ring[v_kind][v_slot], d))
    return d, sc


def test_two_loop_schedule_matches_oracle_recursion(oracle):
    """The two-loop schedule the minimisers launch (csrc/lbfgs.cuh two_loop_step; one entry per fused kernel step),
    run step by step in NumPy, reproduces the oracle's two-loop recursion bit for bit for every ring length m, ring end
    and history length.  Unused scalar-file entries are NaN, so a step that reads a slot nothing wrote shows up."""
    lib = _lib.load()
    rng = np.random.default_rng(7)
    n = 5
    steps = np.zeros(33 * 11, dtype=np.int32)
    sp = steps.ctypes.data_as(C.POINTER(C.c_int))
    for m in range(1, 17):
        for end in range(m):
            for bound in range(1, m + 1):
                count = lib.bioen_b200_selftest_twoloop_schedule(end, bound, m, sp)
                assert count == 2 * bound + 1, (m, end, bound, count)
                g = rng.standard_normal(n)
                S, Y = rng.standard_normal((m, n)), rng.standard_normal((m, n))
                ys_arr = rng.uniform(0.5, 2.0, m)
                newest = (end - 1) % m
                yy = rng.uniform(0.5, 2.0)
                sc = np.full(64, np.nan)
                sc[24:24 + m] = ys_arr
                sc[16], sc[17] = ys_arr[newest], yy
                d, sc = _run_two_loop_schedule(steps[:11 * count].reshape(count, 11), g, S, Y, sc)
                want = oracle.lbfgs_two_loop(g, S, Y, ys_arr, end, bound, ys_arr[newest], yy)
                assert np.array_equal(d, want), (m, end, bound)
                assert sc[19] == float(np.dot(g, want)), (m, end, bound)   # g.d for the next line search
    for bad in ((0, 1, 0), (0, 0, 6), (0, 7, 6), (6, 1, 6), (-1, 1, 6), (0, 17, 17)):
        assert lib.bioen_b200_selftest_twoloop_schedule(*bad, sp) == -1, bad
