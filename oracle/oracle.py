"""oracle/oracle.py -- TEST INFRASTRUCTURE ONLY (CPU checker for the CUDA path; never the product path).

Restates, on the CPU, the algorithms of BioEn's optimisation hot path:

  * evaluation of the log-posterior and gradient (log-weights and forces methods): NumPy restatement
    (`logw_fg_np`, `forces_fg_np`) and a ctypes binding to the plain-C restatement in bioen_oracle.c
    (`logw_fg`, `forces_fg`, ...), which is the faster one for mid-size inputs;
  * the liblbfgs 1.10 driver the reference calls (third-party/liblbfgs-1.10/lib/lbfgs.c) -- `lbfgs()` with the
    More-Thuente and the three backtracking line searches;
  * the GSL 2.5 multimin minimisers the reference calls (third-party/gsl-2.5/multimin/*) together with
    BioEn's own driver loop and stop test (c_bioen_kernels_logw.c:434-452, c_bioen_common.c:112-138) --
    `gsl_minimize()`.

Parity status: PINNED against the unmodified reference (oracle/_ref/libbioen_ref.so) and against the golden
vectors in tests/golden (see tests/test_oracle_cpu.py).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module.
All citations are relative to /root/reference/.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")
_dp = C.POINTER(C.c_double)
DBL_MIN = np.finfo(np.float64).tiny
DBL_EPSILON = 2.2204460492503131e-16


# ======================================================================================================
# 1. evaluation -- NumPy restatement
# ======================================================================================================
def logw_weights_np(g):
    """bioen/optimize/ext/c_bioen_kernels_logw.c:55-94 (no max-subtraction)."""
    e = np.exp(np.asarray(g, dtype=np.float64).ravel())
    s = e.sum()
    return e / s, s


def logw_fg_np(g, G, yTilde, YTilde, theta):
    """f and gradient, c_bioen_kernels_logw.c:96-147 (objective) and 151-268 (gradient)."""
    g = np.asarray(g, dtype=np.float64).ravel()
    G = np.asarray(G, dtype=np.float64).ravel()
    Y = np.asarray(YTilde, dtype=np.float64).ravel()
    yT = np.asarray(yTilde, dtype=np.float64)
    w, s = logw_weights_np(g)
    s0 = np.exp(G).sum()
    prior = theta * (np.dot(g - G, w) - math.log(s) + math.log(s0))
    avg = yT @ w
    r = avg - Y
    f = prior + 0.5 * np.dot(r, r)
    back = yT.T @ r - np.dot(r, avg)          # sum_i r_i (y_ij - avg_i)
    grad = w * theta * (g - np.dot(g, w) - G + np.dot(G, w)) + w * back
    return f, grad


def forces_weights_np(forces, w0, yTilde):
    """c_bioen_kernels_forces.c:111-224: w ~ w0 * exp(+ f . y), stabilised by the max."""
    f = np.asarray(forces, dtype=np.float64).ravel()
    w0 = np.asarray(w0, dtype=np.float64).ravel()
    x = f @ np.asarray(yTilde, dtype=np.float64)
    w = w0 * np.exp(x - x.max())
    return w / w.sum()


def forces_fg_np(forces, w0, yTilde, YTilde, theta):
    """c_bioen_kernels_forces.c:227-277 (objective) and 280-340 (gradient)."""
    w0 = np.asarray(w0, dtype=np.float64).ravel()
    Y = np.asarray(YTilde, dtype=np.float64).ravel()
    yT = np.asarray(yTilde, dtype=np.float64)
    w = forces_weights_np(forces, w0, yT)
    ok = (w >= DBL_MIN) & (w0 >= DBL_MIN)
    lr = np.zeros_like(w)
    lr[ok] = np.log(w[ok]) - np.log(w0[ok])
    avg = yT @ w
    r = avg - Y
    f = theta * np.dot(lr, w) + 0.5 * np.dot(r, r)
    E = (theta * (1.0 + lr) + yT.T @ r) * w
    grad = yT @ E - avg * E.sum()
    return f, grad


# ======================================================================================================
# 2. evaluation -- plain-C restatement (bioen_oracle.c) through ctypes
# ======================================================================================================
_lib = None


def build(force=False):
    if force or not os.path.isfile(_LIB) or (os.path.getmtime(_LIB) <
                                             os.path.getmtime(os.path.join(_HERE, "bioen_oracle.c"))):
        subprocess.check_call(["make", "-s", "-C", _HERE, "port"])


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        sz = C.c_size_t
        L.oracle_logw_weights.restype = C.c_double
        L.oracle_logw_weights.argtypes = [_dp, _dp, sz]
        L.oracle_average.restype = None
        L.oracle_average.argtypes = [_dp, _dp, _dp, sz, sz]
        L.oracle_logw_objective.restype = C.c_double
        L.oracle_logw_objective.argtypes = [_dp, _dp, _dp, _dp, C.c_double, _dp, _dp, sz, sz]
        L.oracle_logw_fg.restype = C.c_double
        L.oracle_logw_fg.argtypes = [_dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, sz, sz]
        L.oracle_forces_weights.restype = None
        L.oracle_forces_weights.argtypes = [_dp, _dp, _dp, _dp, _dp, sz, sz]
        L.oracle_forces_objective.restype = C.c_double
        L.oracle_forces_objective.argtypes = [_dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, sz, sz]
        L.oracle_forces_fg.restype = C.c_double
        L.oracle_forces_fg.argtypes = [_dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, sz, sz]
        _lib = L
    return _lib


_hostgen = None


def hostgen():
    """libhostgen.so (oracle/hostgen.c): host twin of the device's synthetic-data generator, for bench.py's
    reference arm and the tests that compare it with tests/util_rng.py."""
    global _hostgen
    if _hostgen is None:
        path = os.path.join(_HERE, "libhostgen.so")
        src = os.path.join(_HERE, "hostgen.c")
        if not os.path.isfile(path) or os.path.getmtime(path) < os.path.getmtime(src):
            subprocess.check_call(["make", "-s", "-C", _HERE, "hostgen"])
        L = C.CDLL(path)
        L.hostgen_generic_ytilde.restype = None
        L.hostgen_generic_ytilde.argtypes = [_dp, C.c_size_t, C.c_int, C.c_longlong, C.c_ulonglong, C.c_longlong, _dp,
                                             C.c_double]
        _hostgen = L
    return _hostgen


def _p(a):
    return a.ctypes.data_as(_dp)


def _vec(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel())


def _mat(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def logw_weights(g):
    g = _vec(g)
    w = np.empty_like(g)
    s = lib().oracle_logw_weights(_p(g), _p(w), g.size)
    return w, s


def logw_objective(g, G, yTilde, YTilde, theta):
    g, G, Y, yT = _vec(g), _vec(G), _vec(YTilde), _mat(yTilde)
    m, n = yT.shape
    w, avg = np.empty(n), np.empty(m)
    return lib().oracle_logw_objective(_p(g), _p(G), _p(yT), _p(Y), float(theta), _p(w), _p(avg), m, n)


def logw_fg(g, G, yTilde, YTilde, theta):
    g, G, Y, yT = _vec(g), _vec(G), _vec(YTilde), _mat(yTilde)
    m, n = yT.shape
    w, avg, grad = np.empty(n), np.empty(m), np.empty(n)
    f = lib().oracle_logw_fg(_p(g), _p(G), _p(yT), _p(Y), float(theta), _p(grad), _p(w), _p(avg), m, n)
    return f, grad


def forces_weights(forces, w0, yTilde):
    f, w0, yT = _vec(forces), _vec(w0), _mat(yTilde)
    m, n = yT.shape
    w, x = np.empty(n), np.empty(n)
    lib().oracle_forces_weights(_p(w0), _p(yT), _p(f), _p(w), _p(x), m, n)
    return w


def forces_objective(forces, w0, yTilde, YTilde, theta):
    f, w0, Y, yT = _vec(forces), _vec(w0), _vec(YTilde), _mat(yTilde)
    m, n = yT.shape
    w, x, avg = np.empty(n), np.empty(n), np.empty(m)
    return lib().oracle_forces_objective(_p(f), _p(w0), _p(yT), _p(Y), float(theta), _p(w), _p(x), _p(avg),
                                         m, n)


def forces_fg(forces, w0, yTilde, YTilde, theta):
    f, w0, Y, yT = _vec(forces), _vec(w0), _vec(YTilde), _mat(yTilde)
    m, n = yT.shape
    w, x, avg, grad = np.empty(n), np.empty(n), np.empty(m), np.empty(m)
    val = lib().oracle_forces_fg(_p(f), _p(w0), _p(yT), _p(Y), float(theta), _p(grad), _p(w), _p(x),
                                 _p(avg), m, n)
    return val, grad


def average(yTilde, w):
    yT, w = _mat(yTilde), _vec(w)
    m, n = yT.shape
    avg = np.empty(m)
    lib().oracle_average(_p(yT), _p(w), _p(avg), m, n)
    return avg


# ======================================================================================================
# 3. liblbfgs 1.10 restated  (third-party/liblbfgs-1.10/lib/lbfgs.c, include/lbfgs.h)
# ======================================================================================================
LBFGS_SUCCESS = 0
LBFGS_STOP = 1
LBFGS_ALREADY_MINIMIZED = 2
LBFGSERR_UNKNOWNERROR = -1024          # lbfgs.h:83-146, enum order
LBFGSERR_LOGICERROR = -1023
LBFGSERR_OUTOFMEMORY = -1022
LBFGSERR_CANCELED = -1021
LBFGSERR_INVALID_N = -1020
LBFGSERR_INVALID_N_SSE = -1019
LBFGSERR_INVALID_X_SSE = -1018
LBFGSERR_INVALID_EPSILON = -1017
LBFGSERR_INVALID_TESTPERIOD = -1016
LBFGSERR_INVALID_DELTA = -1015
LBFGSERR_INVALID_LINESEARCH = -1014
LBFGSERR_INVALID_MINSTEP = -1013
LBFGSERR_INVALID_MAXSTEP = -1012
LBFGSERR_INVALID_FTOL = -1011
LBFGSERR_INVALID_WOLFE = -1010
LBFGSERR_INVALID_GTOL = -1009
LBFGSERR_INVALID_XTOL = -1008
LBFGSERR_INVALID_MAXLINESEARCH = -1007
LBFGSERR_INVALID_ORTHANTWISE = -1006
LBFGSERR_INVALID_ORTHANTWISE_START = -1005
LBFGSERR_INVALID_ORTHANTWISE_END = -1004
LBFGSERR_OUTOFINTERVAL = -1003
LBFGSERR_INCORRECT_TMINMAX = -1002
LBFGSERR_ROUNDING_ERROR = -1001
LBFGSERR_MINIMUMSTEP = -1000
LBFGSERR_MAXIMUMSTEP = -999
LBFGSERR_MAXIMUMLINESEARCH = -998
LBFGSERR_MAXIMUMITERATION = -997
LBFGSERR_WIDTHTOOSMALL = -996
LBFGSERR_INVALIDPARAMETERS = -995
LBFGSERR_INCREASEGRADIENT = -994

LS_MORETHUENTE = 0
LS_ARMIJO = 1
LS_WOLFE = 2
LS_STRONG_WOLFE = 3

# what BioEn passes (config/bioen_optimize.yaml:33-46) on top of liblbfgs' _defparam (lbfgs.c:113-118)
LBFGS_BIOEN_DEFAULTS = dict(m=6, epsilon=1e-6, past=10, delta=1e-6, max_iterations=5000, linesearch=2,
                            max_linesearch=100, min_step=1e-20, max_step=1e20, ftol=1e-5, wolfe=0.9,
                            gtol=0.9, xtol=1e-16)


def _check_lbfgs_params(n, p):
    """lbfgs.c:286-364 (orthant-wise checks omitted: BioEn never sets orthantwise_c)."""
    if n <= 0:
        return LBFGSERR_INVALID_N
    if p["epsilon"] < 0.0:
        return LBFGSERR_INVALID_EPSILON
    if p["past"] < 0:
        return LBFGSERR_INVALID_TESTPERIOD
    if p["delta"] < 0.0:
        return LBFGSERR_INVALID_DELTA
    if p["min_step"] < 0.0:
        return LBFGSERR_INVALID_MINSTEP
    if p["max_step"] < p["min_step"]:
        return LBFGSERR_INVALID_MAXSTEP
    if p["ftol"] < 0.0:
        return LBFGSERR_INVALID_FTOL
    if p["linesearch"] in (LS_WOLFE, LS_STRONG_WOLFE):
        if p["wolfe"] <= p["ftol"] or 1.0 <= p["wolfe"]:
            return LBFGSERR_INVALID_WOLFE
    if p["gtol"] < 0.0:
        return LBFGSERR_INVALID_GTOL
    if p["xtol"] < 0.0:
        return LBFGSERR_INVALID_XTOL
    if p["max_linesearch"] <= 0:
        return LBFGSERR_INVALID_MAXLINESEARCH
    if p["linesearch"] not in (LS_MORETHUENTE, LS_ARMIJO, LS_WOLFE, LS_STRONG_WOLFE):
        return LBFGSERR_INVALID_LINESEARCH
    return 0


def _cubic_min(u, fu, du, v, fv, dv):
    """lbfgs.c:1021-1035."""
    d = v - u
    theta = (fu - fv) * 3 / d + du + dv
    s = max(abs(theta), abs(du), abs(dv))
    a = theta / s
    gamma = s * math.sqrt(a * a - (du / s) * (dv / s))
    if v < u:
        gamma = -gamma
    p = gamma - du + theta
    q = gamma - du + gamma + dv
    return u + (p / q) * d


def _cubic_min2(u, fu, du, v, fv, dv, xmin, xmax):
    """lbfgs.c:1049-1069."""
    d = v - u
    theta = (fu - fv) * 3 / d + du + dv
    s = max(abs(theta), abs(du), abs(dv))
    a = theta / s
    gamma = s * math.sqrt(max(0.0, a * a - (du / s) * (dv / s)))
    if u < v:
        gamma = -gamma
    p = gamma - dv + theta
    q = gamma - dv + gamma + du
    r = p / q
    if r < 0.0 and gamma != 0.0:
        return v - r * d
    return xmax if a < 0 else xmin


def _quad_min(u, fu, du, v, fv):
    """lbfgs.c:1080-1082."""
    a = v - u
    return u + du / ((fu - fv) / a + du) / 2 * a


def _quad_min2(u, du, v, dv):
    """lbfgs.c:1092-1094."""
    a = u - v
    return v + dv / (dv - du) * a


def _update_trial_interval(st):
    """lbfgs.c:1125-1292. `st` is a dict with x,fx,dx,y,fy,dy,t,ft,dt,tmin,tmax,brackt; updated in place."""
    x, fx, dx = st["x"], st["fx"], st["dx"]
    y, fy, dy = st["y"], st["fy"], st["dy"]
    t, ft, dt = st["t"], st["ft"], st["dt"]
    tmin, tmax, brackt = st["tmin"], st["tmax"], st["brackt"]
    dsign = (dt * (dx / abs(dx)) < 0.0) if dx != 0.0 else False   # fsigndiff (arithmetic_ansi.h:38)
    if brackt:
        if t <= min(x, y) or max(x, y) <= t:
            return LBFGSERR_OUTOFINTERVAL
        if 0.0 <= dx * (t - x):
            return LBFGSERR_INCREASEGRADIENT
        if tmax < tmin:
            return LBFGSERR_INCORRECT_TMINMAX
    if fx < ft:
        brackt, bound = True, True
        mc = _cubic_min(x, fx, dx, t, ft, dt)
        mq = _quad_min(x, fx, dx, t, ft)
        newt = mc if abs(mc - x) < abs(mq - x) else mc + 0.5 * (mq - mc)
    elif dsign:
        brackt, bound = True, False
        mc = _cubic_min(x, fx, dx, t, ft, dt)
        mq = _quad_min2(x, dx, t, dt)
        newt = mc if abs(mc - t) > abs(mq - t) else mq
    elif abs(dt) < abs(dx):
        bound = True
        mc = _cubic_min2(x, fx, dx, t, ft, dt, tmin, tmax)
        mq = _quad_min2(x, dx, t, dt)
        if brackt:
            newt = mc if abs(t - mc) < abs(t - mq) else mq
        else:
            newt = mc if abs(t - mc) > abs(t - mq) else mq
    else:
        bound = False
        if brackt:
            newt = _cubic_min(t, ft, dt, y, fy, dy)
        elif x < t:
            newt = tmax
        else:
            newt = tmin
    if fx < ft:
        y, fy, dy = t, ft, dt
    else:
        if dsign:
            y, fy, dy = x, fx, dx
        x, fx, dx = t, ft, dt
    if tmax < newt:
        newt = tmax
    if newt < tmin:
        newt = tmin
    if brackt and bound:
        mq = x + 0.66 * (y - x)
        if x < y:
            if mq < newt:
                newt = mq
        else:
            if newt < mq:
                newt = mq
    st.update(x=x, fx=fx, dx=dx, y=y, fy=fy, dy=dy, t=newt, brackt=brackt)
    return 0


def _ls_backtracking(evaluate, x, f, g, s, stp, xp, p):
    """lbfgs.c:645-734. Returns (ls, f, stp); x and g are updated in place."""
    if stp <= 0.0:
        return LBFGSERR_INVALIDPARAMETERS, f, stp
    dginit = float(np.dot(g, s))
    if 0 < dginit:
        return LBFGSERR_INCREASEGRADIENT, f, stp
    finit = f
    dgtest = p["ftol"] * dginit
    count = 0
    while True:
        x[:] = xp
        x += stp * s
        f = evaluate(x, g)
        count += 1
        if f > finit + stp * dgtest:
            width = 0.5
        else:
            if p["linesearch"] == LS_ARMIJO:
                return count, f, stp
            dg = float(np.dot(g, s))
            if dg < p["wolfe"] * dginit:
                width = 2.1
            else:
                if p["linesearch"] == LS_WOLFE:
                    return count, f, stp
                if dg > -p["wolfe"] * dginit:
                    width = 0.5
                else:
                    return count, f, stp
        if stp < p["min_step"]:
            return LBFGSERR_MINIMUMSTEP, f, stp
        if stp > p["max_step"]:
            return LBFGSERR_MAXIMUMSTEP, f, stp
        if p["max_linesearch"] <= count:
            return LBFGSERR_MAXIMUMLINESEARCH, f, stp
        stp *= width


def _ls_morethuente(evaluate, x, f, g, s, stp, xp, p):
    """lbfgs.c:812-1001."""
    if stp <= 0.0:
        return LBFGSERR_INVALIDPARAMETERS, f, stp
    dginit = float(np.dot(g, s))
    if 0 < dginit:
        return LBFGSERR_INCREASEGRADIENT, f, stp
    brackt, stage1, uinfo, count = False, True, 0, 0
    finit = f
    dgtest = p["ftol"] * dginit
    width = p["max_step"] - p["min_step"]
    prev_width = 2.0 * width
    stx = sty = 0.0
    fx = fy = finit
    dgx = dgy = dginit
    while True:
        if brackt:
            stmin, stmax = min(stx, sty), max(stx, sty)
        else:
            stmin, stmax = stx, stp + 4.0 * (stp - stx)
        if stp < p["min_step"]:
            stp = p["min_step"]
        if p["max_step"] < stp:
            stp = p["max_step"]
        if (brackt and ((stp <= stmin or stmax <= stp) or p["max_linesearch"] <= count + 1 or uinfo != 0)) \
                or (brackt and (stmax - stmin <= p["xtol"] * stmax)):
            stp = stx
        x[:] = xp
        x += stp * s
        f = evaluate(x, g)
        dg = float(np.dot(g, s))
        ftest1 = finit + stp * dgtest
        count += 1
        if brackt and ((stp <= stmin or stmax <= stp) or uinfo != 0):
            return LBFGSERR_ROUNDING_ERROR, f, stp
        if stp == p["max_step"] and f <= ftest1 and dg <= dgtest:
            return LBFGSERR_MAXIMUMSTEP, f, stp
        if stp == p["min_step"] and (ftest1 < f or dgtest <= dg):
            return LBFGSERR_MINIMUMSTEP, f, stp
        if brackt and (stmax - stmin) <= p["xtol"] * stmax:
            return LBFGSERR_WIDTHTOOSMALL, f, stp
        if p["max_linesearch"] <= count:
            return LBFGSERR_MAXIMUMLINESEARCH, f, stp
        if f <= ftest1 and abs(dg) <= p["gtol"] * (-dginit):
            return count, f, stp
        if stage1 and f <= ftest1 and min(p["ftol"], p["gtol"]) * dginit <= dg:
            stage1 = False
        if stage1 and ftest1 < f and f <= fx:
            st = dict(x=stx, fx=fx - stx * dgtest, dx=dgx - dgtest, y=sty, fy=fy - sty * dgtest,
                      dy=dgy - dgtest, t=stp, ft=f - stp * dgtest, dt=dg - dgtest, tmin=stmin, tmax=stmax,
                      brackt=brackt)
            uinfo = _update_trial_interval(st)
            stx, sty, stp, brackt = st["x"], st["y"], st["t"], st["brackt"]
            fx = st["fx"] + stx * dgtest
            fy = st["fy"] + sty * dgtest
            dgx = st["dx"] + dgtest
            dgy = st["dy"] + dgtest
        else:
            st = dict(x=stx, fx=fx, dx=dgx, y=sty, fy=fy, dy=dgy, t=stp, ft=f, dt=dg, tmin=stmin,
                      tmax=stmax, brackt=brackt)
            uinfo = _update_trial_interval(st)
            stx, fx, dgx = st["x"], st["fx"], st["dx"]
            sty, fy, dgy = st["y"], st["fy"], st["dy"]
            stp, brackt = st["t"], st["brackt"]
        if brackt:
            if 0.66 * prev_width <= abs(sty - stx):
                stp = stx + 0.5 * (sty - stx)
            prev_width = width
            width = abs(sty - stx)


def lbfgs_two_loop(g, S, Yv, ys_arr, end, bound, ys, yy):
    """liblbfgs' two-loop recursion (lbfgs.c:572-598): d = -H g over the `bound` newest pairs of the ring (S, Yv),
    the newest in slot end - 1; ys_arr[j] = y_j.s_j, and ys, yy of the newest pair scale H0."""
    m = len(ys_arr)
    alpha = np.zeros(m)
    d = -np.asarray(g, dtype=np.float64)
    j = end
    for _ in range(bound):
        j = (j + m - 1) % m
        alpha[j] = float(np.dot(S[j], d)) / ys_arr[j]
        d += (-alpha[j]) * Yv[j]
    d *= ys / yy
    for _ in range(bound):
        beta = float(np.dot(Yv[j], d)) / ys_arr[j]
        d += (alpha[j] - beta) * S[j]
        j = (j + 1) % m
    return d


def lbfgs(fg, x0, **params):
    """liblbfgs `lbfgs()` (lbfgs.c:245-641) restated for NumPy vectors.

    `fg(x) -> (f, grad)`.  Returns dict(x, fx, code, iterations, evaluations, trace).
    BioEn's driver (c_bioen_kernels_logw.c:581-669) copies x out and reports `code` whatever it is.
    """
    p = dict(LBFGS_BIOEN_DEFAULTS)
    p.update(params)
    x = np.array(x0, dtype=np.float64).ravel().copy()
    n = x.size
    info = dict(x=x, fx=0.0, code=0, iterations=0, evaluations=0, trace=[])
    code = _check_lbfgs_params(n, p)
    if code:
        info["code"] = code
        return info
    m = p["m"]
    nev = [0]

    def evaluate(xx, gout):
        f, gr = fg(xx)
        gout[:] = gr
        nev[0] += 1
        return float(f)

    linesearch = _ls_morethuente if p["linesearch"] == LS_MORETHUENTE else _ls_backtracking
    g = np.empty(n)
    xp, gp = np.empty(n), np.empty(n)
    S, Yv = np.zeros((m, n)), np.zeros((m, n))
    ys_arr = np.zeros(m)
    pf = np.zeros(p["past"]) if p["past"] > 0 else None

    fx = evaluate(x, g)
    if pf is not None:
        pf[0] = fx
    d = -g
    xnorm = max(1.0, math.sqrt(np.dot(x, x)))
    gnorm = math.sqrt(np.dot(g, g))
    if gnorm / xnorm <= p["epsilon"]:
        info.update(fx=fx, code=LBFGS_ALREADY_MINIMIZED, evaluations=nev[0])
        return info
    step = 1.0 / math.sqrt(np.dot(d, d))
    k, end = 1, 0
    while True:
        xp[:] = x
        gp[:] = g
        ls, fx, step = linesearch(evaluate, x, fx, g, d, step, xp, p)
        if ls < 0:
            x[:] = xp
            g[:] = gp
            code = ls
            break
        xnorm = math.sqrt(np.dot(x, x))
        gnorm = math.sqrt(np.dot(g, g))
        info["iterations"] += 1                       # progress callback (kernels_logw.c:565-576)
        info["trace"].append((k, fx, xnorm, gnorm, step, ls))
        if xnorm < 1.0:
            xnorm = 1.0
        if gnorm / xnorm <= p["epsilon"]:
            code = LBFGS_SUCCESS
            break
        if pf is not None:
            if p["past"] <= k:
                rate = (pf[k % p["past"]] - fx) / fx
                if rate < p["delta"]:
                    code = LBFGS_STOP
                    break
            pf[k % p["past"]] = fx
        if p["max_iterations"] != 0 and p["max_iterations"] < k + 1:
            code = LBFGSERR_MAXIMUMITERATION
            break
        S[end] = x - xp
        Yv[end] = g - gp
        ys = float(np.dot(Yv[end], S[end]))
        yy = float(np.dot(Yv[end], Yv[end]))
        ys_arr[end] = ys
        bound = m if m <= k else k
        k += 1
        end = (end + 1) % m
        d[:] = lbfgs_two_loop(g, S, Yv, ys_arr, end, bound, ys, yy)
        step = 1.0
    info.update(fx=fx, code=code, evaluations=nev[0])
    return info


# ======================================================================================================
# 4. GSL 2.5 multimin restated (third-party/gsl-2.5/multimin/*) + BioEn's driver loop
# ======================================================================================================
GSL_SUCCESS = 0
GSL_CONTINUE = -2
GSL_EBADTOL = 13
GSL_ENOPROG = 27
GSL_ALGORITHMS = {"conjugate_fr": 0, "conjugate_pr": 1, "bfgs2": 2, "bfgs": 3, "steepest_descent": 4}


def _nrm2(v):
    return math.sqrt(float(np.dot(v, v)))


def _solve_quadratic(a, b, c):
    """poly/solve_quadratic.c:27-88 -> list of real roots (ascending)."""
    if a == 0:
        return [] if b == 0 else [-c / b]
    disc = b * b - 4 * a * c
    if disc > 0:
        if b == 0:
            r = math.sqrt(-c / a)
            return [-r, r]
        sgnb = 1 if b > 0 else -1
        temp = -0.5 * (b + sgnb * math.sqrt(disc))
        r1, r2 = temp / a, c / temp
        return [r1, r2] if r1 < r2 else [r2, r1]
    if disc == 0:
        return [-0.5 * b / a, -0.5 * b / a]
    return []


def _interp_quad(f0, fp0, f1, zl, zh):
    """linear_minimize.c:10-30."""
    fl = f0 + zl * (fp0 + zl * (f1 - f0 - fp0))
    fh = f0 + zh * (fp0 + zh * (f1 - f0 - fp0))
    c = 2 * (f1 - f0 - fp0)
    zmin, fmin = zl, fl
    if fh < fmin:
        zmin, fmin = zh, fh
    if c > 0:
        z = -fp0 / c
        if zl < z < zh:
            f = f0 + z * (fp0 + z * (f1 - f0 - fp0))
            if f < fmin:
                zmin, fmin = z, f
    return zmin


def _interp_cubic(f0, fp0, f1, fp1, zl, zh):
    """linear_minimize.c:41-93."""
    eta = 3 * (f1 - f0) - 2 * fp0 - fp1
    xi = fp0 + fp1 - 2 * (f1 - f0)
    c0, c1, c2, c3 = f0, fp0, eta, xi

    def cubic(z):
        return c0 + z * (c1 + z * (c2 + z * c3))

    zmin, fmin = zl, cubic(zl)
    y = cubic(zh)
    if y < fmin:
        zmin, fmin = zh, y
    for z in _solve_quadratic(3 * c3, 2 * c2, c1):
        if zl < z < zh:
            y = cubic(z)
            if y < fmin:
                zmin, fmin = z, y
    return zmin


def _interpolate(a, fa, fpa, b, fb, fpb, xmin, xmax, order):
    """linear_minimize.c:96-124."""
    zmin = (xmin - a) / (b - a)
    zmax = (xmax - a) / (b - a)
    if zmin > zmax:
        zmin, zmax = zmax, zmin
    if order > 2 and math.isfinite(fpb):      # GSL_IS_REAL
        z = _interp_cubic(fa, fpa * (b - a), fb, fpb * (b - a), zmin, zmax)
    else:
        z = _interp_quad(fa, fpa * (b - a), fb, zmin, zmax)
    return a + z * (b - a)


class _Wrapper:
    """linear_wrapper.c:25-185: 1-d view f(alpha) = F(x + alpha p) with alpha-keyed caches."""

    def __init__(self, F, x, f, g, p):
        self.F, self.x, self.g, self.p = F, x, g, p
        self.x_alpha, self.g_alpha = x.copy(), g.copy()
        self.x_key = self.f_key = self.g_key = self.df_key = 0.0
        self.f_alpha = f
        self.df_alpha = float(np.dot(self.g_alpha, p))

    def moveto(self, alpha):
        if alpha == self.x_key:
            return
        self.x_alpha[:] = self.x
        self.x_alpha += alpha * self.p
        self.x_key = alpha

    def f(self, alpha):
        if alpha == self.f_key:
            return self.f_alpha
        self.moveto(alpha)
        self.f_alpha = self.F.f(self.x_alpha)
        self.f_key = alpha
        return self.f_alpha

    def df(self, alpha):
        if alpha == self.df_key:
            return self.df_alpha
        self.moveto(alpha)
        if alpha != self.g_key:
            self.g_alpha[:] = self.F.df(self.x_alpha)
            self.g_key = alpha
        self.df_alpha = float(np.dot(self.g_alpha, self.p))
        self.df_key = alpha
        return self.df_alpha

    def fdf(self, alpha):
        if alpha == self.f_key and alpha == self.df_key:
            return self.f_alpha, self.df_alpha
        if alpha == self.f_key or alpha == self.df_key:
            return self.f(alpha), self.df(alpha)
        self.moveto(alpha)
        self.f_alpha, gr = self.F.fdf(self.x_alpha)
        self.g_alpha[:] = gr
        self.f_key = self.g_key = alpha
        self.df_alpha = float(np.dot(self.g_alpha, self.p))
        self.df_key = alpha
        return self.f_alpha, self.df_alpha

    def update_position(self, alpha, x, g):
        self.fdf(alpha)
        x[:] = self.x_alpha
        g[:] = self.g_alpha
        return self.f_alpha

    def change_direction(self):
        self.x_alpha[:] = self.x
        self.x_key = 0.0
        self.f_key = 0.0
        self.g_alpha[:] = self.g
        self.g_key = 0.0
        self.df_alpha = float(np.dot(self.g_alpha, self.p))
        self.df_key = 0.0


def _fletcher_minimize(w, rho, sigma, tau1, tau2, tau3, order, alpha1):
    """linear_minimize.c:130-247. Returns (status, alpha)."""
    f0, fp0 = w.fdf(0.0)
    falpha_prev, fpalpha_prev = f0, fp0
    alpha, alpha_prev = alpha1, 0.0
    a, b, fa, fb, fpa, fpb = 0.0, alpha, f0, 0.0, fp0, 0.0
    i = 0
    while i < 100:                       # bracket_iters
        i += 1
        falpha = w.f(alpha)
        if falpha > f0 + alpha * rho * fp0 or falpha >= falpha_prev:
            a, fa, fpa = alpha_prev, falpha_prev, fpalpha_prev
            b, fb, fpb = alpha, falpha, float("nan")
            break
        fpalpha = w.df(alpha)
        if abs(fpalpha) <= -sigma * fp0:
            return GSL_SUCCESS, alpha
        if fpalpha >= 0:
            a, fa, fpa = alpha, falpha, fpalpha
            b, fb, fpb = alpha_prev, falpha_prev, fpalpha_prev
            break
        delta = alpha - alpha_prev
        alpha_next = _interpolate(alpha_prev, falpha_prev, fpalpha_prev, alpha, falpha, fpalpha,
                                  alpha + delta, alpha + tau1 * delta, order)
        alpha_prev, falpha_prev, fpalpha_prev = alpha, falpha, fpalpha
        alpha = alpha_next
    else:
        i += 1                           # `while (i++ < bracket_iters)` leaves i = 101 on exhaustion
    while i < 100:                       # section_iters (shares the counter i, as in the C code)
        i += 1
        delta = b - a
        alpha = _interpolate(a, fa, fpa, b, fb, fpb, a + tau2 * delta, b - tau3 * delta, order)
        falpha = w.f(alpha)
        if (a - alpha) * fpa <= DBL_EPSILON:
            return GSL_ENOPROG, alpha
        if falpha > f0 + rho * alpha * fp0 or falpha >= fa:
            b, fb, fpb = alpha, falpha, float("nan")
        else:
            fpalpha = w.df(alpha)
            if abs(fpalpha) <= -sigma * fp0:
                return GSL_SUCCESS, alpha
            if ((b - a) >= 0 and fpalpha >= 0) or ((b - a) <= 0 and fpalpha <= 0):
                b, fb, fpb = a, fa, fpa
            a, fa, fpa = alpha, falpha, fpalpha
    # linear_minimize.c:246: falling out of the sectioning loop returns GSL_SUCCESS *without* writing
    # *alpha_new, so the caller keeps its initial `alpha = 0.0` (vector_bfgs2.c:213).
    return GSL_SUCCESS, 0.0


class _Functions:
    """The three callbacks BioEn registers (c_bioen_kernels_logw.c:426-431): f-only, df-only, fdf."""

    def __init__(self, fg, f_only=None):
        self._fg = fg
        self._f = f_only
        self.n_f = self.n_df = self.n_fdf = 0

    def f(self, x):
        self.n_f += 1
        return float(self._f(x)) if self._f is not None else float(self._fg(x)[0])

    def df(self, x):
        self.n_df += 1
        return self._fg(x)[1]

    def fdf(self, x):
        self.n_fdf += 1
        f, g = self._fg(x)
        return float(f), g


class _Bfgs2:
    """multimin/vector_bfgs2.c:143-318."""

    def __init__(self, F, x, step_size, tol):
        self.F = F
        self.x = x
        self.f, g = F.fdf(x)
        self.g = np.array(g, dtype=np.float64)
        self.dx = np.zeros_like(x)
        self.step, self.delta_f = step_size, 0.0
        self.x0, self.g0 = x.copy(), self.g.copy()
        self.g0norm = _nrm2(self.g0)
        self.p = self.g * (-1 / self.g0norm)
        self.pnorm = _nrm2(self.p)
        self.fp0 = -self.g0norm
        self.w = _Wrapper(F, self.x0, self.f, self.g0, self.p)
        self.rho, self.sigma, self.tau1, self.tau2, self.tau3, self.order = 0.01, tol, 9.0, 0.05, 0.5, 3

    def iterate(self):
        f0 = self.f
        if self.pnorm == 0.0 or self.g0norm == 0.0 or self.fp0 == 0:
            self.dx[:] = 0
            return GSL_ENOPROG
        if self.delta_f < 0:
            dl = max(-self.delta_f, 10 * DBL_EPSILON * abs(f0))
            alpha1 = min(1.0, 2.0 * dl / (-self.fp0))
        else:
            alpha1 = abs(self.step)
        status, alpha = _fletcher_minimize(self.w, self.rho, self.sigma, self.tau1, self.tau2, self.tau3,
                                           self.order, alpha1)
        if status != GSL_SUCCESS:
            return status
        self.f = self.w.update_position(alpha, self.x, self.g)
        self.delta_f = self.f - f0
        dx0 = self.x - self.x0
        self.dx[:] = dx0
        dg0 = self.g - self.g0
        dxg, dgg, dxdg = float(np.dot(dx0, self.g)), float(np.dot(dg0, self.g)), float(np.dot(dx0, dg0))
        dgnorm = _nrm2(dg0)
        if dxdg != 0:
            B = dxg / dxdg
            A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg
        else:
            A = B = 0.0
        self.p[:] = self.g
        self.p += (-A) * dx0
        self.p += (-B) * dg0
        self.g0[:] = self.g
        self.x0[:] = self.x
        self.g0norm = _nrm2(self.g0)
        self.pnorm = _nrm2(self.p)
        pg = float(np.dot(self.p, self.g))
        dirn = -1.0 if pg >= 0.0 else 1.0
        self.p *= dirn / self.pnorm
        self.pnorm = _nrm2(self.p)
        self.fp0 = float(np.dot(self.p, self.g0))
        self.w.change_direction()
        return GSL_SUCCESS


def _take_step(x, p, step, lam):
    """directional_minimize.c:20-29 -> (x1, dx)."""
    dx = (-step * lam) * p
    return x + dx, dx


def _intermediate_point(F, x, p, lam, pg, stepc, fa, fc):
    """directional_minimize.c:31-83 -> (x1, dx, gradient, step, f)."""
    while True:
        u = abs(pg * lam * stepc)
        stepb = 0.5 * stepc * u / ((fc - fa) + u)
        x1, dx = _take_step(x, p, stepb, lam)
        if np.array_equal(x, x1):
            return x1, dx, F.df(x1), 0.0, fa
        fb = F.f(x1)
        if fb >= fa and stepb > 0.0:
            fc, stepc = fb, stepb
            continue
        return x1, dx, F.df(x1), stepb, fb


def _directional_minimize(F, x, p, lam, stepa, stepb, stepc, fa, fb, fc, tol, x1, dx1, gradient):
    """directional_minimize.c:85-248 -> (x2, dx2, gradient, step, f, gnorm)."""
    u, v, w = stepb, stepa, stepc
    fu, fv, fw = fb, fa, fc
    old2, old1 = abs(w - v), abs(v - u)
    x2, dx2 = x1.copy(), dx1.copy()
    f, step, gnorm = fb, stepb, _nrm2(gradient)
    it = 0
    while True:
        it += 1
        if it > 10:
            return x2, dx2, gradient, step, f, gnorm
        dw, dv, du = w - u, v - u, 0.0
        e1 = (fv - fu) * dw * dw + (fu - fw) * dv * dv
        e2 = 2.0 * ((fv - fu) * dw + (fu - fw) * dv)
        if e2 != 0.0:
            du = e1 / e2
        if du > 0.0 and du < (stepc - stepb) and abs(du) < 0.5 * old2:
            stepm = u + du
        elif du < 0.0 and du > (stepa - stepb) and abs(du) < 0.5 * old2:
            stepm = u + du
        elif (stepc - stepb) > (stepb - stepa):
            stepm = 0.38 * (stepc - stepb) + stepb
        else:
            stepm = stepb - 0.38 * (stepb - stepa)
        x1, dx1 = _take_step(x, p, stepm, lam)
        fm = F.f(x1)
        if fm > fb:
            if fm < fv:
                w, v, fw, fv = v, stepm, fv, fm
            elif fm < fw:
                w, fw = stepm, fm
            if stepm < stepb:
                stepa, fa = stepm, fm
            else:
                stepc, fc = stepm, fm
            continue
        elif fm <= fb:
            old2 = old1
            old1 = abs(u - stepm)
            w, v, u = v, u, stepm
            fw, fv, fu = fv, fu, fm
            x2, dx2 = x1.copy(), dx1.copy()
            gradient = np.array(F.df(x1), dtype=np.float64)
            pg = float(np.dot(p, gradient))
            gnorm1 = _nrm2(gradient)
            f, step, gnorm = fm, stepm, gnorm1
            if abs(pg * lam / gnorm1) < tol:
                return x2, dx2, gradient, step, f, gnorm
            if stepm < stepb:
                stepc, fc, stepb, fb = stepb, fb, stepm, fm
            else:
                stepa, fa, stepb, fb = stepb, fb, stepm, fm
            continue
        else:  # NaN: neither branch in the C code either -> falls out of the function
            return x2, dx2, gradient, step, f, gnorm


class _Directional:
    """conjugate_fr.c:100-256, conjugate_pr.c (beta at 238-243), vector_bfgs.c:142-337."""

    def __init__(self, F, x, step_size, tol, kind):
        self.F, self.x, self.kind = F, x, kind
        self.f, g = F.fdf(x)
        self.g = np.array(g, dtype=np.float64)
        self.dx = np.zeros_like(x)
        self.iter = 0
        self.step = self.max_step = step_size
        self.tol = tol
        self.p, self.g0 = self.g.copy(), self.g.copy()
        self.x0 = x.copy()
        self.pnorm = self.g0norm = _nrm2(self.g)

    def iterate(self):
        F, x, p = self.F, self.x, self.p
        fa, stepa, stepc, tol = self.f, 0.0, self.step, self.tol
        if self.pnorm == 0.0 or self.g0norm == 0.0:
            self.dx[:] = 0
            return GSL_ENOPROG
        pg = float(np.dot(p, self.g))
        dirn = 1.0 if pg >= 0.0 else -1.0
        lam = dirn / self.pnorm
        x1, dx = _take_step(x, p, stepc, lam)
        self.dx[:] = dx
        fc = F.f(x1)
        if fc < fa:
            self.step = stepc * 2.0
            self.f = fc
            x[:] = x1
            self.g[:] = F.df(x1)
            return GSL_SUCCESS
        x1, dx1, grad, stepb, fb = _intermediate_point(F, x, p, lam, pg, stepc, fa, fc)
        self.g[:] = grad
        if stepb == 0.0:
            return GSL_ENOPROG
        x2, dx2, grad, self.step, self.f, g1norm = _directional_minimize(
            F, x, p, lam, stepa, stepb, stepc, fa, fb, fc, tol, x1, dx1, self.g.copy())
        self.g[:] = grad
        self.dx[:] = dx2
        x[:] = x2
        self.iter = (self.iter + 1) % x.size
        if self.iter == 0:
            p[:] = self.g
            self.pnorm = g1norm
        elif self.kind == "conjugate_fr":
            beta = -((g1norm / self.g0norm) ** 2.0)
            p *= -beta
            p += self.g
            self.pnorm = _nrm2(p)
        elif self.kind == "conjugate_pr":
            self.g0 -= self.g
            g0g1 = float(np.dot(self.g0, self.g))
            beta = g0g1 / (self.g0norm * self.g0norm)
            p *= -beta
            p += self.g
            self.pnorm = _nrm2(p)
        else:  # vector_bfgs
            dx0 = x - self.x0
            dg0 = self.g - self.g0
            dxg, dgg, dxdg = float(np.dot(dx0, self.g)), float(np.dot(dg0, self.g)), float(np.dot(dx0, dg0))
            dgnorm = _nrm2(dg0)
            if dxdg != 0:
                B = dxg / dxdg
                A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg
            else:
                A = B = 0.0
            p[:] = self.g
            p += (-A) * dx0
            p += (-B) * dg0
            self.pnorm = _nrm2(p)
        if self.kind == "bfgs":
            self.g0[:] = self.g
            self.x0[:] = x
            self.g0norm = _nrm2(self.g0)
        else:
            self.g0norm = g1norm
            self.g0[:] = self.g
        return GSL_SUCCESS


class _SteepestDescent:
    """steepest_descent.c:63-163."""

    def __init__(self, F, x, step_size, tol):
        self.F, self.x = F, x
        self.f, g = F.fdf(x)
        self.g = np.array(g, dtype=np.float64)
        self.dx = np.zeros_like(x)
        self.step = self.max_step = step_size
        self.tol = tol

    def iterate(self):
        f0, step, tol = self.f, self.step, self.tol
        failed = False
        gnorm = _nrm2(self.g)
        if gnorm == 0.0:
            self.dx[:] = 0
            return GSL_ENOPROG
        while True:
            self.dx[:] = (-step / gnorm) * self.g
            x1 = self.x + self.dx
            if np.array_equal(self.x, x1):
                return GSL_ENOPROG
            f1, g1 = self.F.fdf(x1)
            if f1 > f0:
                failed = True
                step *= tol
                continue
            break
        step = step * tol if failed else step * 2.0
        self.step = step
        self.x[:] = x1
        self.g[:] = g1
        self.f = f1
        return GSL_SUCCESS


def gsl_minimize(fg, x0, algorithm="bfgs2", step_size=0.01, tol=0.001, max_iterations=5000, f_only=None):
    """BioEn's GSL driver: c_bioen_kernels_logw.c:367-509 (forces twin kernels_forces.c:431-570).

    Returns dict(x, fx, code, iterations, n_f, n_df, n_fdf).  `code` is what the driver writes to *error:
    0 (||g||_inf < tol), GSL_CONTINUE (-2, max_iterations reached) or the non-zero status of iterate().
    """
    if isinstance(algorithm, str):
        algorithm = GSL_ALGORITHMS[algorithm]
    F = _Functions(fg, f_only)
    x = np.array(x0, dtype=np.float64).ravel().copy()
    if algorithm == 2:
        s = _Bfgs2(F, x, step_size, tol)
    elif algorithm == 4:
        s = _SteepestDescent(F, x, step_size, tol)
    else:
        s = _Directional(F, x, step_size, tol, {0: "conjugate_fr", 1: "conjugate_pr", 3: "bfgs"}[algorithm])
    it = 0
    while True:
        status = s.iterate()
        if status:
            break
        # gsl_multimin_test_gradient__scipy_optimize_vecnorm (c_bioen_common.c:112-138)
        if tol < 0.0:
            status = GSL_EBADTOL
        else:
            # `if (temp > norm) norm = temp` skips NaNs, hence fmax
            status = GSL_SUCCESS if np.fmax.reduce(np.abs(s.g), initial=0.0) < tol else GSL_CONTINUE
        it += 1
        if not (status == GSL_CONTINUE and it < max_iterations):
            break
    return dict(x=s.x.copy(), fx=s.f, code=status, iterations=it, n_f=F.n_f, n_df=F.n_df, n_fdf=F.n_fdf)


# ======================================================================================================
# 5. synthetic "generic data" problems (SURVEY.md section 8d; recipe of bioen/optimize/forces.py:19-68)
# ======================================================================================================
def synthetic_problem(M, N, seed=12345, sig_exp=0.5, sig_sim=1.0, dtype=np.float64):
    rng = np.random.default_rng(seed)
    YTrue = rng.standard_normal(M)
    YObs = YTrue + sig_exp * rng.standard_normal(M)
    y = YTrue[:, None] + sig_sim * rng.standard_normal((M, N))
    yTilde = np.ascontiguousarray(y / sig_exp, dtype=dtype)
    YTilde = (YObs / sig_exp)[None, :]
    w0 = np.full((N, 1), 1.0 / N)
    G = np.zeros((N, 1))
    return dict(M=M, N=N, y=y, yTilde=yTilde, YTilde=YTilde, w0=w0, G=G, GInit=G.copy(),
                forces_init=np.zeros((M, 1)))
