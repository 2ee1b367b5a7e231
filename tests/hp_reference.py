"""Extended-precision reference of both BioEn methods, with a running error bound for every output.

The fp64 oracle (oracle/bioen_oracle.c) restates the reference's formulas and summation order, so it is the right
yardstick for bit-level parity in the regime the reference itself evaluates well.  It cannot judge a kernel where the
reference's own fp64 arithmetic breaks down: its softmax is not stabilised (log-weights beyond a range of ~709
overflow), and where f is a small difference of large numbers two fp64 evaluations agree with each other no better
than with the truth.  This module computes the same quantities in x86-64 extended precision (64-bit mantissa, 11 more
bits than fp64), stabilised by the maximum, so the result is defined wherever the mathematical value is.

Every output comes with a SCALE: the same expression with every term replaced by its absolute value (running error
analysis).  An fp64 implementation that evaluates the expression in any order, with any blocking and any stabilising
maxima, is within a small multiple of u * scale (u = 2^-53) of the exact value; a kernel is accepted when

    |gpu - ref| <= C * u * scale + floor        (componentwise)

with C a constant of the test file and floor a few 2^-1074 where subnormal results are possible.  Inputs are fp64 and
therefore exact here; the reference itself is good to ~2^-64 * scale, far inside the bound.

Semantics are the reference's (bioen/optimize/ext/c_bioen_kernels_logw.c, c_bioen_kernels_forces.c):
  log-weights  w = softmax(g);  f = theta (sum (g - G) w - log s + log s0) + chi^2;
               grad_j = w_j theta (g_j - gbar - G_j + Gbar) + w_j sum_i c_i r_i (y_ij - avg_i)
  forces       x = f . y;  w = w0 e^x / sum;  lr_j = log w_j - log w0_j where fl(w_j) >= DBL_MIN and w0_j >= DBL_MIN,
               else 0;  KL = sum w lr;  f = theta KL + chi^2;  grad_i = sum_j (y_ij - avg_i) E_j,
               E_j = (theta (1 + lr_j) + t_j) w_j,  t_j = sum_i y_ij c_i r_i
  with chi^2 = 1/2 sum_i c_i r_i^2, r = avg - YTilde, avg = y . w and observable weights c (1 unless given: the
  batched replicates' row weights).
"""
import numpy as np

LD = np.longdouble
U = 2.0 ** -53
TINY = np.finfo(np.float64).tiny          # DBL_MIN
SUB = 2.0 ** -1074                         # smallest subnormal


def available():
    """True where np.longdouble is the x86-64 80-bit format (64-bit mantissa)"""
    return np.finfo(np.longdouble).nmant >= 63


def _ld(a):
    return np.asarray(a, dtype=np.float64).astype(LD)


def _rows(c, M):
    return np.ones(M, dtype=LD) if c is None else _ld(c).reshape(M)


def _observables(y, w, wsc, Y, c):
    """avg, r, chi^2 and their scales for weights w whose absolute error scale is wsc"""
    M = y.shape[0]
    ay = np.abs(y)
    avg = y @ w
    s_avg = ay @ wsc
    Yv = _ld(Y).reshape(M)
    r = avg - Yv
    s_r = s_avg + np.abs(Yv)
    c = _rows(c, M)
    chi2 = LD(0.5) * np.sum(c * r * r)
    s_chi2 = np.sum(c * np.abs(r) * s_r) + chi2
    return dict(avg=avg, s_avg=s_avg, r=r, s_r=s_r, c=c, chi2=chi2, s_chi2=s_chi2)


def logw(g, G, y, Y, theta, c=None):
    """log-weights method at g.  Returns a dict of longdouble arrays: f, grad, w, avg, chi2, prior (theta * KL) and
    kl (= prior / theta: the relative entropy of w to softmax(G)), each with its scale s_<name>; s_w is absolute."""
    g, G, y = _ld(g).ravel(), _ld(G).ravel(), _ld(y)
    th = LD(theta)
    N = g.size
    m = np.max(g)
    e = np.exp(g - m)
    S = np.sum(e)
    w = e / S
    mG = np.max(G)
    S0 = np.sum(np.exp(G - mG))
    logs, logs0 = m + np.log(S), mG + np.log(S0)
    # weights: exp of a rounded difference (|g_j - m| u relative), the normalisation; subnormal e_j lose absolute 2^-1075
    relw = 1 + np.abs(g - m) + np.log2(LD(N) + 1)
    wsc = w * relw + LD(SUB / U) / S
    o = _observables(y, w, wsc, Y, c)
    d = g - G
    kl = np.sum(d * w) - logs + logs0
    s_kl = np.sum(np.abs(d) * wsc) + abs(m) + abs(np.log(S)) + abs(mG) + abs(np.log(S0)) + 1
    gbar, Gbar = np.sum(g * w), np.sum(G * w)
    agbar, aGbar = np.sum(np.abs(g) * wsc), np.sum(np.abs(G) * wsc)
    cr = o["c"] * o["r"]
    ay = np.abs(y)
    col = cr @ y - np.dot(cr, o["avg"])                    # sum_i c_i r_i (y_ij - avg_i)
    grad = w * th * (g - gbar - G + Gbar) + w * col
    # |c r| (|y| + |avg|) plus the error of r and avg carried through: c (|r| + s_r) (|y| + s_avg)
    acr = o["c"] * (np.abs(o["r"]) + o["s_r"])
    s_col = acr @ ay + np.dot(acr, o["s_avg"])
    s_grad = wsc * (abs(th) * (np.abs(g) + agbar + np.abs(G) + aGbar) + s_col)
    prior = th * kl
    out = dict(f=prior + o["chi2"], s_f=abs(th) * s_kl + o["s_chi2"], grad=grad, s_grad=s_grad, w=w, s_w=wsc,
               prior=prior, s_prior=abs(th) * s_kl, kl=kl, s_kl=s_kl)
    out.update(avg=o["avg"], s_avg=o["s_avg"], chi2=o["chi2"], s_chi2=o["s_chi2"])
    return out


def forces(f, w0, y, Y, theta, c=None, guard_w0=True):
    """forces method at f (same outputs as logw; kl is the guarded relative entropy sum w lr).  guard_w0=False drops
    the reference's w0_j >= DBL_MIN condition (what a kernel without that guard computes)."""
    f, w0v, y = _ld(f).ravel(), np.asarray(w0, dtype=np.float64).ravel(), _ld(y)
    w0 = w0v.astype(LD)
    th = LD(theta)
    M, N = y.shape
    ay = np.abs(y)
    x = f @ y
    s_x = np.abs(f) @ ay
    pos = w0v > 0
    if not pos.any():
        raise ValueError("w0 has no positive entry")
    m = np.max(x[pos])                                    # stabilised over the structures that carry weight
    u = w0 * np.exp(x - m)
    S = np.sum(u)
    w = u / S
    logS = np.log(S)
    # the weights as the reference forms them, w0 e^{x - max_all x} / sum: x_j and the maximum carry their rounding,
    # the products may be subnormal (absolute 2^-1075 each, on u and on the sum)
    mall = np.max(x)
    Sall = np.sum(w0 * np.exp(x - mall))
    eps_sub = LD(N) * LD(SUB / U) / Sall
    relw = 1 + s_x + np.max(s_x) + np.log2(LD(N) + 1) + eps_sub
    wsc = w * relw + LD(SUB / U) / Sall
    o = _observables(y, w, wsc, Y, c)
    w64 = w.astype(np.float64)
    ok = (w64 >= TINY) & ((w0v >= TINY) if guard_w0 else True)
    lr = np.where(ok, x - m - logS, LD(0))
    s_lr = np.where(ok, np.abs(x) + s_x + abs(m) + np.max(s_x) + abs(logS) + 1, LD(0))
    kl = np.sum(w * lr)
    s_kl = np.sum(np.abs(lr) * wsc + w * s_lr)
    cr = o["c"] * o["r"]
    t = cr @ y
    acr = o["c"] * (np.abs(o["r"]) + o["s_r"])
    s_t = acr @ ay
    E = (th * (1 + lr) + t) * w
    s_E = (abs(th) * (1 + np.abs(lr)) + np.abs(t)) * wsc + w * (abs(th) * s_lr + s_t)
    grad = y @ E - o["avg"] * np.sum(E)
    s_grad = ay @ s_E + o["s_avg"] * np.sum(s_E)
    out = dict(f=th * kl + o["chi2"], s_f=abs(th) * s_kl + o["s_chi2"], grad=grad, s_grad=s_grad, w=w, s_w=wsc,
               prior=th * kl, s_prior=abs(th) * s_kl, kl=kl, s_kl=s_kl, x=x, lr=lr)
    out.update(avg=o["avg"], s_avg=o["s_avg"], chi2=o["chi2"], s_chi2=o["s_chi2"])
    return out


def ratio(got, ref, scale, floor=0.0):
    """max_k |got_k - ref_k| / (u scale_k), after subtracting an absolute floor; inf where got is not finite but ref
    is (a NaN or inf from a kernel is never within the bound)"""
    got = np.asarray(got, dtype=np.float64).ravel()
    ref, scale = np.asarray(ref, dtype=LD).ravel(), np.asarray(scale, dtype=LD).ravel()
    if got.shape != ref.shape:
        raise ValueError("shape mismatch %s vs %s" % (got.shape, ref.shape))
    if not np.all(np.isfinite(got)):
        return float("inf")
    err = np.maximum(np.abs(got.astype(LD) - ref) - LD(floor), LD(0))
    den = LD(U) * scale
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(err == 0, LD(0), err / den)
    return float(np.max(q)) if q.size else 0.0


# what each compared output is allowed beyond C u scale: weights and their products may be subnormal
FLOORS = dict(w=4 * SUB, grad=4 * SUB, avg=0.0, f=0.0, chi2=0.0, kl=0.0, prior=0.0)


def ratios(ref, **got):
    """{name: ratio} for the outputs given as keyword arguments (f=..., grad=..., w=..., avg=..., chi2=..., kl=...)"""
    return {k: ratio(v, ref[k], ref["s_" + k], FLOORS.get(k, 0.0)) for k, v in got.items() if v is not None}
