"""Extended-precision reference of one L-BFGS direction update, with a first-order error scale for every output.

liblbfgs (lbfgs.c:543-598) forms the new pair s = x - xp, y = g - gp, ys = y.s, yy = y.y, stores them in ring slot
`end_old`, and runs the two-loop recursion d = -H g over the `bound` newest pairs:

    d = -g;  for j = newest .. oldest:  alpha_j = (s_j . d) / ys_j;  d -= alpha_j y_j
    d *= ys / yy
    for j = oldest .. newest:  beta = (y_j . d) / ys_j;  d += (alpha_j - beta) s_j

The device keeps the raw s_j . d of the first loop in the scalar file (SC_ALPHA0 + j) and g . d of the new direction
(SC_DGINIT).  Here every operation runs in x86-64 extended precision (64-bit mantissa) on the fp64 inputs, and every
output carries a SCALE propagated alongside it (first order, in units of u = 2^-53):
  - a dot product a . b contributes  sum |a_i b_i| (ceil(log2 n) + 1)  (the reduction depth), plus the inputs' scales
    carried through (sum |a_i| scale(b_i)), plus n 2^-1074 / u for products that may underflow;
  - a quotient a / ys carries scale(a) / |ys| + |a / ys| scale(ys) / |ys| + |a / ys|, so cancellation in ys widens it;
  - each axpy or scaling adds |result| (+ 2^-1074 / u for a subnormal result).
A kernel is accepted when |gpu - ref| <= C u scale componentwise.  The ring's ys of the older pairs are inputs (the
device's own values), exact here.  Where an input makes an output non-finite (ys = 0: a pair that did not move), the
reference is non-finite in exactly the components the device must be non-finite in.

The coefficient-space engine (Gram) rounds along another formula: the recursion runs on 13 coefficients c over the
basis b = [s_0..s_5, y_0..y_5, g] with a Gram matrix of dot products, and d = sum_k c_k b_k.  gram() restates it with
its own scale: every c_k G_row,k of the recursion in absolute value, then sum |c_k| |b_k| for the combine.
"""
import math

import numpy as np

LD = np.longdouble
U = 2.0 ** -53
SUB = 2.0 ** -1074
M = 6                                   # liblbfgs' history length (BioEn never changes it)
GRAM_B = 2 * M + 1


def _ld(a):
    return np.asarray(a, dtype=np.float64).astype(LD)


def _depth(n):
    return LD(math.ceil(math.log2(n)) + 1 if n > 1 else 1)


def _dot(a, b, sb=None):
    """a . b with a exact (fp64 input) and b carrying the scale sb"""
    n = a.size
    v = np.sum(a * b)
    s = _depth(n) * np.sum(np.abs(a * b)) + LD(n) * LD(SUB / U)
    if sb is not None:
        s = s + np.sum(np.abs(a) * sb)
    return v, s


def _quot(a, sa, b, sb):
    q = a / b
    aq, ab = abs(q), abs(b)
    return q, sa / ab + aq * sb / ab + aq


def _axpy(d, sd, c, sc, v):
    """d + c v with the scale of d, of c, and the rounding of the result"""
    r = d + c * v
    return r, sd + np.abs(v) * sc + np.abs(r) + LD(SUB / U)


def newest_first(end, bound):
    """ring slots of the `bound` newest pairs when the newest sits in slot end - 1"""
    return [(end - 1 - i) % M for i in range(bound)]


def two_loop(g, S, Y, ys_ring, s_ring, end, bound, ys, s_ys, yy, s_yy, mutant=None):
    """the recursion on a ring that already holds the new pair (in slot end - 1).  ys_ring, s_ring: longdouble values
    and scales of the ring's ys; ys, yy of the newest pair (with scales) set H0.  mutant (tests of the rule's
    sharpness) names one way a broken implementation would go wrong."""
    g = _ld(g)
    S, Y = [_ld(v) for v in S], [_ld(v) for v in Y]
    js = newest_first(end, bound - 1 if mutant == "bound_minus_1" else bound)
    first = js[::-1] if mutant == "order" else js
    d, sd = -g, np.zeros_like(g)
    alpha, s_alpha, araw, s_araw = {}, {}, {}, {}
    nan = LD("nan")

    def lost(i):
        """a non-finite coefficient makes every component of d non-finite (inf * 0 is NaN too): the rest of the
        recursion is NaN (computed directly: extended-precision NaN arithmetic is slow)"""
        for j in first[i:]:
            araw.setdefault(j, nan)
            s_araw.setdefault(j, nan)
        return dict(d=np.full(g.shape, nan, dtype=LD), s_d=np.full(g.shape, nan, dtype=LD), alpha=araw,
                    s_alpha=s_araw, dg=nan, s_dg=nan)

    with np.errstate(all="ignore"):
        for i, j in enumerate(first):
            araw[j], s_araw[j] = _dot(S[j], d, sd)
            alpha[j], s_alpha[j] = _quot(araw[j], s_araw[j], ys_ring[j], s_ring[j])
            if not np.isfinite(alpha[j]):
                return lost(i + 1)
            d, sd = _axpy(d, sd, -alpha[j], s_alpha[j], Y[j])
        if mutant == "gamma_oldest":
            o = js[-1]
            yyo, s_yyo = _dot(Y[o], Y[o])
            h0, s_h0 = _quot(ys_ring[o], s_ring[o], yyo, s_yyo)
        else:
            h0, s_h0 = _quot(ys, s_ys, yy, s_yy)
        if not np.isfinite(h0):
            return lost(len(first))
        d0 = d
        d = d0 * h0
        sd = sd * abs(h0) + np.abs(d0) * s_h0 + np.abs(d) + LD(SUB / U)
        for j in first[::-1]:
            braw, s_braw = _dot(Y[j], d, sd)
            den = (j + 1) % M if mutant == "beta_slot" else j
            beta, s_beta = _quot(braw, s_braw, ys_ring[den], s_ring[den])
            c = (beta - alpha[j]) if mutant == "sign" else (alpha[j] - beta)
            sc = s_alpha[j] + s_beta + abs(c)
            if not np.isfinite(c):
                return lost(len(first))
            d, sd = _axpy(d, sd, c, sc, S[j])
        dg, s_dg = _dot(g, d, sd)
    return dict(d=d, s_d=sd, alpha=araw, s_alpha=s_araw, dg=dg, s_dg=s_dg)


def update(x, xp, g, gp, S, Y, ys_ring, end_old, bound, mutant=None):
    """One update from the state the device is given: fp64 x, xp, g, gp (n), ring S, Y (m x n) and ys_ring (m) of the
    older pairs.  Returns s, y (fp64: the device must match them bit for bit), S, Y after the update, and longdouble ys,
    yy, alpha {slot: raw s_j . d}, d, dg, each with its scale s_<name>.  mutant "end_not_advanced": the recursion
    starts from slot end_old instead of end_old + 1."""
    x, xp, g, gp = (np.asarray(v, dtype=np.float64) for v in (x, xp, g, gp))
    s, y = x - xp, g - gp
    S2, Y2 = np.array(S, dtype=np.float64, copy=True), np.array(Y, dtype=np.float64, copy=True)
    S2[end_old], Y2[end_old] = s, y
    sl, yl = _ld(s), _ld(y)
    ys, s_ys = _dot(yl, sl)
    yy, s_yy = _dot(yl, yl)
    ring, s_ring = _ld(ys_ring).copy(), np.zeros(M, dtype=LD)
    ring[end_old], s_ring[end_old] = ys, s_ys
    end = end_old if mutant == "end_not_advanced" else (end_old + 1) % M
    out = two_loop(g, S2, Y2, ring, s_ring, end, bound, ys, s_ys, yy, s_yy,
                   mutant=None if mutant == "end_not_advanced" else mutant)
    out.update(s=s, y=y, S=S2, Y=Y2, ys=ys, s_ys=s_ys, yy=yy, s_yy=s_yy)
    return out


def gram(g, S, Y, end_old, bound, ys_ring):
    """The coefficient-space engine's arithmetic on a ring that already holds the new pair in slot end_old (reachable
    states only: the valid slots are [0, bound)).  The Gram diagonal s_j . y_j of the older pairs is ys_ring[j], exact
    (in a minimisation it is the very value the ring holds); the other entries are exact dot products with their
    scales.  Returns d, dg, ys, yy with the Gram engine's own scales."""
    n = np.asarray(g).size
    basis = [_ld(v) for v in S] + [_ld(v) for v in Y] + [_ld(g)]
    Gm = np.empty((GRAM_B, GRAM_B), dtype=LD)
    sG = np.empty((GRAM_B, GRAM_B), dtype=LD)
    for a in range(GRAM_B):
        for b in range(a, GRAM_B):
            Gm[a, b], sG[a, b] = _dot(basis[a], basis[b])
            Gm[b, a], sG[b, a] = Gm[a, b], sG[a, b]
    for j in range(bound):
        if j != end_old:
            Gm[j, M + j] = Gm[M + j, j] = LD(float(ys_ring[j]))
            sG[j, M + j] = sG[M + j, j] = 0
    c, sc = np.zeros(GRAM_B, dtype=LD), np.zeros(GRAM_B, dtype=LD)
    c[-1] = -1

    def dotq(row):
        t = c * Gm[row]
        return np.sum(t), np.sum(np.abs(c) * sG[row] + sc * np.abs(Gm[row])) + GRAM_B * np.sum(np.abs(t))

    js = newest_first((end_old + 1) % M, bound)
    alpha, s_alpha = {}, {}
    with np.errstate(all="ignore"):
        for j in js:
            q, sq = dotq(j)
            alpha[j], s_alpha[j] = _quot(q, sq, Gm[j, M + j], sG[j, M + j])
            c[M + j] -= alpha[j]
            sc[M + j] += s_alpha[j] + abs(c[M + j])
        i_s, i_y = end_old, M + end_old
        h0, s_h0 = _quot(Gm[i_s, i_y], sG[i_s, i_y], Gm[i_y, i_y], sG[i_y, i_y])
        c0 = c.copy()
        c = c0 * h0
        sc = sc * abs(h0) + np.abs(c0) * s_h0 + np.abs(c)
        for j in js[::-1]:
            q, sq = dotq(M + j)
            beta, s_beta = _quot(q, sq, Gm[j, M + j], sG[j, M + j])
            c[j] += alpha[j] - beta
            sc[j] += s_alpha[j] + s_beta + abs(alpha[j] - beta) + abs(c[j])
        dg, s_dg = dotq(GRAM_B - 1)
        used = [k for k in range(GRAM_B) if k == GRAM_B - 1 or k % M < bound]
        d = np.zeros(n, dtype=LD)
        sd = np.zeros(n, dtype=LD)
        for k in used:
            d = d + c[k] * basis[k]
            sd = sd + GRAM_B * np.abs(c[k] * basis[k]) + sc[k] * np.abs(basis[k])
        sd = sd + LD(SUB / U)
    return dict(d=d, s_d=sd, dg=dg, s_dg=s_dg, ys=Gm[i_s, i_y], s_ys=sG[i_s, i_y], yy=Gm[i_y, i_y], s_yy=sG[i_y, i_y])


def ratio(got, ref, scale):
    """max_k |got_k - ref_k| / (u scale_k) over the components where ref is finite; inf when got is finite in other
    components than ref (a kernel must be non-finite exactly where the reference is)"""
    got = np.atleast_1d(np.asarray(got, dtype=np.float64)).ravel()
    ref, scale = np.atleast_1d(np.asarray(ref, dtype=LD)).ravel(), np.atleast_1d(np.asarray(scale, dtype=LD)).ravel()
    if got.shape != ref.shape:
        raise ValueError("shape mismatch %s vs %s" % (got.shape, ref.shape))
    fin = np.isfinite(ref)
    if np.any(np.isfinite(got) != fin):
        return float("inf")
    err = np.abs(got[fin].astype(LD) - ref[fin])
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(err == 0, LD(0), err / (LD(U) * scale[fin]))
    return float(np.max(q)) if q.size else 0.0
