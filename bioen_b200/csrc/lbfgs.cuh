// lbfgs.cuh -- device-resident L-BFGS with liblbfgs 1.10 semantics.
//
// What the reference does (third-party/liblbfgs-1.10/lib/lbfgs.c, driven by c_bioen_kernels_logw.c:581-669 and
// c_bioen_kernels_forces.c:574-662): all vectors live in host memory, every dot product is a sequential host
// loop, every trial point calls back into the OpenMP kernels.
//
// Here: x, g, xp, gp, d and the m = 6 (s, y) pairs live in HBM for the whole minimisation.  The trial point
// x = xp + stp*d is formed inside the first evaluation kernel, g.d / ||g||^2 / ||x||^2 come out of the last
// one, the (s, y) update and the two-loop recursion are 2*bound+2 fused kernels chained through the device
// scalar file.  The *scalar* state machine of liblbfgs (line searches, stop tests, return codes) is kept on
// the host, bit for bit in the same order of tests, and costs one 512-byte read-back per trial point (plus one
// per iteration for the new direction's slope g.d).
// With N sharded across GPUs the vector kernels see the local slice and the raw dot products are
// all-reduced in-stream (forces: the M-dimensional state is replicated, nothing to reduce).
#pragma once
#include <cmath>
#include <cstdio>
#include <vector>

#include "context.cuh"

namespace bioen {

enum {
    LBFGS_SUCCESS = 0,
    LBFGS_STOP = 1,
    LBFGS_ALREADY_MINIMIZED = 2,
    LBFGSERR_UNKNOWNERROR = -1024,
    LBFGSERR_LOGICERROR,
    LBFGSERR_OUTOFMEMORY,
    LBFGSERR_CANCELED,
    LBFGSERR_INVALID_N,
    LBFGSERR_INVALID_N_SSE,
    LBFGSERR_INVALID_X_SSE,
    LBFGSERR_INVALID_EPSILON,
    LBFGSERR_INVALID_TESTPERIOD,
    LBFGSERR_INVALID_DELTA,
    LBFGSERR_INVALID_LINESEARCH,
    LBFGSERR_INVALID_MINSTEP,
    LBFGSERR_INVALID_MAXSTEP,
    LBFGSERR_INVALID_FTOL,
    LBFGSERR_INVALID_WOLFE,
    LBFGSERR_INVALID_GTOL,
    LBFGSERR_INVALID_XTOL,
    LBFGSERR_INVALID_MAXLINESEARCH,
    LBFGSERR_INVALID_ORTHANTWISE,
    LBFGSERR_INVALID_ORTHANTWISE_START,
    LBFGSERR_INVALID_ORTHANTWISE_END,
    LBFGSERR_OUTOFINTERVAL,
    LBFGSERR_INCORRECT_TMINMAX,
    LBFGSERR_ROUNDING_ERROR,
    LBFGSERR_MINIMUMSTEP,
    LBFGSERR_MAXIMUMSTEP,
    LBFGSERR_MAXIMUMLINESEARCH,
    LBFGSERR_MAXIMUMITERATION,
    LBFGSERR_WIDTHTOOSMALL,
    LBFGSERR_INVALIDPARAMETERS,
    LBFGSERR_INCREASEGRADIENT
};

struct LbfgsParams {  // lbfgs.h lbfgs_parameter_t with _defparam (lbfgs.c:113-118)
    int m = 6;
    double epsilon = 1e-5;
    int past = 0;
    double delta = 1e-5;
    int max_iterations = 0;
    int linesearch = 0;
    int max_linesearch = 40;
    double min_step = 1e-20, max_step = 1e20, ftol = 1e-4, wolfe = 0.9, gtol = 0.9, xtol = 1e-16;
};

struct LbfgsStats {
    int iterations = 0, evaluations = 0;
    int gradients_skipped = 0;   // trials whose gradient pass was not needed (sufficient-decrease test failed)
    double seconds = 0.0;
    double gpu_eval_ms = 0.0, gpu_update_ms = 0.0;   // BIOEN_B200_TRACE=1
};

inline int lbfgs_check_params(int n, const LbfgsParams& p) {  // lbfgs.c:286-364
    if (n <= 0) return LBFGSERR_INVALID_N;
    if (p.epsilon < 0.) return LBFGSERR_INVALID_EPSILON;
    if (p.past < 0) return LBFGSERR_INVALID_TESTPERIOD;
    if (p.delta < 0.) return LBFGSERR_INVALID_DELTA;
    if (p.min_step < 0.) return LBFGSERR_INVALID_MINSTEP;
    if (p.max_step < p.min_step) return LBFGSERR_INVALID_MAXSTEP;
    if (p.ftol < 0.) return LBFGSERR_INVALID_FTOL;
    if (p.linesearch == 2 || p.linesearch == 3) {
        if (p.wolfe <= p.ftol || 1. <= p.wolfe) return LBFGSERR_INVALID_WOLFE;
    }
    if (p.gtol < 0.) return LBFGSERR_INVALID_GTOL;
    if (p.xtol < 0.) return LBFGSERR_INVALID_XTOL;
    if (p.max_linesearch <= 0) return LBFGSERR_INVALID_MAXLINESEARCH;
    if (p.linesearch < 0 || p.linesearch > 3) return LBFGSERR_INVALID_LINESEARCH;
    if (p.m <= 0 || p.m > 16) return LBFGSERR_INVALIDPARAMETERS;
    return 0;
}

// ---- More-Thuente helpers: cubic / quadratic interpolation (lbfgs.c:1021-1094) -------------------------
namespace mt {
inline double max3(double a, double b, double c) { return std::fmax(std::fmax(a, b), c); }
inline double cubic(double u, double fu, double du, double v, double fv, double dv) {
    const double d = v - u, theta = (fu - fv) * 3 / d + du + dv;
    const double s = max3(std::fabs(theta), std::fabs(du), std::fabs(dv)), a = theta / s;
    double gamma = s * std::sqrt(a * a - (du / s) * (dv / s));
    if (v < u) gamma = -gamma;
    const double p = gamma - du + theta, q = gamma - du + gamma + dv;
    return u + (p / q) * d;
}
inline double cubic2(double u, double fu, double du, double v, double fv, double dv, double xmin, double xmax) {
    const double d = v - u, theta = (fu - fv) * 3 / d + du + dv;
    const double s = max3(std::fabs(theta), std::fabs(du), std::fabs(dv)), a = theta / s;
    double gamma = s * std::sqrt(std::fmax(0.0, a * a - (du / s) * (dv / s)));
    if (u < v) gamma = -gamma;
    const double p = gamma - dv + theta, q = gamma - dv + gamma + du, r = p / q;
    if (r < 0. && gamma != 0.) return v - r * d;
    return a < 0 ? xmax : xmin;
}
inline double quad(double u, double fu, double du, double v, double fv) {
    const double a = v - u;
    return u + du / ((fu - fv) / a + du) / 2 * a;
}
inline double quad2(double u, double du, double v, double dv) {
    const double a = u - v;
    return v + dv / (dv - du) * a;
}
// update_trial_interval (lbfgs.c:1125-1292)
inline int update(double& x, double& fx, double& dx, double& y, double& fy, double& dy, double& t, double ft,
                  double dt, double tmin, double tmax, int& brackt) {
    int bound;
    const bool dsign = (dt * (dx / std::fabs(dx)) < 0.);
    double mc, mq, newt;
    if (brackt) {
        if (t <= std::fmin(x, y) || std::fmax(x, y) <= t) return LBFGSERR_OUTOFINTERVAL;
        if (0. <= dx * (t - x)) return LBFGSERR_INCREASEGRADIENT;
        if (tmax < tmin) return LBFGSERR_INCORRECT_TMINMAX;
    }
    if (fx < ft) {
        brackt = 1; bound = 1;
        mc = cubic(x, fx, dx, t, ft, dt);
        mq = quad(x, fx, dx, t, ft);
        newt = (std::fabs(mc - x) < std::fabs(mq - x)) ? mc : mc + 0.5 * (mq - mc);
    } else if (dsign) {
        brackt = 1; bound = 0;
        mc = cubic(x, fx, dx, t, ft, dt);
        mq = quad2(x, dx, t, dt);
        newt = (std::fabs(mc - t) > std::fabs(mq - t)) ? mc : mq;
    } else if (std::fabs(dt) < std::fabs(dx)) {
        bound = 1;
        mc = cubic2(x, fx, dx, t, ft, dt, tmin, tmax);
        mq = quad2(x, dx, t, dt);
        if (brackt) newt = (std::fabs(t - mc) < std::fabs(t - mq)) ? mc : mq;
        else newt = (std::fabs(t - mc) > std::fabs(t - mq)) ? mc : mq;
    } else {
        bound = 0;
        if (brackt) newt = cubic(t, ft, dt, y, fy, dy);
        else if (x < t) newt = tmax;
        else newt = tmin;
    }
    if (fx < ft) {
        y = t; fy = ft; dy = dt;
    } else {
        if (dsign) { y = x; fy = fx; dy = dx; }
        x = t; fx = ft; dx = dt;
    }
    if (tmax < newt) newt = tmax;
    if (newt < tmin) newt = tmin;
    if (brackt && bound) {
        mq = x + 0.66 * (y - x);
        if (x < y) { if (mq < newt) newt = mq; }
        else { if (newt < mq) newt = mq; }
    }
    t = newt;
    return 0;
}
}  // namespace mt

// ------------------------------------------------------------------------------------------------
// line searches of liblbfgs as resumable state machines: prepare() -> step to evaluate, update(f, dg) -> verdict
// (the arithmetic and order of tests of lbfgs.c:645-734 and 812-1001).  Used by the single-problem driver below,
// by the lockstep theta scan (batched.cuh), and -- host-only -- by the CPU test hook bioen_b200_selftest_linesearch.
// ------------------------------------------------------------------------------------------------
struct LineSearchState {
    const LbfgsParams* prm = nullptr;
    int count = 0;
    double finit = 0, dginit = 0, stp = 0;
    // More-Thuente
    int brackt = 0, stage1 = 1, uinfo = 0;
    double width = 0, prev_width = 0, stx = 0, sty = 0, fx = 0, fy = 0, dgx = 0, dgy = 0, stmin = 0, stmax = 0;

    void start(const LbfgsParams& p, double f, double dg, double step) {
        prm = &p; count = 0; finit = f; dginit = dg; stp = step;
        brackt = 0; stage1 = 1; uinfo = 0;
        width = p.max_step - p.min_step; prev_width = 2.0 * width;
        stx = sty = 0.0; fx = fy = f; dgx = dgy = dg;
    }
    void set_slope(double dg) { dginit = dg; dgx = dgy = dg; }
    // step length of the next trial
    double prepare() {
        if (prm->linesearch != 0) return stp;
        if (brackt) { stmin = std::fmin(stx, sty); stmax = std::fmax(stx, sty); }
        else { stmin = stx; stmax = stp + 4.0 * (stp - stx); }
        if (stp < prm->min_step) stp = prm->min_step;
        if (prm->max_step < stp) stp = prm->max_step;
        if ((brackt && ((stp <= stmin || stmax <= stp) || prm->max_linesearch <= count + 1 || uinfo != 0)) ||
            (brackt && (stmax - stmin <= prm->xtol * stmax)))
            stp = stx;
        return stp;
    }
    // backtracking searches look at the slope of a trial only when its value passes the sufficient-decrease
    // test (lbfgs.c:683-709), so the caller may skip the gradient of a trial that fails it
    bool needs_slope(double f) const {
        if (prm->linesearch == 0) return true;
        const double dgtest = prm->ftol * dginit;
        return !(f > finit + stp * dgtest);
    }
    // 0: another trial needed (stp updated); > 0: accepted after that many trials; < 0: liblbfgs error code
    int update(double f, double dg) {
        const LbfgsParams& p = *prm;
        ++count;
        if (p.linesearch != 0) {
            double w;
            if (!needs_slope(f)) {
                w = 0.5;
            } else {
                if (p.linesearch == 1) return count;
                if (dg < p.wolfe * dginit) {
                    w = 2.1;
                } else {
                    if (p.linesearch == 2) return count;
                    if (dg > -p.wolfe * dginit) w = 0.5;
                    else return count;
                }
            }
            if (stp < p.min_step) return LBFGSERR_MINIMUMSTEP;
            if (stp > p.max_step) return LBFGSERR_MAXIMUMSTEP;
            if (p.max_linesearch <= count) return LBFGSERR_MAXIMUMLINESEARCH;
            stp *= w;
            return 0;
        }
        const double dgtest = p.ftol * dginit;
        const double ftest1 = finit + stp * dgtest;
        if (brackt && ((stp <= stmin || stmax <= stp) || uinfo != 0)) return LBFGSERR_ROUNDING_ERROR;
        if (stp == p.max_step && f <= ftest1 && dg <= dgtest) return LBFGSERR_MAXIMUMSTEP;
        if (stp == p.min_step && (ftest1 < f || dgtest <= dg)) return LBFGSERR_MINIMUMSTEP;
        if (brackt && (stmax - stmin) <= p.xtol * stmax) return LBFGSERR_WIDTHTOOSMALL;
        if (p.max_linesearch <= count) return LBFGSERR_MAXIMUMLINESEARCH;
        if (f <= ftest1 && std::fabs(dg) <= p.gtol * (-dginit)) return count;
        if (stage1 && f <= ftest1 && std::fmin(p.ftol, p.gtol) * dginit <= dg) stage1 = 0;
        if (stage1 && ftest1 < f && f <= fx) {
            double fm = f - stp * dgtest, fxm = fx - stx * dgtest, fym = fy - sty * dgtest;
            double dgm = dg - dgtest, dgxm = dgx - dgtest, dgym = dgy - dgtest;
            uinfo = mt::update(stx, fxm, dgxm, sty, fym, dgym, stp, fm, dgm, stmin, stmax, brackt);
            fx = fxm + stx * dgtest;
            fy = fym + sty * dgtest;
            dgx = dgxm + dgtest;
            dgy = dgym + dgtest;
        } else {
            uinfo = mt::update(stx, fx, dgx, sty, fy, dgy, stp, f, dg, stmin, stmax, brackt);
        }
        if (brackt) {
            if (0.66 * prev_width <= std::fabs(sty - stx)) stp = stx + 0.5 * (sty - stx);
            prev_width = width;
            width = std::fabs(sty - stx);
        }
        return 0;
    }
};

// ------------------------------------------------------------------------------------------------
// liblbfgs' iteration loop for one problem (lbfgs.c:412-598 without the vector arithmetic): the stop tests in their
// order, the `past` ring of objective values and the position in the (s, y) ring.  Lbfgs::run drives one problem with
// it, ThetaScan::run (batched.cuh) K problems in lockstep; each enqueues its own trials, updates and reverts.
// ------------------------------------------------------------------------------------------------
struct LbfgsIteration {
    const LbfgsParams* prm = nullptr;
    int k = 1, end = 0, iterations = 0;
    double fx = 0.0;
    std::vector<double> pf;     // objective of the last `past` iterations
    LineSearchState ls;         // the running search
    bool slope_known = false;   // false: ls waits for the slope g.d of the new direction (ls.set_slope)

    // h: scalar file of the start point.  0: the first search is started (d = -g, step 1/||g||, slope -||g||^2);
    // otherwise LBFGS_ALREADY_MINIMIZED.
    int first_point(const LbfgsParams& p, const double* h) {
        prm = &p;
        fx = h[SC_F];
        pf.assign(p.past > 0 ? p.past : 0, 0.0);
        if (!pf.empty()) pf[0] = fx;
        double xnorm = std::sqrt(h[SC_XNORM2]);
        const double gnorm = std::sqrt(h[SC_GNORM2]);
        if (xnorm < 1.0) xnorm = 1.0;
        if (gnorm / xnorm <= p.epsilon) return LBFGS_ALREADY_MINIMIZED;
        ls.start(p, fx, -h[SC_GNORM2], 1.0 / gnorm);
        slope_known = true;
        return 0;
    }

    // the search ended with `verdict` (!= 0); h: scalar file of its last trial.  true: the new pair goes to ring slot
    // `slot`, the two-loop recursion runs over `bound` pairs, and the next search is started with step 1 and an
    // unknown slope.  false: the minimisation ends with the liblbfgs code `code`; on a failed search (verdict < 0) the
    // caller reverts x and g.
    bool search_finished(int verdict, const double* h, int& slot, int& bound, int& code) {
        // a failed search leaves its last trial's f in fx (lbfgs.c:466-481), except on a positive initial slope,
        // where liblbfgs returns before the first trial
        if (verdict != LBFGSERR_INCREASEGRADIENT) fx = h[SC_F];
        code = verdict;
        if (verdict < 0) return false;
        ++iterations;   // the progress callback (c_bioen_kernels_logw.c:565-576)
        double xnorm = std::sqrt(h[SC_XNORM2]);
        const double gnorm = std::sqrt(h[SC_GNORM2]);
        if (xnorm < 1.0) xnorm = 1.0;
        if (gnorm / xnorm <= prm->epsilon) {
            code = LBFGS_SUCCESS;
            return false;
        }
        if (!pf.empty()) {
            if (prm->past <= k && (pf[k % prm->past] - fx) / fx < prm->delta) {
                code = LBFGS_STOP;
                return false;
            }
            pf[k % prm->past] = fx;
        }
        if (prm->max_iterations != 0 && prm->max_iterations < k + 1) {
            code = LBFGSERR_MAXIMUMITERATION;
            return false;
        }
        code = 0;
        slot = end;
        bound = (prm->m <= k) ? prm->m : k;
        ++k;
        end = (end + 1) % prm->m;
        ls.start(*prm, fx, 0.0, 1.0);
        slope_known = false;
        return true;
    }
};

// ------------------------------------------------------------------------------------------------
// The two-loop recursion of lbfgs.c:572-598 over the `bound` newest pairs of an m-slot ring whose newest pair sits in
// slot end - 1, as 2*bound + 1 fused steps (k_lbfgs_twoloop, kb_twoloop).  Step t does
//     d <- (init ? -g : d) + coef * u ;  d *= sc[SC_YS] / sc[SC_YY] when scale ;  sc[out] = v . d
// with coef = csign * sc[c_num] / sc[c_den], minus sc[c2_num] / sc[c_den] when c2_num >= 0.  The alpha ring holds the
// raw s_j . d, SC_BETA / SC_BETA2 alternately the raw y_j . d; the last step leaves g . d in SC_DGINIT.
// ------------------------------------------------------------------------------------------------
enum { TL_NONE = 0, TL_S = 1, TL_Y = 2, TL_G = 3 };   // a step's vectors: none, s_slot, y_slot, the gradient

struct TwoLoopStep {
    int init;
    int u_kind, u_slot;       // u_kind TL_NONE: no axpy
    int v_kind, v_slot;       // v_kind TL_NONE: no dot
    int c_num, c_den, csign;
    int c2_num;               // -1: unused
    int scale;
    int out;
};

inline TwoLoopStep two_loop_step(int t, int end, int bound, int m) {
    auto js = [&](int i) { return ((end - 1 - i) % m + m) % m; };   // newest ... oldest
    TwoLoopStep st{};
    st.c2_num = -1;
    if (t == 0) {                   // d = -g ; alpha_raw[j0] = s_j0 . d
        st.init = 1;
        st.v_kind = TL_S; st.v_slot = js(0); st.out = SC_ALPHA0 + js(0);
    } else if (t <= bound) {        // d -= alpha_j y_j ; then either the next alpha, or (last) the H0 scaling and the first beta
        const int i = t - 1;
        st.u_kind = TL_Y; st.u_slot = js(i);
        st.c_num = SC_ALPHA0 + js(i); st.c_den = SC_YS0 + js(i); st.csign = -1;
        if (i + 1 < bound) {
            st.v_kind = TL_S; st.v_slot = js(i + 1); st.out = SC_ALPHA0 + js(i + 1);
        } else {
            st.scale = 1;
            st.v_kind = TL_Y; st.v_slot = js(i); st.out = SC_BETA;
        }
    } else {                        // d += (alpha_j - beta_j) s_j ; then the next beta, or (last) g.d
        const int i = 2 * bound - t;              // bound-1 ... 0
        const bool odd = (t - bound - 1) & 1;     // the beta slots alternate
        st.u_kind = TL_S; st.u_slot = js(i);
        st.c_num = SC_ALPHA0 + js(i); st.c_den = SC_YS0 + js(i); st.csign = 1;
        st.c2_num = odd ? SC_BETA2 : SC_BETA;
        if (i > 0) {
            st.v_kind = TL_Y; st.v_slot = js(i - 1); st.out = odd ? SC_BETA : SC_BETA2;
        } else {
            st.v_kind = TL_G; st.out = SC_DGINIT;
        }
    }
    return st;
}

class Lbfgs {
   public:
    Context& C;
    const bool forces;   // false: log-weights (n = N, sharded when C.nranks > 1); true: forces (n = M, replicated)
    const int n;
    LbfgsParams prm;
    int verbose = 0;
    LbfgsStats stats;
    bool trace = false;                                   // BIOEN_B200_TRACE: GPU time of evaluations vs updates
    cudaEvent_t tev[3] = {nullptr, nullptr, nullptr};
    ~Lbfgs() {
        for (auto& e : tev) if (e) cudaEventDestroy(e);
    }

    double *x = nullptr, *g = nullptr, *xp = nullptr, *gp = nullptr, *d = nullptr;
    std::vector<double*> S, Yv;
    int vec_blocks;
    bool reduce;

    Lbfgs(Context& ctx, bool is_forces, const LbfgsParams& p)
        : C(ctx), forces(is_forces), n(is_forces ? ctx.M : ctx.N), prm(p) {
        vec_blocks = is_forces ? ctx.vec_blocks_m : ctx.vec_blocks_n;
        reduce = (!is_forces) && ctx.nranks > 1;
    }

    // x_dev (device, n doubles): start point on entry, end point on exit.  Returns the liblbfgs code.
    int run(double* x_dev, double* fx_out) {
        NvtxRange nvtx("bioen:lbfgs");
        x = x_dev;
        trace = getenv("BIOEN_B200_TRACE") != nullptr;
        int ret = lbfgs_check_params(n, prm);
        if (ret) { *fx_out = 0.0; return ret; }
        bind_store();
        const double* h = C.h_sc;

        // initial evaluation (lbfgs.c:412)
        eval(nullptr, nullptr, 0.0, nullptr);
        C.fetch_scalars();
        LbfgsIteration it;
        ret = it.first_point(prm, h);
        if (ret) { *fx_out = it.fx; return ret; }
        k_axpby<<<vec_blocks, kVecThreads, 0, C.stream>>>(n, -1.0, g, 0.0, nullptr, d);   // d = -g
        C.d2d(xp, x, n);
        C.d2d(gp, g, n);

        for (;;) {
            NvtxRange nvtx_it("bioen:lbfgs_iteration");
            const int verdict = linesearch(it);
            int slot = 0, bound = 0;
            const bool more = it.search_finished(verdict, h, slot, bound, ret);
            stats.iterations = it.iterations;
            if (verdict > 0 && verbose && it.iterations % 1000 == 0) printf("\t\tOpt Iteration %d\n", it.iterations);
            if (verdict < 0) {
                // revert to the previous point (lbfgs.c:475-481)
                C.d2d(x, xp, n);
                C.d2d(g, gp, n);
                C.sync();
            }
            if (!more) break;
            // s, y, ys, yy; xp <- x, gp <- g (lbfgs.c:543-555, 462-463); then the two-loop recursion
            update_direction(slot, bound, prm.m);
        }
        *fx_out = it.fx;
        return ret;
    }

    // point g, xp, gp, d and the (s, y) ring at the context's L-BFGS store (bioen_b200_debug_read 5 reads it back):
    // [g | xp | gp | d | s_0 .. s_{m-1} | y_0 .. y_{m-1}], each n rounded up to 16.  The work vectors are reused by the
    // next minimisation of the same size (every vector is written before it is read, so no clearing is needed); the
    // Gram matrix of the coefficient-space update starts from zero.
    void bind_store() {
        const int m = prm.m;
        const size_t np = ((size_t)n + 15) & ~(size_t)15;
        C.lbfgs_store.reserve(np * (4 + 2 * (size_t)m));
        g = C.lbfgs_store.p; xp = g + np; gp = xp + np; d = gp + np;
        S.resize(m); Yv.resize(m);
        for (int i = 0; i < m; ++i) { S[i] = d + np * (1 + i); Yv[i] = d + np * (1 + m + i); }
        if (gram_mode()) {
            C.lbfgs_gram.reserve(kGramB * kGramB + kGramB + 3);
            C.lbfgs_gram_partials.reserve((size_t)vec_blocks * kGramK + 8);
            CUDA_CHECK(cudaMemsetAsync(C.lbfgs_gram.p, 0, (kGramB * kGramB + kGramB) * sizeof(double), C.stream));
        }
    }

    // the new pair into ring slot end_old and the two-loop recursion over `bound` pairs, on whichever engine the
    // context selects (Gram, small, multi-kernel).  Also bioen_b200_selftest_lbfgs_update.
    void update_direction(int end_old, int bound, int m) {
        if (gram_mode()) enqueue_update_gram(end_old, bound);
        else if (small_mode()) enqueue_update_small(end_old, bound);
        else enqueue_update(end_old, bound, m);
    }

    bool gram_mode() const {
        // sharded runs need the in-kernel exchange (the peer-memory path); m is liblbfgs' default 6
        return C.options.lbfgs_gram_opt && prm.m == kGramM && (!reduce || C.fuse_exchange());
    }
    // small problems (n <= 1024): pair + two-loop recursion as ONE single-CTA kernel (k_lbfgs_update_small)
    bool small_mode() const {
        return C.options.lbfgs_small_opt && n <= kSmallUpdateMaxN && prm.m == kSmallUpdateM && !reduce;
    }

   private:
    // enqueue one f+g evaluation at x (= xp + stp*dir when xp_ given); dg direction optional
    // returns true when h_sc already holds everything the caller will read (objective-only trial)
    bool eval(const double* xp_, const double* dir, double stp, const double* ddir,
              const LineSearchState* ls = nullptr) {
        bool fetched = false;
        if (trace) {
            if (!tev[0]) for (auto& e : tev) cudaEventCreate(&e);
            cudaEventRecord(tev[2], C.stream);          // end of the previous update phase
            if (stats.evaluations > 0) {
                cudaEventSynchronize(tev[2]);
                float a = 0.f, b = 0.f;
                cudaEventElapsedTime(&a, tev[0], tev[1]);
                cudaEventElapsedTime(&b, tev[1], tev[2]);
                stats.gpu_eval_ms += a;
                stats.gpu_update_ms += b;
            }
            cudaEventRecord(tev[0], C.stream);
        }
        if (!ls) {
            if (forces) C.forces_eval(x, xp_, dir, stp, g, ddir);
            else C.logw_eval(x, xp_, dir, stp, g, ddir);
        } else {
            // line-search trial: the objective first (one pass over Y); the gradient pass only if the search will
            // look at the slope.  A trial that fails the sufficient-decrease test is discarded by liblbfgs without
            // its gradient ever being read (the next trial overwrites it; on failure x and g are restored), so
            // skipping it changes no result.
            if (forces) C.forces_eval_f(x, xp_, dir, stp);
            else C.logw_eval_f(x, xp_, dir, stp);
            C.fetch_scalars();
            if (take_spec_slope()) {
                ++stats.evaluations;
                return true;
            }
            if (ls->needs_slope(C.h_sc[SC_F])) {
                if (forces) C.forces_eval_g(g, ddir);
                else C.logw_eval_g(x, g, ddir);
            } else {
                ++stats.gradients_skipped;
                fetched = true;
            }
        }
        if (trace) cudaEventRecord(tev[1], C.stream);
        ++stats.evaluations;
        return fetched;
    }

    // one line-search trial at x = xp + stp*d: evaluation + scalar read-back (host side of lbfgs.c:645-1001)
    void trial(double stp, const LineSearchState& ls) {
        // More-Thuente reads the slope of every trial: plain f+g evaluation, one read-back
        // (not on the slice kernel: there a combined f+g launch costs ~4 us more than the objective alone, less than the
        // second launch and host round trip the split costs the ~87 % of trials whose gradient IS read)
        if (!eval(xp, d, stp, d, (prm.linesearch != 0 && C.options.lazy_gradient && !C.slice_ok()) ? &ls : nullptr)) {
            C.fetch_scalars();
            take_spec_slope();
        }
    }
    // first trial of a search whose initial slope was not fetched beforehand: it is in the scalar file just read
    bool spec_slope = false, spec_bad = false;
    LineSearchState* spec_ls = nullptr;
    bool take_spec_slope() {
        if (!spec_slope) return false;
        spec_slope = false;
        const double dg0 = C.h_sc[SC_DGINIT];
        spec_ls->set_slope(dg0);
        spec_bad = 0 < dg0;
        return spec_bad;
    }

    void enqueue_update(int end_old, int bound, int m) {
        NvtxRange nvtx("bioen:lbfgs_update(pair+two_loop)");
        const bool fused = reduce && C.fuse_exchange();
        PairArgs a{n, x, g, xp, gp, S[end_old], Yv[end_old], end_old, C.red_partials.p, C.ticket.p, C.sc.p, {}};
        if (fused) a.p2p = C.p2p_dev(); else a.p2p.nranks = 1;
        k_lbfgs_pair<<<vec_blocks, kVecThreads, 0, C.stream>>>(a);
        ++C.kernels_launched;
        if (reduce && !fused) {
            C.comm->allreduce_sum(C.sc.p + SC_YS, 2, C.stream);
            C.d2d(C.sc.p + SC_YS0 + end_old, C.sc.p + SC_YS, 1);
        }
        two_loop(bound, (end_old + 1) % m, m);
    }
    // opt-in: the whole update as 2 kernels and 1 exchange (coefficient-space recursion, vector_kernels.cuh)
    void enqueue_update_gram(int end_old, int bound) {
        NvtxRange nvtx("bioen:lbfgs_update(gram)");
        GramPairArgs a{};
        a.n = n; a.x = x; a.g = g; a.xp = xp; a.gp = gp;
        for (int t = 0; t < kGramM; ++t) { a.S[t] = S[t]; a.Y[t] = Yv[t]; }
        a.end = end_old; a.bound = bound; a.gram = C.lbfgs_gram.p; a.partials = C.lbfgs_gram_partials.p;
        a.ticket = C.ticket.p; a.sc = C.sc.p;
        if (reduce && C.fuse_exchange()) a.p2p = C.p2p_dev(); else a.p2p.nranks = 1;
        k_lbfgs_gram_pair<<<vec_blocks, kVecThreads, 0, C.stream>>>(a);
        GramCombineArgs b{};
        b.n = n; b.g = g; b.coef = C.lbfgs_gram.p + kGramB * kGramB; b.bound = bound; b.d = d;
        for (int t = 0; t < kGramM; ++t) { b.S[t] = S[t]; b.Y[t] = Yv[t]; }
        k_lbfgs_combine<<<vec_blocks, kVecThreads, 0, C.stream>>>(b);
        C.kernels_launched += 2;
    }
    void enqueue_update_small(int end_old, int bound) {
        NvtxRange nvtx("bioen:lbfgs_update(small)");
        SmallUpdateArgs a{};
        a.n = n; a.x = x; a.g = g; a.xp = xp; a.gp = gp; a.d = d;
        for (int t = 0; t < kSmallUpdateM; ++t) { a.S[t] = S[t]; a.Y[t] = Yv[t]; }
        a.end = end_old; a.bound = bound; a.sc = C.sc.p;
        k_lbfgs_update_small<<<1, ((n + 31) / 32) * 32, 0, C.stream>>>(a);
        ++C.kernels_launched;
    }

    // the recursion of lbfgs.c:572-598 as the 2*bound+1 fused kernels of two_loop_step
    void two_loop(int bound, int end, int m) {
        const bool fused = reduce && C.fuse_exchange();
        auto vec = [&](int kind, int slot) -> const double* {
            return kind == TL_S ? S[slot] : kind == TL_Y ? Yv[slot] : kind == TL_G ? g : nullptr;
        };
        for (int t = 0; t <= 2 * bound; ++t) {
            const TwoLoopStep st = two_loop_step(t, end, bound, m);
            TwoLoopArgs a{};
            a.n = n; a.d = d; a.g = g; a.init = st.init;
            a.u = vec(st.u_kind, st.u_slot); a.c_num = st.c_num; a.c_den = st.c_den; a.csign = st.csign;
            a.c2_num = st.c2_num; a.c2_den = st.c_den; a.c2sign = -1.0;
            a.s_num = st.scale ? SC_YS : -1; a.s_den = SC_YY;
            a.v = vec(st.v_kind, st.v_slot); a.out = st.out;
            a.partials = C.red_partials.p; a.ticket = C.ticket.p; a.sc = C.sc.p;
            if (fused && a.v) a.p2p = C.p2p_dev(); else a.p2p.nranks = 1;
            k_lbfgs_twoloop<<<vec_blocks, kVecThreads, 0, C.stream>>>(a);
            ++C.kernels_launched;
            if (reduce && !fused && a.v) C.comm->allreduce_sum(C.sc.p + a.out, 1, C.stream);
        }
    }

    // one line search (lbfgs.c:645-734 backtracking, 812-1001 More-Thuente) driven by it.ls: every trial is one f+g
    // evaluation on the device and one 512-byte read-back.  Returns the verdict; h_sc holds the last trial's scalars.
    int linesearch(LbfgsIteration& it) {
        const double* h = C.h_sc;
        // g.d of the new direction was left in the scalar file (SC_DGINIT) by the update kernels.  The first trial
        // point xp + stp*d does not depend on it, so the trial is enqueued right behind the update and the slope
        // arrives with the trial's own scalars: one host round trip per iteration instead of two.  (The one case
        // where the slope matters beforehand -- 0 < g.d, LBFGSERR_INCREASEGRADIENT -- then costs one evaluation
        // that liblbfgs would not have made; x and g are restored by the caller as after any failed search.)
        spec_slope = !it.slope_known && C.options.lbfgs_speculative;
        if (!it.slope_known && !spec_slope) {
            C.fetch_scalars();
            it.ls.set_slope(h[SC_DGINIT]);
            it.slope_known = true;
        }
        if (it.slope_known && 0 < it.ls.dginit) return LBFGSERR_INCREASEGRADIENT;
        spec_ls = &it.ls;
        for (;;) {
            trial(it.ls.prepare(), it.ls);
            if (spec_bad) {   // the slope that came with the first trial is positive
                spec_bad = false;
                return LBFGSERR_INCREASEGRADIENT;
            }
            it.slope_known = true;
            const int verdict = it.ls.update(h[SC_F], h[SC_DG]);
            if (verdict != 0) return verdict;
        }
    }
};

}  // namespace bioen
