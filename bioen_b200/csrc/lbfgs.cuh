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
#include <chrono>
#include <cmath>
#include <cstdio>
#include <map>

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
    double gpu_eval_ms = 0.0, gpu_update_ms = 0.0, host_wait_s = 0.0;   // BIOEN_B200_TRACE=1
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
    // CUDA graphs (single-GPU runs): one graph replays a whole line-search trial (step length H2D, the
    // evaluation kernels, scalar file D2H), one graph per (ring slot, history length) replays the L-BFGS update
    // (pair kernel + two-loop recursion): ~20 launches per iteration become 2.  Results are identical (the GPU
    // test-suite passes with it), but on this driver the replays cost ~1 ms each, so it is opt-in:
    // BIOEN_B200_GRAPHS=1.
    bool use_graphs = false;
    cudaGraphExec_t g_trial = nullptr;
    long long g_trial_kernels = 0;
    std::map<int, std::pair<cudaGraphExec_t, long long>> g_update;
    ~Lbfgs() {
        if (g_trial) cudaGraphExecDestroy(g_trial);
        for (auto& kv : g_update) cudaGraphExecDestroy(kv.second.first);
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
        {
            // opt-in: measured on B200 / driver 580 the replays are SLOWER than plain launches here (config 1,
            // N=1e5 x M=500: 0.73 s vs 0.12 s to the optimum, i.e. ~1 ms per cudaGraphLaunch of these graphs)
            const char* e = getenv("BIOEN_B200_GRAPHS");
            use_graphs = C.nranks == 1 && !trace && (e && e[0] == '1');
        }
        int ret = lbfgs_check_params(n, prm);
        if (ret) { *fx_out = 0.0; return ret; }
        const int m = prm.m;
        bind_store();
        std::vector<double> pf(prm.past > 0 ? prm.past : 0);
        const double* h = C.h_sc;

        // initial evaluation (lbfgs.c:412)
        eval(nullptr, nullptr, 0.0, nullptr);
        C.fetch_scalars();
        double fx = h[SC_F];
        if (!pf.empty()) pf[0] = fx;
        double xnorm = std::sqrt(h[SC_XNORM2]), gnorm = std::sqrt(h[SC_GNORM2]);
        if (xnorm < 1.0) xnorm = 1.0;
        if (gnorm / xnorm <= prm.epsilon) { *fx_out = fx; return LBFGS_ALREADY_MINIMIZED; }
        // d = -g ; step = 1/||d|| ; dginit = g.d = -||g||^2
        k_axpby<<<vec_blocks, kVecThreads, 0, C.stream>>>(n, -1.0, g, 0.0, nullptr, d);
        double step = 1.0 / gnorm;
        double dginit = -h[SC_GNORM2];
        bool dginit_known = true;
        C.d2d(xp, x, n);
        C.d2d(gp, g, n);

        int k = 1, end = 0;
        for (;;) {
            NvtxRange nvtx_it("bioen:lbfgs_iteration");
            int ls = linesearch(fx, step, dginit, dginit_known);
            if (ls < 0) {
                // revert to the previous point (lbfgs.c:475-481)
                C.d2d(x, xp, n);
                C.d2d(g, gp, n);
                C.sync();
                ret = ls;
                break;
            }
            xnorm = std::sqrt(h[SC_XNORM2]);
            gnorm = std::sqrt(h[SC_GNORM2]);
            ++stats.iterations;  // progress callback (c_bioen_kernels_logw.c:565-576)
            if (verbose && stats.iterations % 1000 == 0) printf("\t\tOpt Iteration %d\n", stats.iterations);
            if (xnorm < 1.0) xnorm = 1.0;
            if (gnorm / xnorm <= prm.epsilon) { ret = LBFGS_SUCCESS; break; }
            if (!pf.empty()) {
                if (prm.past <= k) {
                    const double rate = (pf[k % prm.past] - fx) / fx;
                    if (rate < prm.delta) { ret = LBFGS_STOP; break; }
                }
                pf[k % prm.past] = fx;
            }
            if (prm.max_iterations != 0 && prm.max_iterations < k + 1) { ret = LBFGSERR_MAXIMUMITERATION; break; }

            // s, y, ys, yy; xp <- x, gp <- g (lbfgs.c:543-555, 462-463); then the two-loop recursion
            const int bound = (m <= k) ? m : k;
            update_direction(end, bound, m);
            ++k;
            end = (end + 1) % m;
            step = 1.0;
            dginit_known = false;  // sc[SC_DGINIT] is read at the start of the next line search
        }
        *fx_out = fx;
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
    // context selects (Gram, small, multi-kernel; CUDA graphs when enabled).  Also bioen_b200_selftest_lbfgs_update.
    void update_direction(int end_old, int bound, int m) {
        if (gram_mode()) {
            enqueue_update_gram(end_old, bound);
            return;
        }
        if (small_mode()) {
            enqueue_update_small(end_old, bound);
            return;
        }
        if (use_graphs) {
            const int key = end_old * 64 + bound;
            auto it = g_update.find(key);
            if (it == g_update.end()) {
                long long nk = 0;
                cudaGraphExec_t ex = capture([&] { enqueue_update(end_old, bound, m); }, &nk);
                if (!ex) {
                    use_graphs = false;
                    enqueue_update(end_old, bound, m);
                    return;
                }
                it = g_update.emplace(key, std::make_pair(ex, nk)).first;
            }
            CUDA_CHECK(cudaGraphLaunch(it->second.first, C.stream));
            C.kernels_launched += it->second.second;
            return;
        }
        enqueue_update(end_old, bound, m);
    }
    bool gram_mode() const {
        // sharded runs need the in-kernel exchange (the peer-memory path); m is liblbfgs' default 6
        return C.lbfgs_gram_opt && prm.m == kGramM && (!reduce || C.fuse_exchange());
    }
    // small problems (n <= 1024): pair + two-loop recursion as ONE single-CTA kernel (k_lbfgs_update_small)
    bool small_mode() const {
        return C.lbfgs_small_opt && n <= kSmallUpdateMaxN && prm.m == kSmallUpdateM && !reduce;
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

    // ---- CUDA-graph plumbing ---------------------------------------------------------------------------
    template <class F>
    cudaGraphExec_t capture(F&& enqueue, long long* kernels) {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        const long long k0 = C.kernels_launched;
        if (cudaStreamBeginCapture(C.stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        bool ok = true;
        try {
            enqueue();
        } catch (...) {
            ok = false;
        }
        if (cudaStreamEndCapture(C.stream, &graph) != cudaSuccess || !graph) ok = false;
        if (ok && cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) ok = false;
        if (graph) cudaGraphDestroy(graph);
        *kernels = C.kernels_launched - k0;
        C.kernels_launched = k0;          // nothing ran yet; replays are counted when launched
        if (!ok) {
            cudaGetLastError();
            if (exec) cudaGraphExecDestroy(exec);
            return nullptr;
        }
        return exec;
    }

    // one line-search trial at x = xp + stp*d: evaluation + scalar read-back (host side of lbfgs.c:645-1001)
    void trial(double stp, const LineSearchState& ls) {
        if (use_graphs) {
            // BIOEN_B200_GRAPHS_NOMEMCPY=1 (diagnostics): keep the two tiny copies (step length in, scalar file out)
            // OUTSIDE the graph, so that it holds kernel nodes only
            static const bool nomemcpy = getenv("BIOEN_B200_GRAPHS_NOMEMCPY") != nullptr;
            if (!g_trial) {
                g_trial = capture([&] {
                    if (!nomemcpy)
                        CUDA_CHECK(cudaMemcpyAsync(C.sc.p + SC_STP, C.h_stp, sizeof(double), cudaMemcpyHostToDevice, C.stream));
                    if (forces) C.forces_eval(x, xp, d, 0.0, g, d, C.sc.p + SC_STP);
                    else C.logw_eval(x, xp, d, 0.0, g, d, C.sc.p + SC_STP);
                    if (!nomemcpy) C.d2h(C.h_sc, C.sc.p, SC_COUNT);
                }, &g_trial_kernels);
                if (!g_trial) use_graphs = false;   // capture not possible here: plain launches from now on
            }
            if (g_trial) {
                *C.h_stp = stp;
                const auto t0 = std::chrono::steady_clock::now();
                if (nomemcpy)
                    CUDA_CHECK(cudaMemcpyAsync(C.sc.p + SC_STP, C.h_stp, sizeof(double), cudaMemcpyHostToDevice, C.stream));
                CUDA_CHECK(cudaGraphLaunch(g_trial, C.stream));
                if (nomemcpy) C.d2h(C.h_sc, C.sc.p, SC_COUNT);
                const auto t1 = std::chrono::steady_clock::now();
                C.kernels_launched += g_trial_kernels;
                C.spin_sync();
                const auto t2 = std::chrono::steady_clock::now();
                stats.host_wait_s += std::chrono::duration<double>(t2 - t1).count();
                stats.gpu_eval_ms += 1e3 * std::chrono::duration<double>(t1 - t0).count();   // host time in launch
                ++stats.evaluations;
                return;
            }
        }
        // More-Thuente reads the slope of every trial: plain f+g evaluation, one read-back
        // (not on the slice kernel: there a combined f+g launch costs ~4 us more than the objective alone, less than the
        // second launch and host round trip the split costs the ~87 % of trials whose gradient IS read)
        if (!eval(xp, d, stp, d, (prm.linesearch != 0 && C.lazy_gradient && !C.slice_ok()) ? &ls : nullptr)) {
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

    // the recursion of lbfgs.c:572-598 as 2*bound+1 fused kernels; the last one also leaves g.d in SC_DGINIT
    void two_loop(int bound, int end, int m) {
        const bool fused = reduce && C.fuse_exchange();
        auto launch = [&](TwoLoopArgs& a) {
            a.n = n; a.d = d; a.g = g; a.partials = C.red_partials.p; a.ticket = C.ticket.p; a.sc = C.sc.p;
            if (fused && a.v) a.p2p = C.p2p_dev(); else a.p2p.nranks = 1;
            k_lbfgs_twoloop<<<vec_blocks, kVecThreads, 0, C.stream>>>(a);
            ++C.kernels_launched;
            if (reduce && !fused && a.v) C.comm->allreduce_sum(C.sc.p + a.out, 1, C.stream);
        };
        std::vector<int> js(bound);
        int j = end;
        for (int i = 0; i < bound; ++i) { j = (j + m - 1) % m; js[i] = j; }   // newest ... oldest
        {   // d = -g ; alpha_raw[j0] = s_j0 . d
            TwoLoopArgs a{};
            a.init = 1; a.u = nullptr; a.c_num = a.c_den = 0; a.c2_num = -1; a.s_num = -1;
            a.v = S[js[0]]; a.out = SC_ALPHA0 + js[0];
            launch(a);
        }
        for (int i = 0; i < bound; ++i) {
            // d -= alpha_j y_j ; then either the next alpha, or (last) the H0 scaling and the first beta
            TwoLoopArgs a{};
            a.u = Yv[js[i]]; a.c_num = SC_ALPHA0 + js[i]; a.c_den = SC_YS0 + js[i]; a.csign = -1.0; a.c2_num = -1;
            if (i + 1 < bound) {
                a.s_num = -1; a.v = S[js[i + 1]]; a.out = SC_ALPHA0 + js[i + 1];
            } else {
                a.s_num = SC_YS; a.s_den = SC_YY; a.v = Yv[js[i]]; a.out = SC_BETA;
            }
            launch(a);
        }
        int beta_slot = SC_BETA;
        for (int i = bound - 1; i >= 0; --i) {
            // d += (alpha_j - beta_j) s_j ; then the next beta, or (last) g.d
            TwoLoopArgs a{};
            a.u = S[js[i]];
            a.c_num = SC_ALPHA0 + js[i]; a.c_den = SC_YS0 + js[i]; a.csign = 1.0;
            a.c2_num = beta_slot; a.c2_den = SC_YS0 + js[i]; a.c2sign = -1.0;
            a.s_num = -1;
            beta_slot = (beta_slot == SC_BETA) ? SC_BETA2 : SC_BETA;
            if (i > 0) { a.v = Yv[js[i - 1]]; a.out = beta_slot; }
            else { a.v = g; a.out = SC_DGINIT; }
            launch(a);
        }
    }

    // one line search (lbfgs.c:645-734 backtracking, 812-1001 More-Thuente) driven by LineSearchState: every
    // trial is one f+g evaluation on the device and one 512-byte read-back.  On success h_sc holds the scalars
    // of the accepted point.
    int linesearch(double& f, double& stp, double& dginit, bool& dginit_known) {
        const double* h = C.h_sc;
        if (stp <= 0.) return LBFGSERR_INVALIDPARAMETERS;
        // g.d of the new direction was left in the scalar file (SC_DGINIT) by the update kernels.  The first trial
        // point xp + stp*d does not depend on it, so the trial is enqueued right behind the update and the slope
        // arrives with the trial's own scalars: one host round trip per iteration instead of two.  (The one case
        // where the slope matters beforehand -- 0 < g.d, LBFGSERR_INCREASEGRADIENT -- then costs one evaluation
        // that liblbfgs would not have made; x and g are restored by the caller as after any failed search.)
        spec_slope = !dginit_known && !use_graphs && C.lbfgs_speculative;
        if (!dginit_known && !spec_slope) {
            C.fetch_scalars();
            dginit = h[SC_DGINIT];
            dginit_known = true;
        }
        if (dginit_known && 0 < dginit) return LBFGSERR_INCREASEGRADIENT;
        LineSearchState ls;
        ls.start(prm, f, dginit_known ? dginit : 0.0, stp);
        spec_ls = &ls;
        for (;;) {
            stp = ls.prepare();
            trial(stp, ls);
            if (spec_bad) {   // the slope that came with the first trial is positive
                spec_bad = false;
                dginit = h[SC_DGINIT];
                dginit_known = true;
                return LBFGSERR_INCREASEGRADIENT;
            }
            if (!dginit_known) { dginit = ls.dginit; dginit_known = true; }
            f = h[SC_F];
            const int verdict = ls.update(f, h[SC_DG]);
            if (verdict != 0) return verdict;
        }
    }
};

}  // namespace bioen
