// gsl_min.cuh -- the five GSL 2.5 `multimin` gradient minimisers BioEn can select, re-implemented on device
// vectors, plus BioEn's own driver loop and stop test.
//
// Reference behaviour being reproduced (third-party/gsl-2.5/multimin/ and the BioEn drivers):
//   driver loop + "max_i |g_i| < tol" stop test   c_bioen_kernels_logw.c:434-452, c_bioen_common.c:112-138
//   vector_bfgs2  (Fletcher line search)          vector_bfgs2.c:143-318, linear_minimize.c, linear_wrapper.c
//   conjugate_fr / conjugate_pr / vector_bfgs     conjugate_fr.c:100-256, conjugate_pr.c:238-243,
//                                                 vector_bfgs.c:142-337, directional_minimize.c
//   steepest_descent                              steepest_descent.c:63-163
//
// All n-vectors (x, gradient, p, x0, g0, dx0, dg0, x_alpha, g_alpha, x1, x2 ...) stay in HBM; level-1 BLAS
// becomes small fused kernels; the branchy scalar logic runs on the host.  GSL calls three different
// callbacks: f only (line-search probes: ONE pass over yTilde here), df only, and fdf.
#pragma once
#include <cmath>
#include <cstdio>
#include <vector>

#include "context.cuh"

namespace bioen {

enum { GSL_SUCCESS = 0, GSL_FAILURE = -1, GSL_CONTINUE = -2, GSL_EBADTOL = 13, GSL_ENOPROG = 27 };
constexpr double kGslDblEpsilon = 2.2204460492503131e-16;

// max_j |x_j| with the reference's NaN behaviour (`if (temp > norm) norm = temp` skips NaNs -> fmax)
__global__ void __launch_bounds__(kVecThreads)
    k_grid_max_abs(int n, const double* x, double* out, double* partials, unsigned int* ticket) {
    __shared__ double red[2 * 32];
    double v[2] = {0.0, 0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x)
        v[1] = fmax(v[1], fabs(x[j]));
    grid_sum_max<1>(v, partials, ticket, red, [=](const double(&t)[2]) { out[0] = t[1]; });
}

__global__ void __launch_bounds__(kVecThreads) k_count_diff(int n, const double* a, const double* b, unsigned int* out) {
    unsigned int c = 0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) c += (a[j] != b[j]);
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

struct GslStats {
    int iterations = 0, n_f = 0, n_df = 0, n_fdf = 0;
    int n_df_continued = 0;   // evaluations that ran one half only: df of the point f() had just evaluated, or an
                              // fdf whose gradient the algorithm discards (steepest descent's rejected steps)
};

// vector toolbox on the context's stream
class VecOps {
   public:
    Context& C;
    const bool forces;
    const int n;
    const size_t np;
    int blocks;
    bool reduce;
    std::vector<double*> pool;
    DevBuf<double> store;
    size_t used = 0, cap;
    GslStats stats;
    long long n_total;   // GSL's x->size: all of N when the log-weights are sharded

    VecOps(Context& ctx, bool is_forces, int nvec)
        : C(ctx), forces(is_forces), n(is_forces ? ctx.M : ctx.N), np(((size_t)n + 15) & ~(size_t)15), cap(nvec) {
        n_total = is_forces ? ctx.M : ctx.N_total;
        blocks = is_forces ? ctx.vec_blocks_m : ctx.vec_blocks_n;
        reduce = (!is_forces) && ctx.nranks > 1;
        store.alloc(np * cap);
    }
    double* vec() {
        if (used >= cap) throw std::logic_error("bioen_b200: vector pool exhausted");
        return store.p + np * used++;
    }
    void copy(double* dst, const double* src) { C.d2d(dst, src, n); }
    void zero(double* dst) { CUDA_CHECK(cudaMemsetAsync(dst, 0, n * sizeof(double), C.stream)); }
    // y += alpha * x
    void axpy(double alpha, const double* x, double* y) {
        k_axpby<<<blocks, kVecThreads, 0, C.stream>>>(n, alpha, x, 1.0, y, y);
    }
    // z = alpha * x + beta * y
    void axpby(double alpha, const double* x, double beta, const double* y, double* z) {
        k_axpby<<<blocks, kVecThreads, 0, C.stream>>>(n, alpha, x, beta, y, z);
    }
    void scal(double alpha, double* x) { k_axpby<<<blocks, kVecThreads, 0, C.stream>>>(n, alpha, x, 0.0, nullptr, x); }
    // up to three dot products in one sweep + one read-back
    void dots(const double* a0, const double* b0, const double* a1, const double* b1, const double* a2,
              const double* b2, double out[3]) {
        Dot3Args a{n, a0, b0, a1, b1, a2, b2, C.sc.p + SC_TMP0, C.red_partials.p, C.ticket.p};
        k_dot3<<<blocks, kVecThreads, 0, C.stream>>>(a);
        if (reduce) C.comm->allreduce_sum(C.sc.p + SC_TMP0, 3, C.stream);
        C.d2h(C.h_sc + SC_TMP0, C.sc.p + SC_TMP0, 3);
        C.sync();
        out[0] = C.h_sc[SC_TMP0]; out[1] = C.h_sc[SC_TMP0 + 1]; out[2] = C.h_sc[SC_TMP0 + 2];
    }
    double dot(const double* a, const double* b) {
        double o[3];
        dots(a, b, nullptr, nullptr, nullptr, nullptr, o);
        return o[0];
    }
    double nrm2(const double* a) { return std::sqrt(dot(a, a)); }
    bool equal(const double* a, const double* b) {
        unsigned int* cnt = C.ticket.p + 2;
        CUDA_CHECK(cudaMemsetAsync(cnt, 0, sizeof(unsigned int), C.stream));
        k_count_diff<<<blocks, kVecThreads, 0, C.stream>>>(n, a, b, cnt);
        unsigned int h = 0;
        CUDA_CHECK(cudaMemcpyAsync(&h, cnt, sizeof h, cudaMemcpyDeviceToHost, C.stream));
        C.sync();
        double v = (double)h;
        if (reduce) {  // any rank differing makes the vectors differ
            CUDA_CHECK(cudaMemcpyAsync(C.sc.p + SC_TMP0, &v, sizeof v, cudaMemcpyHostToDevice, C.stream));
            C.comm->allreduce_sum(C.sc.p + SC_TMP0, 1, C.stream);
            C.d2h(&v, C.sc.p + SC_TMP0, 1);
            C.sync();
        }
        return v == 0.0;
    }
    // ---- the three GSL callbacks (c_bioen_kernels_logw.c:274-362, c_bioen_kernels_forces.c:347-428)
    long long f_gen = -1;        // C.eval_gen right after the last f(): df_same_point may continue it
    const double* f_x = nullptr;
    double f(double* x) {
        ++stats.n_f;
        if (forces) C.forces_eval(x, nullptr, nullptr, 0.0, nullptr, nullptr);
        else C.logw_eval(x, nullptr, nullptr, 0.0, nullptr, nullptr);
        C.fetch_scalars();
        f_gen = C.eval_gen;
        f_x = x;
        return C.h_sc[SC_F];
    }
    // fdf(x, g) for a caller that discards the gradient when f > f_limit (steepest_descent.c:117-127 retries with a
    // shorter step): the gradient half runs only when it will be kept
    double fdf_unless_above(double* x, double* g, double f_limit) {
        if (!C.options.lazy_gradient) return fdf(x, g);
        ++stats.n_fdf;
        if (forces) C.forces_eval_f(x, nullptr, nullptr, 0.0);
        else C.logw_eval_f(x, nullptr, nullptr, 0.0);
        C.fetch_scalars();
        const double fx = C.h_sc[SC_F];
        if (fx > f_limit) {
            ++stats.n_df_continued;
            return fx;
        }
        if (forces) C.forces_eval_g(g, nullptr);
        else C.logw_eval_g(x, g, nullptr);
        return fx;
    }
    // df(x, g) for call sites where x still holds the point the immediately preceding f(x) evaluated
    // (directional_minimize.c evaluates f at a trial point and, if it is kept, the gradient there)
    void df_same_point(double* x, double* g) {
        if (C.options.lazy_gradient && f_x == x && f_gen == C.eval_gen) df_continue(x, g);
        else df(x, g);
    }
    void df(double* x, double* g) {
        ++stats.n_df;
        if (forces) C.forces_eval(x, nullptr, nullptr, 0.0, g, nullptr);
        else C.logw_eval(x, nullptr, nullptr, 0.0, g, nullptr);
    }
    // gradient at the point the context evaluated LAST with f() (weights, averages and residuals are still on the
    // device): only the gradient half of the evaluation runs.  The caller guarantees the point is the same.
    void df_continue(double* x, double* g) {
        ++stats.n_df;
        ++stats.n_df_continued;
        if (forces) C.forces_eval_g(g, nullptr);
        else C.logw_eval_g(x, g, nullptr);
    }
    double fdf(double* x, double* g) {
        ++stats.n_fdf;
        if (forces) C.forces_eval(x, nullptr, nullptr, 0.0, g, nullptr);
        else C.logw_eval(x, nullptr, nullptr, 0.0, g, nullptr);
        C.fetch_scalars();
        return C.h_sc[SC_F];
    }
    // max_i |g_i| of the most recent gradient evaluation (kept in the scalar file by the gradient kernels)
    double last_grad_inf() {
        if (reduce) {
            C.comm->allreduce_max(C.sc.p + SC_GINF, 1, C.stream);
        }
        C.fetch_scalars();
        return C.h_sc[SC_GINF];
    }
};

// ---- Fletcher's line minimisation (linear_minimize.c) ----------------------------------------------------
namespace fletcher {
inline int solve_quadratic(double a, double b, double c, double& x0, double& x1) {  // poly/solve_quadratic.c
    if (a == 0) {
        if (b == 0) return 0;
        x0 = -c / b;
        return 1;
    }
    const double disc = b * b - 4 * a * c;
    if (disc > 0) {
        if (b == 0) {
            const double r = std::sqrt(-c / a);
            x0 = -r; x1 = r;
        } else {
            const double sgnb = (b > 0 ? 1 : -1);
            const double temp = -0.5 * (b + sgnb * std::sqrt(disc));
            const double r1 = temp / a, r2 = c / temp;
            if (r1 < r2) { x0 = r1; x1 = r2; } else { x0 = r2; x1 = r1; }
        }
        return 2;
    } else if (disc == 0) {
        x0 = x1 = -0.5 * b / a;
        return 2;
    }
    return 0;
}
inline double interp_quad(double f0, double fp0, double f1, double zl, double zh) {
    const double fl = f0 + zl * (fp0 + zl * (f1 - f0 - fp0));
    const double fh = f0 + zh * (fp0 + zh * (f1 - f0 - fp0));
    const double c = 2 * (f1 - f0 - fp0);
    double zmin = zl, fmin = fl;
    if (fh < fmin) { zmin = zh; fmin = fh; }
    if (c > 0) {
        const double z = -fp0 / c;
        if (z > zl && z < zh) {
            const double f = f0 + z * (fp0 + z * (f1 - f0 - fp0));
            if (f < fmin) { zmin = z; fmin = f; }
        }
    }
    return zmin;
}
inline double interp_cubic(double f0, double fp0, double f1, double fp1, double zl, double zh) {
    const double eta = 3 * (f1 - f0) - 2 * fp0 - fp1, xi = fp0 + fp1 - 2 * (f1 - f0);
    const double c0 = f0, c1 = fp0, c2 = eta, c3 = xi;
    auto cubic = [&](double z) { return c0 + z * (c1 + z * (c2 + z * c3)); };
    double zmin = zl, fmin = cubic(zl);
    auto check = [&](double z) {
        const double y = cubic(z);
        if (y < fmin) { zmin = z; fmin = y; }
    };
    check(zh);
    double z0 = 0, z1 = 0;
    const int nr = solve_quadratic(3 * c3, 2 * c2, c1, z0, z1);
    if (nr == 2) {
        if (z0 > zl && z0 < zh) check(z0);
        if (z1 > zl && z1 < zh) check(z1);
    } else if (nr == 1) {
        if (z0 > zl && z0 < zh) check(z0);
    }
    return zmin;
}
inline double interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin,
                          double xmax, int order) {
    double zmin = (xmin - a) / (b - a), zmax = (xmax - a) / (b - a);
    if (zmin > zmax) std::swap(zmin, zmax);
    double z;
    if (order > 2 && std::isfinite(fpb)) z = interp_cubic(fa, fpa * (b - a), fb, fpb * (b - a), zmin, zmax);
    else z = interp_quad(fa, fpa * (b - a), fb, zmin, zmax);
    return a + z * (b - a);
}
}  // namespace fletcher

// 1-d view along a direction with alpha-keyed caches (linear_wrapper.c:25-185)
struct LineWrapper {
    VecOps& V;
    double *x, *g, *p;          // owned by the minimiser state
    double *x_alpha, *g_alpha;
    double f_alpha = 0, df_alpha = 0;
    double f_key = 0, df_key = 0, x_key = 0, g_key = 0;
    // which alpha the context's evaluation state (w, avg, residuals) belongs to: set by f(), void after any other
    // evaluation (eval_gen moves) or a change of x / p.  GSL's Fletcher search asks f(alpha) and then df(alpha).
    double state_key = 0;
    long long state_gen = -1;

    LineWrapper(VecOps& v, double* x_, double f_, double* g_, double* p_, double* xa, double* ga)
        : V(v), x(x_), g(g_), p(p_), x_alpha(xa), g_alpha(ga) {
        V.copy(x_alpha, x);
        f_alpha = f_;
        V.copy(g_alpha, g);
        df_alpha = V.dot(g_alpha, p);
    }
    void moveto(double alpha) {
        if (alpha == x_key) return;
        V.axpby(1.0, x, alpha, p, x_alpha);
        x_key = alpha;
    }
    double f(double alpha) {
        if (alpha == f_key) return f_alpha;
        moveto(alpha);
        f_alpha = V.f(x_alpha);
        f_key = alpha;
        state_key = alpha;
        state_gen = V.C.eval_gen;
        return f_alpha;
    }
    double df(double alpha) {
        if (alpha == df_key) return df_alpha;
        moveto(alpha);
        if (alpha != g_key) {
            if (V.C.options.lazy_gradient && state_gen == V.C.eval_gen && alpha == state_key) V.df_continue(x_alpha, g_alpha);
            else V.df(x_alpha, g_alpha);
            g_key = alpha;
        }
        df_alpha = V.dot(g_alpha, p);
        df_key = alpha;
        return df_alpha;
    }
    void fdf(double alpha, double& f_, double& df_) {
        if (alpha == f_key && alpha == df_key) { f_ = f_alpha; df_ = df_alpha; return; }
        if (alpha == f_key || alpha == df_key) { f_ = f(alpha); df_ = df(alpha); return; }
        moveto(alpha);
        f_alpha = V.fdf(x_alpha, g_alpha);
        f_key = g_key = alpha;
        df_alpha = V.dot(g_alpha, p);
        df_key = alpha;
        f_ = f_alpha; df_ = df_alpha;
    }
    double update_position(double alpha, double* xo, double* go) {
        double a, b;
        fdf(alpha, a, b);
        V.copy(xo, x_alpha);
        V.copy(go, g_alpha);
        return f_alpha;
    }
    void change_direction() {
        state_gen = -1;
        V.copy(x_alpha, x);
        x_key = 0.0;
        f_key = 0.0;
        V.copy(g_alpha, g);
        g_key = 0.0;
        df_alpha = V.dot(g_alpha, p);
        df_key = 0.0;
    }
};

// linear_minimize.c:130-247
inline int fletcher_minimize(LineWrapper& w, double rho, double sigma, double tau1, double tau2, double tau3,
                             int order, double alpha1, double& alpha_new) {
    double f0, fp0, falpha, falpha_prev, fpalpha, fpalpha_prev, delta, alpha_next;
    double alpha = alpha1, alpha_prev = 0.0;
    double a, b, fa, fb, fpa, fpb;
    const size_t bracket_iters = 100, section_iters = 100;
    size_t i = 0;
    w.fdf(0.0, f0, fp0);
    falpha_prev = f0;
    fpalpha_prev = fp0;
    a = 0.0; b = alpha; fa = f0; fb = 0.0; fpa = fp0; fpb = 0.0;
    while (i++ < bracket_iters) {
        falpha = w.f(alpha);
        if (falpha > f0 + alpha * rho * fp0 || falpha >= falpha_prev) {
            a = alpha_prev; fa = falpha_prev; fpa = fpalpha_prev;
            b = alpha; fb = falpha; fpb = NAN;
            break;
        }
        fpalpha = w.df(alpha);
        if (std::fabs(fpalpha) <= -sigma * fp0) { alpha_new = alpha; return GSL_SUCCESS; }
        if (fpalpha >= 0) {
            a = alpha; fa = falpha; fpa = fpalpha;
            b = alpha_prev; fb = falpha_prev; fpb = fpalpha_prev;
            break;
        }
        delta = alpha - alpha_prev;
        alpha_next = fletcher::interpolate(alpha_prev, falpha_prev, fpalpha_prev, alpha, falpha, fpalpha,
                                           alpha + delta, alpha + tau1 * delta, order);
        alpha_prev = alpha; falpha_prev = falpha; fpalpha_prev = fpalpha;
        alpha = alpha_next;
    }
    while (i++ < section_iters) {
        delta = b - a;
        alpha = fletcher::interpolate(a, fa, fpa, b, fb, fpb, a + tau2 * delta, b - tau3 * delta, order);
        falpha = w.f(alpha);
        if ((a - alpha) * fpa <= kGslDblEpsilon) return GSL_ENOPROG;
        if (falpha > f0 + rho * alpha * fp0 || falpha >= fa) {
            b = alpha; fb = falpha; fpb = NAN;
        } else {
            fpalpha = w.df(alpha);
            if (std::fabs(fpalpha) <= -sigma * fp0) { alpha_new = alpha; return GSL_SUCCESS; }
            if (((b - a) >= 0 && fpalpha >= 0) || ((b - a) <= 0 && fpalpha <= 0)) { b = a; fb = fa; fpb = fpa; }
            a = alpha; fa = falpha; fpa = fpalpha;
        }
    }
    return GSL_SUCCESS;  // alpha_new untouched, as in GSL
}

// common state of every fdfminimizer (fdfminimizer.c): x, f, gradient, dx
struct MinimizerBase {
    VecOps& V;
    double *x, *gradient, *dx;
    double f = 0.0;
    explicit MinimizerBase(VecOps& v) : V(v) { x = V.vec(); gradient = V.vec(); dx = V.vec(); }
    virtual ~MinimizerBase() {}
    virtual int iterate() = 0;
};

struct Bfgs2 : MinimizerBase {  // vector_bfgs2.c
    double step, g0norm, pnorm, delta_f = 0, fp0;
    double *x0, *g0, *p, *dx0, *dg0, *x_alpha, *g_alpha;
    LineWrapper* wrap = nullptr;
    double rho = 0.01, sigma, tau1 = 9, tau2 = 0.05, tau3 = 0.5;
    int order = 3;
    Bfgs2(VecOps& v, double step_size, double tol) : MinimizerBase(v), step(step_size), sigma(tol) {
        x0 = V.vec(); g0 = V.vec(); p = V.vec(); dx0 = V.vec(); dg0 = V.vec(); x_alpha = V.vec(); g_alpha = V.vec();
    }
    ~Bfgs2() override { delete wrap; }
    void set() {
        f = V.fdf(x, gradient);
        V.copy(x0, x);
        V.copy(g0, gradient);
        g0norm = V.nrm2(g0);
        V.axpby(-1 / g0norm, gradient, 0.0, nullptr, p);
        pnorm = V.nrm2(p);
        fp0 = -g0norm;
        wrap = new LineWrapper(V, x0, f, g0, p, x_alpha, g_alpha);
    }
    int iterate() override {
        double alpha = 0.0, alpha1;
        const double f0 = f;
        if (pnorm == 0.0 || g0norm == 0.0 || fp0 == 0) { V.zero(dx); return GSL_ENOPROG; }
        if (delta_f < 0) {
            const double del = std::fmax(-delta_f, 10 * kGslDblEpsilon * std::fabs(f0));
            alpha1 = std::fmin(1.0, 2.0 * del / (-fp0));
        } else {
            alpha1 = std::fabs(step);
        }
        const int status = fletcher_minimize(*wrap, rho, sigma, tau1, tau2, tau3, order, alpha1, alpha);
        if (status != GSL_SUCCESS) return status;
        f = wrap->update_position(alpha, x, gradient);
        delta_f = f - f0;
        V.axpby(1.0, x, -1.0, x0, dx0);          // dx0 = x - x0
        V.copy(dx, dx0);
        V.axpby(1.0, gradient, -1.0, g0, dg0);   // dg0 = g - g0
        double d3[3], dn[3];
        V.dots(dx0, gradient, dg0, gradient, dx0, dg0, d3);
        V.dots(dg0, dg0, nullptr, nullptr, nullptr, nullptr, dn);
        const double dxg = d3[0], dgg = d3[1], dxdg = d3[2], dgnorm = std::sqrt(dn[0]);
        double A, B;
        if (dxdg != 0) {
            B = dxg / dxdg;
            A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg;
        } else {
            B = 0; A = 0;
        }
        V.copy(p, gradient);
        V.axpy(-A, dx0, p);
        V.axpy(-B, dg0, p);
        V.copy(g0, gradient);
        V.copy(x0, x);
        double t[3];
        V.dots(g0, g0, p, p, p, gradient, t);
        g0norm = std::sqrt(t[0]);
        pnorm = std::sqrt(t[1]);
        const double pg = t[2];
        const double dir = (pg >= 0.0) ? -1.0 : +1.0;
        V.scal(dir / pnorm, p);
        V.dots(p, p, p, g0, nullptr, nullptr, t);
        pnorm = std::sqrt(t[0]);
        fp0 = t[1];
        wrap->change_direction();
        return GSL_SUCCESS;
    }
};

// conjugate_fr / conjugate_pr / vector_bfgs share directional_minimize.c
struct Directional : MinimizerBase {
    int kind;  // 0 fr, 1 pr, 3 bfgs
    int iter = 0;
    double step, max_step, tol, pnorm, g0norm;
    double *x1, *dx1, *x2, *p, *g0, *x0, *dx0, *dg0, *dx2;
    Directional(VecOps& v, int kind_, double step_size, double tol_)
        : MinimizerBase(v), kind(kind_), step(step_size), max_step(step_size), tol(tol_) {
        x1 = V.vec(); dx1 = V.vec(); x2 = V.vec(); p = V.vec(); g0 = V.vec(); x0 = V.vec(); dx0 = V.vec();
        dg0 = V.vec(); dx2 = V.vec();
    }
    void set() {
        f = V.fdf(x, gradient);
        V.copy(x0, x);
        V.copy(p, gradient);
        V.copy(g0, gradient);
        pnorm = g0norm = V.nrm2(gradient);
    }
    // directional_minimize.c:20-29
    void take_step(const double* xx, const double* pp, double stp, double lambda, double* xo, double* dxo) {
        V.axpby(-stp * lambda, pp, 0.0, nullptr, dxo);
        V.axpby(1.0, xx, 1.0, dxo, xo);
    }
    int iterate() override {
        double fa = f, fb, fc, stepa = 0.0, stepb, stepc = step, g1norm;
        if (pnorm == 0.0 || g0norm == 0.0) { V.zero(dx); return GSL_ENOPROG; }
        const double pg = V.dot(p, gradient);
        const double dir = (pg >= 0.0) ? +1.0 : -1.0;
        const double lambda = dir / pnorm;
        take_step(x, p, stepc, lambda, x1, dx);
        fc = V.f(x1);
        if (fc < fa) {
            step = stepc * 2.0;
            f = fc;
            V.copy(x, x1);
            V.df_same_point(x1, gradient);
            return GSL_SUCCESS;
        }
        // intermediate_point (directional_minimize.c:31-83)
        {
            double fcc = fc, stepcc = stepc;
            for (;;) {
                const double u = std::fabs(pg * lambda * stepcc);
                stepb = 0.5 * stepcc * u / ((fcc - fa) + u);
                take_step(x, p, stepb, lambda, x1, dx1);
                if (V.equal(x, x1)) {
                    stepb = 0; fb = fa;
                    V.df(x1, gradient);
                    break;
                }
                fb = V.f(x1);
                if (fb >= fa && stepb > 0.0) { fcc = fb; stepcc = stepb; continue; }
                V.df_same_point(x1, gradient);
                break;
            }
        }
        if (stepb == 0.0) return GSL_ENOPROG;
        // minimize (directional_minimize.c:85-248)
        {
            double u = stepb, v = stepa, w = stepc, fu = fb, fv = fa, fw = fc;
            double old2 = std::fabs(w - v), old1 = std::fabs(v - u), stepm, fm;
            double sa = stepa, sb = stepb, sc_ = stepc, fA = fa, fB = fb, fC = fc;
            int it = 0;
            V.copy(x2, x1);
            V.copy(dx2, dx1);
            f = fb;
            step = stepb;
            g1norm = V.nrm2(gradient);
            for (;;) {
                if (++it > 10) break;
                const double dw = w - u, dv = v - u;
                double du = 0.0;
                const double e1 = ((fv - fu) * dw * dw + (fu - fw) * dv * dv);
                const double e2 = 2.0 * ((fv - fu) * dw + (fu - fw) * dv);
                if (e2 != 0.0) du = e1 / e2;
                if (du > 0.0 && du < (sc_ - sb) && std::fabs(du) < 0.5 * old2) stepm = u + du;
                else if (du < 0.0 && du > (sa - sb) && std::fabs(du) < 0.5 * old2) stepm = u + du;
                else if ((sc_ - sb) > (sb - sa)) stepm = 0.38 * (sc_ - sb) + sb;
                else stepm = sb - 0.38 * (sb - sa);
                take_step(x, p, stepm, lambda, x1, dx1);
                fm = V.f(x1);
                if (fm > fB) {
                    if (fm < fv) { w = v; v = stepm; fw = fv; fv = fm; }
                    else if (fm < fw) { w = stepm; fw = fm; }
                    if (stepm < sb) { sa = stepm; fA = fm; } else { sc_ = stepm; fC = fm; }
                    continue;
                } else if (fm <= fB) {
                    old2 = old1;
                    old1 = std::fabs(u - stepm);
                    w = v; v = u; u = stepm;
                    fw = fv; fv = fu; fu = fm;
                    V.copy(x2, x1);
                    V.copy(dx2, dx1);
                    V.df_same_point(x1, gradient);
                    double t[3];
                    V.dots(p, gradient, gradient, gradient, nullptr, nullptr, t);
                    const double pg1 = t[0], gnorm1 = std::sqrt(t[1]);
                    f = fm; step = stepm; g1norm = gnorm1;
                    if (std::fabs(pg1 * lambda / gnorm1) < tol) break;
                    if (stepm < sb) { sc_ = sb; fC = fB; sb = stepm; fB = fm; }
                    else { sa = sb; fA = fB; sb = stepm; fB = fm; }
                    continue;
                }
                break;  // NaN
            }
            (void)fA; (void)fC;
        }
        V.copy(x, x2);
        V.copy(dx, dx2);
        iter = (int)((iter + 1) % V.n_total);
        if (iter == 0) {
            V.copy(p, gradient);
            pnorm = g1norm;
        } else if (kind == 0) {
            const double beta = -std::pow(g1norm / g0norm, 2.0);
            V.axpby(-beta, p, 1.0, gradient, p);
            pnorm = V.nrm2(p);
        } else if (kind == 1) {
            V.axpy(-1.0, gradient, g0);
            const double g0g1 = V.dot(g0, gradient);
            const double beta = g0g1 / (g0norm * g0norm);
            V.axpby(-beta, p, 1.0, gradient, p);
            pnorm = V.nrm2(p);
        } else {
            V.axpby(1.0, x, -1.0, x0, dx0);
            V.axpby(1.0, gradient, -1.0, g0, dg0);
            double d3[3], dn[3];
            V.dots(dx0, gradient, dg0, gradient, dx0, dg0, d3);
            V.dots(dg0, dg0, nullptr, nullptr, nullptr, nullptr, dn);
            const double dxg = d3[0], dgg = d3[1], dxdg = d3[2], dgnorm = std::sqrt(dn[0]);
            double A, B;
            if (dxdg != 0) {
                B = dxg / dxdg;
                A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg;
            } else {
                B = 0; A = 0;
            }
            V.copy(p, gradient);
            V.axpy(-A, dx0, p);
            V.axpy(-B, dg0, p);
            pnorm = V.nrm2(p);
        }
        if (kind == 3) {
            V.copy(g0, gradient);
            V.copy(x0, x);
            g0norm = V.nrm2(g0);
        } else {
            g0norm = g1norm;
            V.copy(g0, gradient);
        }
        return GSL_SUCCESS;
    }
};

struct SteepestDescent : MinimizerBase {  // steepest_descent.c
    double step, max_step, tol;
    double *x1, *g1;
    SteepestDescent(VecOps& v, double step_size, double tol_)
        : MinimizerBase(v), step(step_size), max_step(step_size), tol(tol_) {
        x1 = V.vec(); g1 = V.vec();
    }
    void set() { f = V.fdf(x, gradient); }
    int iterate() override {
        const double f0 = f;
        double f1, stp = step;
        bool failed = false;
        const double gnorm = V.nrm2(gradient);
        if (gnorm == 0.0) { V.zero(dx); return GSL_ENOPROG; }
        for (;;) {
            V.axpby(-stp / gnorm, gradient, 0.0, nullptr, dx);
            V.axpby(1.0, x, 1.0, dx, x1);
            if (V.equal(x, x1)) return GSL_ENOPROG;
            f1 = V.fdf_unless_above(x1, g1, f0);
            if (f1 > f0) { failed = true; stp *= tol; continue; }
            break;
        }
        stp = failed ? stp * tol : stp * 2.0;
        step = stp;
        V.copy(x, x1);
        V.copy(gradient, g1);
        f = f1;
        return GSL_SUCCESS;
    }
};

// BioEn's driver (c_bioen_kernels_logw.c:367-509).  x_dev: start point in, end point out.
inline int gsl_minimize(Context& C, bool forces, double* x_dev, int algorithm, double step_size, double tol,
                        int max_iterations, int verbose, double* fmin, GslStats* out_stats) {
    if (algorithm < 0 || algorithm > 4) throw std::invalid_argument("bioen_b200: unknown GSL algorithm id");
    VecOps V(C, forces, 16);
    MinimizerBase* s = nullptr;
    Bfgs2* b2 = nullptr; Directional* dm = nullptr; SteepestDescent* sd = nullptr;
    if (algorithm == 2) s = b2 = new Bfgs2(V, step_size, tol);
    else if (algorithm == 4) s = sd = new SteepestDescent(V, step_size, tol);
    else s = dm = new Directional(V, algorithm, step_size, tol);
    int status = GSL_SUCCESS, iter = 0;
    try {
        V.copy(s->x, x_dev);
        V.zero(s->dx);
        if (b2) b2->set(); else if (sd) sd->set(); else dm->set();
        do {
            if (verbose && iter != 0 && iter % 1000 == 0) printf("\t\titeration %d\n", iter);
            status = s->iterate();
            if (status) break;
            // scipy-style stop test on the infinity norm (c_bioen_common.c:112-138)
            if (tol < 0.0) {
                status = GSL_EBADTOL;
            } else {
                // the gradient vector of the minimiser state may be older than the last kernel-side max (line
                // searches evaluate other points), so take the max of the state vector itself
                k_grid_max_abs<<<V.blocks, kVecThreads, 0, C.stream>>>(V.n, s->gradient, C.sc.p + SC_GINF,
                                                                      C.red_partials.p, C.ticket.p);
                const double ginf = V.last_grad_inf();
                status = (ginf < tol) ? GSL_SUCCESS : GSL_CONTINUE;
            }
            ++iter;
        } while (status == GSL_CONTINUE && iter < max_iterations);
        V.copy(x_dev, s->x);
        C.sync();
        *fmin = s->f;
    } catch (...) {
        delete s;
        throw;
    }
    V.stats.iterations = iter;
    if (out_stats) *out_stats = V.stats;
    delete s;
    return status;
}

}  // namespace bioen
