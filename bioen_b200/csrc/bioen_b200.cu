// bioen_b200.cu -- the C ABI of libbioen_b200.so (see include/bioen_b200.h).
//
// Part 1 re-exports the symbols of the reference's C extension with the same signatures and host-pointer
// ownership rules (bioen/optimize/ext/c_bioen.pyx:10-129 is the binding a maintainer keeps unchanged);
// every call uploads its inputs, runs on the GPU and copies the results back.  Part 2 is the handle API with
// yTilde resident in HBM that the Python mirror and bench.py use.
//
// There is no CPU fallback anywhere in this file: without a usable sm_100 device every entry point fails
// (error text in bioen_b200_last_error(), NaN / non-zero status as the return value).
#include "../../include/bioen_b200.h"

#include <chrono>
#include <cmath>
#include <limits>
#include <memory>
#include <mutex>

#include "batched.cuh"
#include "context.cuh"
#include "gsl_min.cuh"
#include "lbfgs.cuh"

using namespace bioen;

// ---------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------
namespace {
thread_local std::string g_last_error;
thread_local int g_error_pending = 0;
int g_fast_flag = 0;

void set_error(const char* where, const std::exception& e) {
    g_last_error = std::string(where) + ": " + e.what();
    g_error_pending = 1;
    fprintf(stderr, "%s\n", g_last_error.c_str());
}

template <class F>
int guarded(const char* where, F&& body) {
    try {
        body();
        return 0;
    } catch (const std::exception& e) {
        set_error(where, e);
        // leave no sticky error behind in the runtime
        cudaGetLastError();
        return 1;
    } catch (...) {
        set_error(where, std::runtime_error("unknown C++ exception"));
        cudaGetLastError();
        return 1;
    }
}

// device used by the reference-compatible (part 1) entry points, which have no device argument
int default_device() {
    if (const char* e = getenv("BIOEN_B200_DEVICE")) return atoi(e);
    return 0;
}
const double kNaN = std::numeric_limits<double>::quiet_NaN();
}  // namespace

struct bioen_b200_ctx {
    Context C;
    std::unique_ptr<Comm> comm;
    DevBuf<double> xn, gn, xm, gm;  // staging vectors for host-pointer calls
    long long pending_gen = -1;     // C.eval_gen of the last objective-only bioen_b200_eval (bioen_b200_grad_continue)
    int pending_method = -1;
    bioen_b200_ctx(int m, int n, int dev) : C(m, n, dev) {}
    double* x_for(int method) {
        if (method == BIOEN_B200_FORCES) {
            if (!xm.p) { xm.alloc(C.Mpad); gm.alloc(C.Mpad); }
            return xm.p;
        }
        if (!xn.p) { xn.alloc(C.Npad); gn.alloc(C.Npad); }
        return xn.p;
    }
    double* g_for(int method) {
        x_for(method);
        return method == BIOEN_B200_FORCES ? gm.p : gn.p;
    }
    int dim(int method) const { return method == BIOEN_B200_FORCES ? C.M : C.N; }
};

// ---------------------------------------------------------------------------------------------------
// synthetic "generic data" generator (bench.py, large-size property tests)
//   yTilde_ij = a_i + b * z(seed, i, col_offset + j),   z ~ N(0,1) from a counter-based hash (splitmix64
//   finaliser on (seed, row, global column)) and Box-Muller.  tests/util_rng.py restates it in NumPy.
// ---------------------------------------------------------------------------------------------------
__host__ __device__ inline unsigned long long mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256) k_generate(double* Y, long long ld, int m, int n, unsigned long long seed,
                                                   long long col_offset, const double* a, double b) {
    const long long total = (long long)m * n;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / n);
        const int j = (int)(t - (long long)i * n);
        const unsigned long long ctr = ((unsigned long long)i << 40) + (unsigned long long)(col_offset + j);
        const unsigned long long h1 = mix64(seed + 0x9E3779B97F4A7C15ULL * (ctr + 1));
        const unsigned long long h2 = mix64(h1 + 0x9E3779B97F4A7C15ULL);
        const double u1 = ((double)(h1 >> 11) + 1.0) * 0x1.0p-53;  // (0, 1]
        const double u2 = (double)(h2 >> 11) * 0x1.0p-53;          // [0, 1)
        const double z = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        Y[(size_t)i * ld + j] = fma(b, z, a[i]);
    }
}

// the same matrix written structure-major (BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY): Yt[j][i] = yTilde_ij
__global__ void __launch_bounds__(256) k_generate_t(double* Yt, long long ldt, int m, int n, unsigned long long seed,
                                                     long long col_offset, const double* a, double b) {
    const long long total = (long long)m * n;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(t / m);
        const int i = (int)(t - (long long)j * m);
        const unsigned long long ctr = ((unsigned long long)i << 40) + (unsigned long long)(col_offset + j);
        const unsigned long long h1 = mix64(seed + 0x9E3779B97F4A7C15ULL * (ctr + 1));
        const unsigned long long h2 = mix64(h1 + 0x9E3779B97F4A7C15ULL);
        const double u1 = ((double)(h1 >> 11) + 1.0) * 0x1.0p-53;  // (0, 1]
        const double u2 = (double)(h2 >> 11) * 0x1.0p-53;          // [0, 1)
        const double z = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        Yt[(size_t)j * ldt + i] = fma(b, z, a[i]);
    }
}

extern "C" {

// ---------------------------------------------------------------------------------------------------
// Part 2 -- handle API
// ---------------------------------------------------------------------------------------------------
const char* bioen_b200_last_error(void) { return g_last_error.c_str(); }

int bioen_b200_error_pending(void) {
    const int p = g_error_pending;
    g_error_pending = 0;
    return p;
}

int bioen_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// Small problems: creating a context (two dozen allocations, pinned memory, a stream) costs ~10 ms, more than a
// whole minimisation at the ala5 size (M = 28, N = 5e4).  The last destroyed small context of a thread is kept and
// handed out again for the same shape; nothing of the previous problem survives (reset_for_reuse), callers upload
// their data as usual, so the stateless entry points stay stateless.
namespace {
constexpr size_t kCacheMaxBytes = (size_t)256 << 20;
constexpr int kCacheSlots = 2;     // find_optimum holds two problems of one shape at a time (yTilde and y)
struct CtxCache {
    bioen_b200_ctx* ctx[kCacheSlots] = {nullptr, nullptr};
    ~CtxCache() {
        for (auto*& c : ctx) { delete c; c = nullptr; }
    }
};
thread_local CtxCache g_cache;
}  // namespace

bioen_b200_ctx* bioen_b200_create(int m, int n, int device) {
    bioen_b200_ctx* ctx = nullptr;
    guarded("bioen_b200_create", [&] {
        for (auto*& c : g_cache.ctx) {
            if (c && c->C.M == m && c->C.N == n && c->C.device == device) {
                bioen_b200_ctx* hit = c;
                c = nullptr;
                CUDA_CHECK(cudaSetDevice(device));
                hit->C.reset_for_reuse();
                hit->comm.reset();
                ctx = hit;
                return;
            }
        }
        ctx = new bioen_b200_ctx(m, n, device);
    });
    return ctx;
}

void bioen_b200_destroy(bioen_b200_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->C.device);
    cudaStreamSynchronize(ctx->C.stream);
    const size_t bytes = (size_t)ctx->C.M * (size_t)ctx->C.N * sizeof(double);
    if (bytes <= kCacheMaxBytes && !ctx->comm) {
        for (auto*& c : g_cache.ctx) {
            if (!c) { c = ctx; return; }
        }
        delete g_cache.ctx[0];                 // both slots taken: drop the older one
        g_cache.ctx[0] = g_cache.ctx[1];
        g_cache.ctx[1] = ctx;
        return;
    }
    delete ctx;
}

int bioen_b200_upload_ytilde(bioen_b200_ctx* ctx, const double* yTilde_host, size_t ld) {
    return guarded("bioen_b200_upload_ytilde", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        if (ctx->C.yt_only) {
            if (ld < (size_t)ctx->C.N) throw std::invalid_argument("bioen_b200: row stride smaller than N");
            ctx->C.alloc_yt();
            ctx->C.upload_rows_yt(0, ctx->C.M, yTilde_host, ld);
        } else {
            ctx->C.upload_matrix(yTilde_host, ld);
        }
        ctx->C.sync();
    });
}

int bioen_b200_adopt_ytilde(bioen_b200_ctx* ctx, double* yTilde_dev, size_t ld) {
    return guarded("bioen_b200_adopt_ytilde", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->C.require_row_major("adopting a row-major device matrix");
        ctx->C.adopt_matrix(yTilde_dev, ld);
    });
}

int bioen_b200_upload_rows(bioen_b200_ctx* ctx, int row0, int nrows, const double* rows_host, size_t ld) {
    return guarded("bioen_b200_upload_rows", [&] {
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        if (row0 < 0 || nrows < 0 || row0 + nrows > C.M) throw std::invalid_argument("bioen_b200: rows out of range");
        if (ld < (size_t)C.N) throw std::invalid_argument("bioen_b200: row stride smaller than N");
        if (C.yt_only) {
            C.upload_rows_yt(row0, nrows, rows_host, ld);
            C.fused_ready = false;
            return;
        }
        if (!C.Y) C.alloc_matrix();
        CUDA_CHECK(cudaMemcpy2DAsync(C.Y + (size_t)row0 * C.ld, C.ld * sizeof(double), rows_host, ld * sizeof(double),
                                     (size_t)C.N * sizeof(double), nrows, cudaMemcpyHostToDevice, C.stream));
        C.sync();
        C.fused_ready = false;     // any structure-major copy is stale now
        C.yt_valid = false;
    });
}

void* bioen_b200_host_alloc(size_t bytes) {
    void* p = nullptr;
    guarded("bioen_b200_host_alloc", [&] { CUDA_CHECK(cudaHostAlloc(&p, bytes, cudaHostAllocPortable)); });
    return p;
}

void bioen_b200_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int bioen_b200_alloc_ytilde(bioen_b200_ctx* ctx) {
    return guarded("bioen_b200_alloc_ytilde", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        if (ctx->C.yt_only) ctx->C.alloc_yt();
        else ctx->C.alloc_matrix();
    });
}

int bioen_b200_set_logw(bioen_b200_ctx* ctx, const double* G_host, const double* YTilde_host, double theta) {
    return guarded("bioen_b200_set_logw", [&] {
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->C.set_observations(YTilde_host);
        ctx->C.set_theta(theta);
        ctx->C.set_logw(G_host, false);
    });
}

int bioen_b200_set_forces(bioen_b200_ctx* ctx, const double* w0_host, const double* YTilde_host, double theta) {
    return guarded("bioen_b200_set_forces", [&] {
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->C.set_observations(YTilde_host);
        ctx->C.set_theta(theta);
        ctx->C.set_forces(w0_host, false);
        ctx->C.sync();
    });
}

int bioen_b200_set_logw_dev(bioen_b200_ctx* ctx, const double* G_dev, const double* YTilde_host, double theta) {
    return guarded("bioen_b200_set_logw_dev", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->C.set_observations(YTilde_host);
        ctx->C.set_theta(theta);
        ctx->C.set_logw(G_dev, true);
    });
}

int bioen_b200_set_forces_dev(bioen_b200_ctx* ctx, const double* w0_dev, const double* YTilde_host, double theta) {
    return guarded("bioen_b200_set_forces_dev", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->C.set_observations(YTilde_host);
        ctx->C.set_theta(theta);
        ctx->C.set_forces(w0_dev, true);
        ctx->C.sync();
    });
}

int bioen_b200_set_option(bioen_b200_ctx* ctx, int option, int value) {
    return guarded("bioen_b200_set_option", [&] {
        ctx->pending_gen = -1;   // a pending objective-only evaluation is not continued across a change of path
        switch (option) {
            case BIOEN_B200_OPT_FUSED_FORCES: ctx->C.options.allow_fused = value != 0; break;
            case BIOEN_B200_OPT_LAZY_GRADIENT: ctx->C.options.lazy_gradient = value != 0; break;
            case BIOEN_B200_OPT_P2P:
                if (ctx->comm) {
                    if (ctx->comm->is_local() && !value)
                        throw std::invalid_argument("bioen_b200: an in-process group has no NCCL path");
                    ctx->comm->use_p2p = value != 0;
                }
                break;
            case BIOEN_B200_OPT_FUSED_EXCHANGE: ctx->C.options.fuse_allowed = value != 0; break;
            case BIOEN_B200_OPT_PERSISTENT: ctx->C.options.persistent_mode = value; break;
            case BIOEN_B200_OPT_LBFGS_GRAM: ctx->C.options.lbfgs_gram_opt = value != 0; break;
            case BIOEN_B200_OPT_SLICE: ctx->C.options.slice_mode = value; break;
            case BIOEN_B200_OPT_LBFGS_SMALL: ctx->C.options.lbfgs_small_opt = value != 0; break;
            case BIOEN_B200_OPT_LBFGS_SPECULATIVE: ctx->C.options.lbfgs_speculative = value != 0; break;
            case BIOEN_B200_OPT_FETCH_ZEROCOPY: ctx->C.options.fetch_zero_copy = value != 0; break;
            case BIOEN_B200_OPT_STRUCTURE_MAJOR_ONLY:
                CUDA_CHECK(cudaSetDevice(ctx->C.device));
                if (value) ctx->C.enter_yt_only();
                else if (ctx->C.yt_only)
                    throw std::invalid_argument("bioen_b200: the row-major matrix is gone; create a new context");
                break;
            case BIOEN_B200_OPT_FP32_STORAGE:
                CUDA_CHECK(cudaSetDevice(ctx->C.device));
                ctx->pending_gen = -1;
                if (value) ctx->C.convert_to_fp32();
                else if (ctx->C.storage_fp32)
                    throw std::invalid_argument("bioen_b200: the fp64 matrix was released; upload yTilde again");
                break;
            default: throw std::invalid_argument("bioen_b200: unknown option");
        }
    });
}

int bioen_b200_set_theta(bioen_b200_ctx* ctx, double theta) {
    ctx->C.set_theta(theta);
    return 0;
}

int bioen_b200_eval(bioen_b200_ctx* ctx, int method, const double* x_host, double* f, double* grad_host) {
    return guarded("bioen_b200_eval", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const int n = ctx->dim(method);
        double* x = ctx->x_for(method);
        double* g = grad_host ? ctx->g_for(method) : nullptr;
        // Log-weights gradient into PAGE-LOCKED host memory: the column pass forms grad_j in its epilogue, so it can
        // store it straight through the mapped host pointer while the pass is still streaming -- the 8*N bytes cross
        // PCIe under the pass instead of in a copy after it.
        bool direct = false;
        if (grad_host && method == BIOEN_B200_LOGW && C.colgrad_eligible()) {
            cudaPointerAttributes attr{};
            if (cudaPointerGetAttributes(&attr, grad_host) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
                attr.devicePointer && (reinterpret_cast<uintptr_t>(attr.devicePointer) & 15) == 0) {
                g = static_cast<double*>(attr.devicePointer);
                direct = true;
            }
            cudaGetLastError();
        }
        C.h2d(x, x_host, n);
        if (method == BIOEN_B200_FORCES) C.forces_eval(x, nullptr, nullptr, 0.0, g, nullptr);
        else C.logw_eval(x, nullptr, nullptr, 0.0, g, nullptr);
        if (grad_host && !direct) C.d2h(grad_host, g, n);
        C.fetch_scalars();
        if (f) *f = C.h_sc[SC_F];
        if (!grad_host) { ctx->pending_gen = C.eval_gen; ctx->pending_method = method; }
    });
}

int bioen_b200_grad_continue(bioen_b200_ctx* ctx, int method, double* grad_host) {
    // nothing evaluated, or the device state has moved on since the objective-only evaluation: not an error
    if (!grad_host || ctx->pending_method != method || ctx->pending_gen != ctx->C.eval_gen) return 2;
    return guarded("bioen_b200_grad_continue", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const int n = ctx->dim(method);
        double* g = ctx->g_for(method);
        if (method == BIOEN_B200_FORCES) C.forces_eval_g(g, nullptr);
        else C.logw_eval_g(ctx->x_for(method), g, nullptr);
        C.d2h(grad_host, g, n);
        C.fetch_scalars();
    });
}

int bioen_b200_weights(bioen_b200_ctx* ctx, int method, const double* x_host, double* w_host, double* sum) {
    return guarded("bioen_b200_weights", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const int n = ctx->dim(method);
        double* x = ctx->x_for(method);
        C.h2d(x, x_host, n);
        if (method == BIOEN_B200_FORCES) C.forces_weights_only(x);
        else C.logw_weights_only(x);
        C.d2h(w_host, C.w.p, C.N);
        C.fetch_scalars();
        // the reference returns the un-stabilised sum_j exp(g_j)
        if (sum) *sum = std::exp(C.h_sc[SC_GMAX]) * C.h_sc[SC_S];
    });
}

int bioen_b200_average(bioen_b200_ctx* ctx, const double* w_host, double* avg_host) {
    return guarded("bioen_b200_average", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        C.h2d(C.w.p, w_host, C.N);
        C.average_of_w(C.avg.p);
        C.d2h(avg_host, C.avg.p, C.M);
        C.sync();
    });
}

int bioen_b200_affine_rows(bioen_b200_ctx* ctx, const double* scale_host, const double* offset_host) {
    return guarded("bioen_b200_affine_rows", [&] {
        NvtxRange nvtx("bioen:affine_rows");
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        C.require_row_major("a row-affine transform");
        if (C.storage_fp32) throw std::logic_error("bioen_b200: row-affine transforms need the fp64 matrix (fp32 storage is on)");
        if (!C.Y) throw std::logic_error("bioen_b200: yTilde has not been uploaded");
        if (!C.Yown.p) throw std::logic_error("bioen_b200: an adopted matrix belongs to the caller and is not modified");
        ++C.eval_gen;
        // scale -> avg, offset -> msum (M-vector scratch of the context; both are rewritten by every evaluation)
        C.h2d(C.avg.p, scale_host, C.M);
        C.h2d(C.msum.p, offset_host, C.M);
        k_affine_rows<<<C.num_sms * 8, 256, 0, C.stream>>>(C.Y, C.ld, C.M, C.N, C.avg.p, C.msum.p);
        CUDA_CHECK(cudaGetLastError());
        ++C.kernels_launched;
        // the structure-major copy (forces method, theta scan) belongs to the old matrix
        const bool had_fused = C.fused_ready;
        C.fused_ready = false;
        C.yt_valid = false;
        if (had_fused && C.have_forces && C.options.allow_fused) C.prepare_fused();
        C.sync();
    });
}

int bioen_b200_forces_from_weights(bioen_b200_ctx* ctx, const double* w_host, double* f, double* grad_host) {
    return guarded("bioen_b200_forces_from_weights", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        double* g = grad_host ? ctx->g_for(BIOEN_B200_FORCES) : nullptr;
        C.h2d(C.w.p, w_host, C.N);
        C.forces_from_weights(g);
        if (grad_host) C.d2h(grad_host, g, C.M);
        C.fetch_scalars();
        if (f) *f = C.h_sc[SC_F];
    });
}

static LbfgsParams to_params(const lbfgs_config_params& c) {
    // c_bioen_kernels_logw.c:607-617: lbfgs_parameter_init then nine overrides; m, min/max_step, xtol stay default
    LbfgsParams p;
    p.linesearch = c.linesearch;
    p.max_iterations = c.max_iterations;
    p.delta = c.delta;
    p.epsilon = c.epsilon;
    p.ftol = c.ftol;
    p.gtol = c.gtol;
    p.wolfe = c.wolfe;
    p.past = c.past;
    p.max_linesearch = c.max_linesearch;
    return p;
}

static void print_lbfgs_header(const lbfgs_config_params& c) {
    printf("L-BFGS minimizer (bioen_b200, device resident)\n");
    printf("\t=========================\n");
    printf("\tlinesearch               : %d\n", c.linesearch);
    printf("\tmax_iterations           : %d\n", c.max_iterations);
    printf("\tdelta                    : %lf\n", c.delta);
    printf("\tepsilon                  : %lf\n", c.epsilon);
    printf("\tftol                     : %lf\n", c.ftol);
    printf("\tgtol                     : %lf\n", c.gtol);
    printf("\twolfe                    : %lf\n", c.wolfe);
    printf("\tpast                     : %d\n", c.past);
    printf("\tmax_linesearch           : %d\n", c.max_linesearch);
    printf("\t=========================\n");
}

static int run_lbfgs_dev(bioen_b200_ctx* ctx, int method, double* x_dev, lbfgs_config_params config,
                         visual_params visual, double* fmin, int info[4]) {
    Context& C = ctx->C;
    if (visual.verbose) print_lbfgs_header(config);
    const auto t0 = std::chrono::steady_clock::now();
    Lbfgs opt(C, method == BIOEN_B200_FORCES, to_params(config));
    opt.verbose = (int)visual.verbose;
    double fx = 0.0;
    const int ret = opt.run(x_dev, &fx);
    C.sync();
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (fmin) *fmin = fx;
    if (info) {
        info[0] = opt.stats.iterations;
        info[1] = opt.stats.evaluations;
        info[2] = opt.stats.gradients_skipped;   // of those evaluations: objective only (one pass over Y)
        info[3] = 0;
    }
    if (opt.trace)
        fprintf(stderr, "[bioen_b200 trace] lbfgs %.3f s wall: %d evals, GPU eval %.1f ms, GPU update+idle %.1f ms\n",
                secs, opt.stats.evaluations, opt.stats.gpu_eval_ms, opt.stats.gpu_update_ms);
    if (visual.verbose) {
        printf("\t%s\n", lbfgs_strerror(ret));
        printf("\tConfig: m=%d and n=%d\n", C.M, C.N);
        printf("\tCurrent function value  = %.6lf\n", fx);
        printf("\tIterations              : %d\n", opt.stats.iterations);
        printf("\tTime(s) of L-BFGS       : %.12lf\n", secs);
        printf("\tTime(s) per iter        : %.12lf\n", secs / (opt.stats.iterations ? opt.stats.iterations : 1));
    }
    return ret;
}

int bioen_b200_opt_lbfgs_dev(bioen_b200_ctx* ctx, int method, double* x_dev, lbfgs_config_params config,
                             visual_params visual, double* fmin, int info[4]) {
    int ret = -2000;
    guarded("bioen_b200_opt_lbfgs_dev", [&] {
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ret = run_lbfgs_dev(ctx, method, x_dev, config, visual, fmin, info);
    });
    return ret;
}

int bioen_b200_opt_lbfgs(bioen_b200_ctx* ctx, int method, const double* x0_host, double* x_host,
                         lbfgs_config_params config, visual_params visual, double* fmin, int info[4]) {
    int ret = -2000;
    guarded("bioen_b200_opt_lbfgs", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const int n = ctx->dim(method);
        double* x = ctx->x_for(method);
        C.h2d(x, x0_host, n);
        const int r = run_lbfgs_dev(ctx, method, x, config, visual, fmin, info);
        C.d2h(x_host, x, n);
        C.sync();
        ret = r;
    });
    return ret;
}

int bioen_b200_opt_gsl(bioen_b200_ctx* ctx, int method, const double* x0_host, double* x_host,
                       gsl_config_params config, visual_params visual, double* fmin, int info[4]) {
    int ret = -2000;
    guarded("bioen_b200_opt_gsl", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const int n = ctx->dim(method);
        double* x = ctx->x_for(method);
        C.h2d(x, x0_host, n);
        if (visual.verbose) {
            static const char* names[] = {"conjugate_fr", "conjugate_pr", "vector_bfgs2", "vector_bfgs",
                                          "steepest_descent"};
            printf("\t=========================\n");
            printf("\tGSL minimizer            : %s (bioen_b200, device resident)\n",
                   (config.algorithm >= 0 && config.algorithm <= 4) ? names[config.algorithm] : "?");
            printf("\ttol                      : %f\n", config.tol);
            printf("\tstep_size                : %f\n", config.step_size);
            printf("\tmax_iteration            : %d\n", config.max_iterations);
            printf("\t=========================\n");
        }
        const auto t0 = std::chrono::steady_clock::now();
        GslStats st;
        double fx = 0.0;
        const int r = gsl_minimize(C, method == BIOEN_B200_FORCES, x, config.algorithm, config.step_size, config.tol,
                                   config.max_iterations, (int)visual.verbose, &fx, &st);
        const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        C.d2h(x_host, x, n);
        C.sync();
        if (fmin) *fmin = fx;
        if (info) {
            info[0] = st.iterations;
            info[1] = st.n_fdf + st.n_df;
            info[2] = st.n_f;
            info[3] = st.n_df_continued;   // of info[1]: ran one half of the evaluation only (see GslStats)
        }
        if (visual.verbose) {
            printf("\t%s\n", bioen_gsl_error(r));
            printf("\tConfig: m=%d and n=%d\n", C.M, C.N);
            printf("\tCurrent function value  = %.6lf\n", fx);
            printf("\tIterations              : %d\n", st.iterations);
            printf("\tMinimization time [s]   : %.12lf\n", secs);
            printf("\tTime [s] per iteration  : %.12lf\n", secs / (st.iterations ? st.iterations : 1));
        }
        ret = r;
    });
    return ret;
}

// the lockstep L-BFGS of K problems (theta scan and batched replicates); avg / chi2 / kl: one objective half at the
// returned points, NaN for a batch whose L-BFGS parameters were refused
static void scan_minimize(bioen_b200_ctx* ctx, int method, int K, const double* thetas, const BatchPlanes& in,
                          const double* x0_host, double* x_host, lbfgs_config_params config, visual_params visual,
                          double* fmin, int* codes, int* info, double* stats, double* avg, double* chi2, double* kl,
                          const char* what) {
    ctx->pending_gen = -1;
    Context& C = ctx->C;
    CUDA_CHECK(cudaSetDevice(C.device));
    C.require_row_major("the batched theta scan");
    const auto t0 = std::chrono::steady_clock::now();
    ThetaScan scan(C, K, to_params(config), method == BIOEN_B200_FORCES, in);
    scan.verbose = (int)visual.verbose;
    const std::vector<ScanResult> res = scan.run(thetas, x0_host, x_host);
    if (avg || chi2 || kl) {
        if (scan.started) {
            scan.evaluate_all(thetas, nullptr, nullptr, nullptr, avg, chi2, kl);
        } else {
            if (avg) std::fill(avg, avg + (size_t)K * C.M, kNaN);
            if (chi2) std::fill(chi2, chi2 + K, kNaN);
            if (kl) std::fill(kl, kl + K, kNaN);
        }
    }
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    for (int q = 0; q < K; ++q) {
        if (fmin) fmin[q] = res[q].fmin;
        if (codes) codes[q] = res[q].code;
        if (info) { info[2 * q] = res[q].iterations; info[2 * q + 1] = res[q].evaluations; }
    }
    if (stats) {
        stats[0] = (double)scan.rounds;
        stats[1] = (double)scan.gemm_launches;
        stats[2] = secs;
        stats[3] = 0.0;
    }
    if (visual.verbose) {
        printf("%s: %d problems, %lld lockstep rounds, %.6f s\n", what, K, scan.rounds, secs);
        for (int q = 0; q < K; ++q)
            printf("\ttheta = %-12g %s  f = %.6lf  iterations %d\n", thetas[q], lbfgs_strerror(res[q].code),
                   res[q].fmin, res[q].iterations);
    }
}

// the per-problem inputs of a bioen_b200_batch, after the checks that do not depend on the data
static BatchPlanes batch_planes(const bioen_b200_ctx* ctx, const bioen_b200_batch* batch) {
    if (!batch || !batch->thetas) throw std::invalid_argument("bioen_b200: batch and batch->thetas are required");
    if (ctx->C.nranks > 1)
        throw std::invalid_argument("bioen_b200: batched replicates are not supported on sharded problems");
    BatchPlanes in;
    in.YTilde = batch->YTilde;
    in.row_weights = batch->row_weights;
    in.w0 = batch->w0;
    in.row_scale = batch->row_scale;
    in.row_offset = batch->row_offset;
    return in;
}

int bioen_b200_theta_scan(bioen_b200_ctx* ctx, int method, int K, const double* thetas, const double* x0_host,
                          double* x_host,
                          lbfgs_config_params config, visual_params visual, double* fmin, int* codes, int* info,
                          double* stats) {
    return guarded("bioen_b200_theta_scan", [&] {
        scan_minimize(ctx, method, K, thetas, BatchPlanes(), x0_host, x_host, config, visual, fmin, codes, info, stats,
                      nullptr, nullptr, nullptr, "theta scan");
    });
}

int bioen_b200_batch_minimize(bioen_b200_ctx* ctx, int method, const bioen_b200_batch* batch, const double* x0_host,
                              double* x_host, lbfgs_config_params config, visual_params visual, double* fmin,
                              int* codes, int* info, double* stats, double* avg, double* chi2, double* kl) {
    return guarded("bioen_b200_batch_minimize", [&] {
        const BatchPlanes in = batch_planes(ctx, batch);
        scan_minimize(ctx, method, batch->K, batch->thetas, in, x0_host, x_host, config, visual, fmin, codes, info,
                      stats, avg, chi2, kl, "batch minimisation");
    });
}

// a batch that is only evaluated, never minimised: no L-BFGS history planes (m = 0 allocates none)
static LbfgsParams evaluation_only() {
    LbfgsParams p;
    p.m = 0;
    return p;
}

int bioen_b200_batch_eval(bioen_b200_ctx* ctx, int method, const bioen_b200_batch* batch, const double* x_host,
                          double* f, double* grad_host, double* avg, double* chi2, double* kl) {
    return guarded("bioen_b200_batch_eval", [&] {
        const BatchPlanes in = batch_planes(ctx, batch);
        if (!x_host) throw std::invalid_argument("bioen_b200: x is required");
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        C.require_row_major("the batched theta scan");
        ThetaScan scan(C, batch->K, evaluation_only(), method == BIOEN_B200_FORCES, in);
        scan.evaluate_all(batch->thetas, x_host, f, grad_host, avg, chi2, kl);
    });
}

// `steps` timed batched f+g evaluations (bioen_b200_time_scan_evals: no planes, sharded contexts allowed)
static void time_batched_evals(bioen_b200_ctx* ctx, int method, int K, const double* thetas, const BatchPlanes& in,
                               const double* x0_host, int warmup, int steps, float* ms, float* gemm_ms, long long* launches) {
    ctx->pending_gen = -1;
    Context& C = ctx->C;
    CUDA_CHECK(cudaSetDevice(C.device));
    C.require_row_major("the batched theta scan");
    ThetaScan scan(C, K, evaluation_only(), method == BIOEN_B200_FORCES, in);
    scan.time_evals(thetas, x0_host, warmup, steps, ms, gemm_ms, launches);
}

int bioen_b200_time_batch_evals(bioen_b200_ctx* ctx, int method, const bioen_b200_batch* batch, const double* x0_host,
                                int warmup, int steps, float* ms, float* gemm_ms, long long* launches) {
    return guarded("bioen_b200_time_batch_evals", [&] {
        const BatchPlanes in = batch_planes(ctx, batch);
        time_batched_evals(ctx, method, batch->K, batch->thetas, in, x0_host, warmup, steps, ms, gemm_ms, launches);
    });
}

int bioen_b200_time_scan_evals(bioen_b200_ctx* ctx, int method, int K, const double* thetas, const double* x0_host,
                               int warmup, int steps, float* ms, float* gemm_ms, long long* launches) {
    return guarded("bioen_b200_time_scan_evals", [&] {
        time_batched_evals(ctx, method, K, thetas, BatchPlanes(), x0_host, warmup, steps, ms, gemm_ms, launches);
    });
}

int bioen_b200_dmma_peak(int device, double* tflops) {
    return guarded("bioen_b200_dmma_peak", [&] {
        CUDA_CHECK(cudaSetDevice(device));
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
        DevBuf<double> sink;
        sink.alloc(1);
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        const int iters = 20000, blocks = prop.multiProcessorCount * 4;
        k_dmma_peak<<<blocks, 256>>>(100, sink.p);
        float best = 1e30f;
        for (int rep = 0; rep < 3; ++rep) {
            CUDA_CHECK(cudaEventRecord(e0));
            k_dmma_peak<<<blocks, 256>>>(iters, sink.p);
            CUDA_CHECK(cudaEventRecord(e1));
            CUDA_CHECK(cudaEventSynchronize(e1));
            float t = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&t, e0, e1));
            best = std::min(best, t);
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        // 8 warps * 8 mma * 512 flop per iteration per block
        *tflops = (double)blocks * 8.0 * 8.0 * 512.0 * iters / (best * 1e-3) / 1e12;
    });
}

int bioen_b200_read_stream_peak(bioen_b200_ctx* ctx, int reps, double* gbs) {
    return guarded("bioen_b200_read_stream_peak", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        if (!C.Y) throw std::logic_error("bioen_b200: yTilde has not been uploaded");
        cudaDeviceProp prop;
        CUDA_CHECK(cudaGetDeviceProperties(&prop, C.device));
        const size_t n2 = (size_t)C.M * C.ld / 2;
        DevBuf<double> sink;
        sink.alloc(1);
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        const int blocks = prop.multiProcessorCount * 2;
        const double2* p = reinterpret_cast<const double2*>(C.Y);
        auto launch = [&] { k_read_stream<<<blocks, 1024, 0, C.stream>>>(p, n2, sink.p); };
        launch();
        double total = 0.0;
        if (reps < 1) reps = 1;
        for (int r = 0; r < reps; ++r) {
            CUDA_CHECK(cudaEventRecord(e0, C.stream));
            launch();
            CUDA_CHECK(cudaEventRecord(e1, C.stream));
            CUDA_CHECK(cudaEventSynchronize(e1));
            float t = 0.f;
            CUDA_CHECK(cudaEventElapsedTime(&t, e0, e1));
            total += t;
        }
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *gbs = (double)n2 * 16.0 * reps / (total * 1e-3) / 1e9;   // mean over reps, like the pass timing
    });
}

// host-only: the line-search state machine on a caller-supplied 1-D function (CPU tests of the host logic)
int bioen_b200_selftest_linesearch(lbfgs_config_params config, double finit, double dginit, double stp0,
                                   void (*phi)(double stp, double* f, double* dg), double* stp_out, double* f_out,
                                   int* ntrials) {
    const LbfgsParams prm = to_params(config);
    if (stp0 <= 0.) return LBFGSERR_INVALIDPARAMETERS;
    if (0 < dginit) return LBFGSERR_INCREASEGRADIENT;
    LineSearchState ls;
    ls.start(prm, finit, dginit, stp0);
    int n = 0;
    for (;;) {
        const double stp = ls.prepare();
        double f = 0.0, dg = 0.0;
        phi(stp, &f, &dg);
        ++n;
        // as the device driver does: where the search will not read the slope, the gradient half of the evaluation
        // is never run -- poison dg so that the CPU tests would notice if update() looked at it after all
        if (!ls.needs_slope(f)) dg = kNaN;
        const int verdict = ls.update(f, dg);
        if (verdict != 0) {
            if (stp_out) *stp_out = stp;
            if (f_out) *f_out = f;
            if (ntrials) *ntrials = n;
            return verdict;
        }
    }
}

// host-only: the interpolation step of GSL's Fletcher line minimisation (linear_minimize.c:25-128)
double bioen_b200_selftest_interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin,
                                       double xmax, int order) {
    return fletcher::interpolate(a, fa, fpa, b, fb, fpb, xmin, xmax, order);
}

// host-only: the tile sequence one CTA of a matrix pass walks (stream_pass.cuh, TileWalk) and the slot it writes its
// partial sums to -- the same code the kernel runs, for CPU tests of coverage and of the slot bookkeeping.
// -1: the row pass has no interleaved order.
long long bioen_b200_selftest_tilewalk(int pass_mode, int nRT, int nCB, int grid, long long chunk, int interleave,
                                       int cta, long long max_tiles, int* rt, int* cb, long long* slot, int* closes) {
    if (pass_mode == kRowPass && interleave) return -1;
    PassArgs a{};
    a.nRT = nRT; a.nCB = nCB; a.T = (long long)nRT * nCB; a.chunk = chunk; a.interleave = interleave;
    TileWalk tw;
    tw.init(pass_mode, a, cta, grid);
    long long n = 0;
    for (; tw.left > 0; tw.advance(), ++n) {
        if (n >= max_tiles) continue;
        rt[n] = (pass_mode == kRowPass) ? (int)tw.run : tw.k;
        cb[n] = (pass_mode == kRowPass) ? tw.k : (int)tw.run;
        slot[n] = tw.slot(cta, chunk);
        closes[n] = tw.closes_run() ? 1 : 0;
    }
    return n;
}
int bioen_b200_selftest_num_slots(long long run, long long L, long long chunk) { return pass_num_slots(run, L, chunk); }
int bioen_b200_selftest_slice_plan(int m, int n, int sms, long long max_dyn_smem, long long out[8]) {
    const SlicePlan p = slice_plan(m, n, sms, (size_t)max_dyn_smem);
    out[0] = p.nc; out[1] = p.ncs; out[2] = p.ms; out[3] = p.grid;
    out[4] = p.cx_log2; out[5] = p.l_log2; out[6] = p.lt_log2; out[7] = (long long)p.smem;
    return p.ok ? 1 : 0;
}

// host-only: the 2*bound+1 steps of the two-loop schedule (lbfgs.cuh, two_loop_step), 11 ints each
int bioen_b200_selftest_twoloop_schedule(int end, int bound, int m, int* steps) {
    if (m < 1 || m > 16 || bound < 1 || bound > m || end < 0 || end >= m) return -1;
    for (int t = 0; t <= 2 * bound; ++t) {
        const TwoLoopStep s = two_loop_step(t, end, bound, m);
        const int v[11] = {s.init, s.u_kind, s.u_slot, s.v_kind, s.v_slot, s.c_num, s.c_den, s.csign, s.c2_num, s.scale,
                           s.out};
        for (int i = 0; i < 11; ++i) steps[11 * t + i] = v[i];
    }
    return 2 * bound + 1;
}

// One L-BFGS direction update from a given state, on the engine the minimisers would run it on (tests compare it with
// an extended-precision two-loop recursion).  Engines 0-2 drive Lbfgs::update_direction on the context's store,
// engine 3 ThetaScan::update_directions on a batch's planes: the same host code as the minimisers.
int bioen_b200_selftest_lbfgs_update(bioen_b200_ctx* ctx, int engine, int method, int K, const int* end_old,
                                     const int* bound, const double* x, const double* g, double* xp, double* gp,
                                     double* S, double* Y, const double* ys_ring, double* d, double* scalars) {
    return guarded("bioen_b200_selftest_lbfgs_update", [&] {
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const bool forces = method == BIOEN_B200_FORCES;
        const int n = ctx->dim(method), m = kGramM;
        const size_t nm = (size_t)n * m;
        if (engine < 0 || engine > 3) throw std::invalid_argument("bioen_b200: engine must be 0..3");
        if (K < 1 || K > (engine == 3 ? kBMaxK : 1))
            throw std::invalid_argument("bioen_b200: K must be 1 (engines 0-2) or 1..32 (engine 3)");
        for (int q = 0; q < K; ++q)
            if (end_old[q] < 0 || end_old[q] >= m || bound[q] < (engine == 3 ? 0 : 1) || bound[q] > m)
                throw std::invalid_argument("bioen_b200: end_old must be in 0..5 and bound in 1..6 (0: inactive, "
                                            "engine 3)");
        auto scalar_file = [&](int q, double* dst) {
            for (int k = 0; k < SC_COUNT; ++k) dst[k] = scalars[(size_t)q * SC_COUNT + k];
            for (int t = 0; t < m; ++t) dst[SC_YS0 + t] = ys_ring[(size_t)q * m + t];
        };
        if (engine == 3) {
            if (C.nranks > 1)
                throw std::invalid_argument("bioen_b200: the batched engine runs on unsharded contexts only (a local "
                                            "group cannot carry its messages)");
            C.require_row_major("the batched theta scan");
            ThetaScan scan(C, K, LbfgsParams(), forces);
            const BatchBufs& B = scan.B;
            const long long KP = scan.KP, ldn = scan.ldn;
            auto hist = [&](double* base, int t, int q) { return base + ((size_t)t * KP + q) * ldn; };
            std::vector<double> row(SC_COUNT);
            for (int q = 0; q < K; ++q) {
                const size_t o = (size_t)q * n;
                C.h2d(B.X + q * ldn, x + o, n);
                C.h2d(B.Gr + q * ldn, g + o, n);
                C.h2d(B.XP + q * ldn, xp + o, n);
                C.h2d(B.GP + q * ldn, gp + o, n);
                C.h2d(B.D + q * ldn, d + o, n);
                for (int t = 0; t < m; ++t) {
                    C.h2d(hist(B.S, t, q), S + q * nm + (size_t)t * n, n);
                    C.h2d(hist(B.Yv, t, q), Y + q * nm + (size_t)t * n, n);
                }
                scalar_file(q, row.data());
                C.h2d(B.scb + q * SC_COUNT, row.data(), SC_COUNT);
            }
            KSlots upd{};
            std::vector<int> bnd(K, 0);
            for (int q = 0; q < K; ++q) {
                upd.mask[q] = bound[q] > 0;
                upd.slot[q] = end_old[q];
                bnd[q] = bound[q];
            }
            scan.update_directions(upd, bnd);
            for (int q = 0; q < K; ++q) {
                const size_t o = (size_t)q * n;
                C.d2h(xp + o, B.XP + q * ldn, n);
                C.d2h(gp + o, B.GP + q * ldn, n);
                C.d2h(d + o, B.D + q * ldn, n);
                for (int t = 0; t < m; ++t) {
                    C.d2h(S + q * nm + (size_t)t * n, hist(B.S, t, q), n);
                    C.d2h(Y + q * nm + (size_t)t * n, hist(B.Yv, t, q), n);
                }
                C.d2h(scalars + (size_t)q * SC_COUNT, B.scb + q * SC_COUNT, SC_COUNT);
            }
            C.sync();
            return;
        }
        Lbfgs opt(C, forces, LbfgsParams());
        if (engine == 1 && (n > kSmallUpdateMaxN || opt.reduce))
            throw std::invalid_argument("bioen_b200: the small engine takes unsharded problems of n <= 1024");
        if (engine == 2 && opt.reduce && !C.fuse_exchange())
            throw std::invalid_argument("bioen_b200: the Gram engine on a sharded context needs the fused exchange");
        // the Gram kernels take ring slots [0, bound) as the valid ones, which holds for the states a minimisation
        // reaches: the ring fills slots 0, 1, ... in order before it wraps
        if (engine == 2 && bound[0] < m && end_old[0] != bound[0] - 1)
            throw std::invalid_argument("bioen_b200: the Gram engine takes reachable states only (bound < 6 needs "
                                        "end_old = bound - 1)");
        // select the engine through the context's switches, as a minimisation would see them; restored below
        const bool gram0 = C.options.lbfgs_gram_opt, small0 = C.options.lbfgs_small_opt;
        C.options.lbfgs_gram_opt = engine == 2;
        C.options.lbfgs_small_opt = engine == 1;
        try {
            opt.x = ctx->x_for(method);
            opt.bind_store();
            C.h2d(opt.x, x, n);
            C.h2d(opt.g, g, n);
            C.h2d(opt.xp, xp, n);
            C.h2d(opt.gp, gp, n);
            C.h2d(opt.d, d, n);
            for (int t = 0; t < m; ++t) {
                C.h2d(opt.S[t], S + (size_t)t * n, n);
                C.h2d(opt.Yv[t], Y + (size_t)t * n, n);
            }
            std::vector<double> row(SC_COUNT);
            scalar_file(0, row.data());
            C.h2d(C.sc.p, row.data(), SC_COUNT);
            if (engine == 2) {
                // the resident Gram matrix of the pairs already in the ring, b = [s_0..s_5, y_0..y_5, g]: one device dot
                // per entry (three per launch along a row), summed over the ranks when sharded.  Its diagonal s_t . y_t
                // is then set to the ring's ys_t: in a minimisation both are the one value k_lbfgs_gram_pair stored.
                double* Gm = C.lbfgs_gram.p;
                auto basis = [&](int k) { return k < m ? opt.S[k] : opt.Yv[k - m]; };
                for (int a = 0; a < 2 * m; ++a)
                    for (int b = 0; b < 2 * m; b += 3) {
                        Dot3Args da{n, basis(a), basis(b), basis(a), basis(b + 1), basis(a), basis(b + 2),
                                    Gm + a * kGramB + b, C.red_partials.p, C.ticket.p};
                        k_dot3<<<opt.vec_blocks, kVecThreads, 0, C.stream>>>(da);
                    }
                CUDA_CHECK(cudaGetLastError());
                if (opt.reduce) C.comm->allreduce_sum(Gm, kGramB * kGramB, C.stream);
                for (int t = 0; t < bound[0]; ++t) {
                    if (t == end_old[0]) continue;
                    C.h2d(Gm + t * kGramB + m + t, ys_ring + t, 1);
                    C.h2d(Gm + (m + t) * kGramB + t, ys_ring + t, 1);
                }
            }
            opt.update_direction(end_old[0], bound[0], m);
            CUDA_CHECK(cudaGetLastError());
            C.d2h(xp, opt.xp, n);
            C.d2h(gp, opt.gp, n);
            C.d2h(d, opt.d, n);
            for (int t = 0; t < m; ++t) {
                C.d2h(S + (size_t)t * n, opt.S[t], n);
                C.d2h(Y + (size_t)t * n, opt.Yv[t], n);
            }
            C.d2h(scalars, C.sc.p, SC_COUNT);
            C.sync();
        } catch (...) {
            C.options.lbfgs_gram_opt = gram0;
            C.options.lbfgs_small_opt = small0;
            throw;
        }
        C.options.lbfgs_gram_opt = gram0;
        C.options.lbfgs_small_opt = small0;
    });
}

int bioen_b200_nccl_unique_id(char id[128]) {
    return guarded("bioen_b200_nccl_unique_id", [&] { Comm::unique_id(id); });
}

int bioen_b200_comm_init(bioen_b200_ctx* ctx, const char id[128], int rank, int nranks, long long n_total) {
    return guarded("bioen_b200_comm_init", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->comm.reset(new Comm(id, rank, nranks));
        ctx->C.set_comm(ctx->comm.get());
        ctx->C.N_total = n_total;
        long long cap = ctx->C.M + 16;
        if (cap < 1024) cap = 1024;
        if (cap > (long long)kP2PMaxCount) cap = (long long)kP2PMaxCount;
        ctx->comm->enable_p2p(cap, ctx->C.stream);
    });
}

// Load every kernel the collective operations launch.  With CUDA's lazy module loading the FIRST launch of a kernel
// loads it, and that load cannot overlap a running kernel of the same context: a rank of an in-process group that
// meets a kernel for the first time while its peer's exchange kernel is already spinning for it would stall both
// until the exchange times out (measured: exactly one timeout per kernel family, first call only).
static void preload_kernels() {
    cudaFuncAttributes at;
#define BIOEN_TOUCH(K) CUDA_CHECK(cudaFuncGetAttributes(&at, K))
    BIOEN_TOUCH(k_p2p_exchange); BIOEN_TOUCH(persistent_eval_kernel<double>);
    BIOEN_TOUCH(k_update_lse); BIOEN_TOUCH(k_logw_weights); BIOEN_TOUCH(k_logw_rows_exchange_finalize);
    BIOEN_TOUCH(k_reduce_row_slots); BIOEN_TOUCH(k_finalize_rows); BIOEN_TOUCH(k_logw_grad);
    BIOEN_TOUCH(k_forces_weights); BIOEN_TOUCH(k_forces_lr_from_w); BIOEN_TOUCH(k_forces_E);
    BIOEN_TOUCH(k_forces_grad); BIOEN_TOUCH(k_forces_update); BIOEN_TOUCH(k_dot3); BIOEN_TOUCH(k_axpby);
    BIOEN_TOUCH(k_lbfgs_pair); BIOEN_TOUCH(k_lbfgs_twoloop); BIOEN_TOUCH(k_lbfgs_gram_pair); BIOEN_TOUCH(k_lbfgs_combine); BIOEN_TOUCH(k_fused_lse_merge);
    BIOEN_TOUCH(k_fused_merge_rows); BIOEN_TOUCH(k_forces_lse_gather); BIOEN_TOUCH(k_forces_rows_finish); BIOEN_TOUCH(k_transpose); BIOEN_TOUCH(k_grid_max_abs);
    BIOEN_TOUCH(stream_colgrad_kernel<double>); BIOEN_TOUCH(k_colgrad_finish); BIOEN_TOUCH(k_colgrad_finish_sharded);
    BIOEN_TOUCH((stream_pass_kernel<kRowPass, false>)); BIOEN_TOUCH((stream_pass_kernel<kRowPass, true>));
    BIOEN_TOUCH((stream_pass_kernel<kColPass, false>)); BIOEN_TOUCH((stream_pass_kernel<kColPass, true>));
#undef BIOEN_TOUCH
}

int bioen_b200_comm_init_local(bioen_b200_ctx* ctx, int group, int rank, int nranks, long long n_total) {
    return guarded("bioen_b200_comm_init_local", [&] {
        ctx->pending_gen = -1;
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->comm.reset(new Comm(group, rank, nranks));
        ctx->C.set_comm(ctx->comm.get());
        ctx->C.N_total = n_total;
        long long cap = ctx->C.M + 16;
        if (cap < 1024) cap = 1024;
        if (cap > (long long)kP2PMaxCount) cap = (long long)kP2PMaxCount;
        // Ranks of an in-process group may share a device, and the CUDA runtime does not let a kernel issued after
        // a device allocation overlap a kernel of another stream issued before it: a rank that allocates between its
        // peer's exchange kernel (already spinning for this rank) and its own would stall both until the exchange
        // times out.  So everything the collective operations allocate lazily is allocated here, before the group
        // assembles (enable_local is the barrier).
        Context& C = ctx->C;
        preload_kernels();
        ctx->x_for(BIOEN_B200_LOGW);
        ctx->x_for(BIOEN_B200_FORCES);
        C.Gv.ensure(C.Npad + 8);
        C.aux_n.ensure(C.Npad + 8);
        C.aux_n2.ensure(C.Npad + 8);
        {
            const size_t nmax = (size_t)std::max(C.N, C.M);
            C.lbfgs_store.reserve(((nmax + 15) & ~(size_t)15) * (4 + 2 * (size_t)LbfgsParams().m));
            C.lbfgs_gram.reserve(kGramB * kGramB + kGramB + 3);
            C.lbfgs_gram_partials.reserve((size_t)std::max(C.vec_blocks_n, C.vec_blocks_m) * kGramK + 8);
        }
        ctx->comm->enable_local(cap, ctx->C.device);
    });
}

int bioen_b200_comm_mode(bioen_b200_ctx* ctx) { return ctx->comm ? ctx->comm->mode() : 0; }

int bioen_b200_eval_dev(bioen_b200_ctx* ctx, int method, double* x_dev, double* grad_dev) {
    return guarded("bioen_b200_eval_dev", [&] {
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        if (method == BIOEN_B200_FORCES) C.forces_eval(x_dev, nullptr, nullptr, 0.0, grad_dev, nullptr);
        else C.logw_eval(x_dev, nullptr, nullptr, 0.0, grad_dev, nullptr);
    });
}

int bioen_b200_fetch(bioen_b200_ctx* ctx, double* f, double* gnorm2) {
    return guarded("bioen_b200_fetch", [&] {
        CUDA_CHECK(cudaSetDevice(ctx->C.device));
        ctx->C.fetch_scalars();
        if (f) *f = ctx->C.h_sc[SC_F];
        if (gnorm2) *gnorm2 = ctx->C.h_sc[SC_GNORM2];
    });
}

int bioen_b200_time_evals(bioen_b200_ctx* ctx, int method, double* x_dev, double* grad_dev, int warmup, int steps,
                          float* ms, float* pass_ms, long long* launches) {
    return guarded("bioen_b200_time_evals", [&] {
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const bool forces = (method == BIOEN_B200_FORCES);
        const int n = forces ? C.M : C.N;
        const int blocks = forces ? C.vec_blocks_m : C.vec_blocks_n;
        // direction: a copy of the start point's gradient scaled tiny, so every step evaluates a new point
        DevBuf<double> xp, dir;
        xp.alloc(((size_t)n + 15) & ~(size_t)15);
        dir.alloc(((size_t)n + 15) & ~(size_t)15);
        C.d2d(xp.p, x_dev, n);
        if (forces) C.forces_eval(x_dev, nullptr, nullptr, 0.0, grad_dev, nullptr);
        else C.logw_eval(x_dev, nullptr, nullptr, 0.0, grad_dev, nullptr);
        C.fetch_scalars();
        const double gn = std::sqrt(C.h_sc[SC_GNORM2]);
        k_axpby<<<blocks, kVecThreads, 0, C.stream>>>(n, gn > 0 ? -1e-6 / gn : 0.0, grad_dev, 0.0, nullptr, dir.p);
        auto one = [&](int k) {
            if (forces) C.forces_eval(x_dev, xp.p, dir.p, (double)(k + 1), grad_dev, dir.p);
            else C.logw_eval(x_dev, xp.p, dir.p, (double)(k + 1), grad_dev, dir.p);
        };
        for (int k = 0; k < warmup; ++k) one(k);
        C.sync();
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        C.begin_pass_timing(steps * 4);
        const long long k0 = bioen_b200_kernels_launched(ctx);
        CUDA_CHECK(cudaEventRecord(e0, C.stream));
        for (int k = 0; k < steps; ++k) one(warmup + k);
        CUDA_CHECK(cudaEventRecord(e1, C.stream));
        CUDA_CHECK(cudaEventSynchronize(e1));
        float total = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&total, e0, e1));
        if (ms) *ms = total;
        if (launches) *launches = bioen_b200_kernels_launched(ctx) - k0;
        float pm = C.end_pass_timing();
        // one-launch evaluations (slice kernel): no per-pass events; report the step's share per algorithmic pass
        // (the same for the persistent kernel: its launches are not bracketed by events either)
        if (pm == 0.f && steps > 0 && C.persistent_for(forces) && (!forces || C.have_forces))
            pm = total / (float)steps / (forces ? 4.f : 2.f);
        if (pass_ms) *pass_ms = pm;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    });
}

int bioen_b200_generate_ytilde(bioen_b200_ctx* ctx, unsigned long long seed, long long col_offset,
                               const double* ytrue_over_sigma_host, double inv_sigma) {
    return guarded("bioen_b200_generate_ytilde", [&] {
        ctx->pending_gen = -1;
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        if (C.yt_only) {
            C.alloc_yt();
            C.h2d(C.avg.p, ytrue_over_sigma_host, C.M);
            k_generate_t<<<C.num_sms * 8, 256, 0, C.stream>>>(C.Yt.p, C.ldt, C.M, C.N, seed, col_offset, C.avg.p, inv_sigma);
            CUDA_CHECK(cudaGetLastError());
            ++C.kernels_launched;
            ++C.eval_gen;
            C.sync();
            return;
        }
        if (!C.Y) C.alloc_matrix();
        C.h2d(C.avg.p, ytrue_over_sigma_host, C.M);
        k_generate<<<C.num_sms * 8, 256, 0, C.stream>>>(C.Y, C.ld, C.M, C.N, seed, col_offset, C.avg.p, inv_sigma);
        CUDA_CHECK(cudaGetLastError());
        ++C.kernels_launched;
        C.sync();
    });
}

int bioen_b200_download_ytilde(bioen_b200_ctx* ctx, int row0, int nrows, long long col0, long long ncols,
                               double* out_host) {
    return guarded("bioen_b200_download_ytilde", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        if (C.storage_fp32) throw std::logic_error("bioen_b200: the resident matrix is stored in fp32 (no fp64 copy to download)");
        if (C.yt_only) {
            if (row0 < 0 || nrows <= 0 || row0 + nrows > C.M || col0 < 0 || ncols <= 0 || col0 + ncols > C.N)
                throw std::invalid_argument("bioen_b200: block out of range");
            C.download_yt(row0, nrows, col0, ncols, out_host);
            return;
        }
        if (!C.Y) throw std::logic_error("bioen_b200: no matrix");
        if (row0 < 0 || nrows < 0 || row0 + nrows > C.M || col0 < 0 || ncols < 0 || col0 + ncols > C.N)
            throw std::invalid_argument("bioen_b200: block out of range");
        CUDA_CHECK(cudaMemcpy2DAsync(out_host, (size_t)ncols * sizeof(double), C.Y + (size_t)row0 * C.ld + col0,
                                     (size_t)C.ld * sizeof(double), (size_t)ncols * sizeof(double), nrows,
                                     cudaMemcpyDeviceToHost, C.stream));
        C.sync();
    });
}

long long bioen_b200_kernels_launched(bioen_b200_ctx* ctx) {
    return ctx->C.kernels_launched + (ctx->comm ? ctx->comm->p2p_launches : 0);
}

long long bioen_b200_query(bioen_b200_ctx* ctx, int what) {
    Context& C = ctx->C;
    switch (what) {
        case 0: return C.forces_fused_now() ? 1 : 0;
        case 1: return C.nranks > 1 ? C.exchanges_per_eval(false) : 0;
        case 2: return C.nranks > 1 ? C.exchanges_per_eval(true) : 0;
        case 3: return C.persistent_for(what == 3 && C.have_forces) ? 1 : 0;
        case 4: return C.storage_fp32 ? 4 : 8;
        case 5: return C.persistent_launches;
        case 6: return C.slice_launches;
        case 7: return C.slice_ok() ? 1 : 0;
        case 8: return (long long)((C.Yown.p ? C.Yown.n * 8 : 0) + (C.Yt.p ? C.Yt.n * 8 : 0) + (C.Y32.p ? C.Y32.n * 4 : 0));
        case 9: return C.yt_only ? 1 : 0;
        case 10: {
            const ContextOptions& o = C.options;
            const ContextOptions d{};
            auto bit = [](bool differs, int option) { return differs ? 1LL << option : 0LL; };
            return bit(o.allow_fused != d.allow_fused, BIOEN_B200_OPT_FUSED_FORCES) |
                   bit(o.lazy_gradient != d.lazy_gradient, BIOEN_B200_OPT_LAZY_GRADIENT) |
                   bit(o.fuse_allowed != d.fuse_allowed, BIOEN_B200_OPT_FUSED_EXCHANGE) |
                   bit(o.persistent_mode != d.persistent_mode, BIOEN_B200_OPT_PERSISTENT) |
                   bit(o.lbfgs_gram_opt != d.lbfgs_gram_opt, BIOEN_B200_OPT_LBFGS_GRAM) |
                   bit(o.slice_mode != d.slice_mode, BIOEN_B200_OPT_SLICE) |
                   bit(o.lbfgs_small_opt != d.lbfgs_small_opt, BIOEN_B200_OPT_LBFGS_SMALL) |
                   bit(o.lbfgs_speculative != d.lbfgs_speculative, BIOEN_B200_OPT_LBFGS_SPECULATIVE) |
                   bit(o.fetch_zero_copy != d.fetch_zero_copy, BIOEN_B200_OPT_FETCH_ZEROCOPY);
        }
        default: return -1;
    }
}

int bioen_b200_debug_read(bioen_b200_ctx* ctx, int what, double* out_host, size_t count) {
    return guarded("bioen_b200_debug_read", [&] {
        Context& C = ctx->C;
        CUDA_CHECK(cudaSetDevice(C.device));
        const double* src = nullptr;
        size_t cap = 0;
        switch (what) {
            case 0: src = C.sc.p; cap = SC_COUNT; break;
            case 1: src = C.w.p; cap = C.N; break;
            case 2: src = C.avg.p; cap = C.M; break;
            case 3: src = C.aux_n.p; cap = C.aux_n.n; break;
            case 4: src = C.aux_n2.p; cap = C.aux_n2.n; break;
            case 5: src = C.lbfgs_store.p; cap = C.lbfgs_store.n; break;
            default: throw std::invalid_argument("bioen_b200: unknown debug buffer");
        }
        if (count > cap) throw std::invalid_argument("bioen_b200: debug read too long");
        C.d2h(out_host, src, count);
        C.sync();
    });
}

void* bioen_b200_stream(bioen_b200_ctx* ctx) { return (void*)ctx->C.stream; }

// ---------------------------------------------------------------------------------------------------
// Part 1 -- reference-compatible symbols (host pointers in, host pointers out)
// ---------------------------------------------------------------------------------------------------
namespace {
struct TempProblem {
    bioen_b200_ctx* ctx = nullptr;
    // fused = false: the caller needs only weights or the given-weights entry points, which run on the tile kernels;
    // no structure-major copy is made then
    TempProblem(int m, int n, const double* yTilde, bool fused = true) {
        ctx = bioen_b200_create(m, n, default_device());
        if (!ctx) throw std::runtime_error(g_last_error);
        try {
            ctx->C.options.allow_fused = fused;
            if (yTilde) ctx->C.upload_matrix(yTilde, (size_t)n);
        } catch (...) {
            bioen_b200_destroy(ctx);
            ctx = nullptr;
            throw;
        }
    }
    ~TempProblem() { bioen_b200_destroy(ctx); }
};
}  // namespace

double _get_weights(const double* g, double* w, size_t n) {
    double s = kNaN;
    guarded("_get_weights", [&] {
        TempProblem P(1, (int)n, nullptr);
        double sum = 0.0;
        Context& C = P.ctx->C;
        double* x = P.ctx->x_for(BIOEN_B200_LOGW);
        C.h2d(x, g, n);
        C.logw_weights_only(x);
        C.d2h(w, C.w.p, n);
        C.fetch_scalars();
        sum = std::exp(C.h_sc[SC_GMAX]) * C.h_sc[SC_S];
        s = sum;
    });
    return s;
}

double _bioen_log_posterior_logw(const double* g, const double* G, const double* yTilde, const double* YTilde,
                                 const double* /*w*/, const double* /*gradient*/, double theta, int /*caching*/,
                                 const double* /*yTildeT*/, double* /*tmp_n*/, double* /*tmp_m*/, int m, int n,
                                 double /*weights_sum*/) {
    double f = kNaN;
    guarded("_bioen_log_posterior_logw", [&] {
        TempProblem P(m, n, yTilde);
        if (bioen_b200_set_logw(P.ctx, G, YTilde, theta)) throw std::runtime_error(g_last_error);
        if (bioen_b200_eval(P.ctx, BIOEN_B200_LOGW, g, &f, nullptr)) throw std::runtime_error(g_last_error);
    });
    return f;
}

void _grad_bioen_log_posterior_logw(const double* g, const double* G, const double* yTilde, const double* YTilde,
                                    const double* /*w*/, double* gradient, double theta, int /*caching*/,
                                    const double* /*yTildeT*/, double* /*tmp_n*/, double* /*tmp_m*/, int m, int n,
                                    double /*weights_sum*/) {
    guarded("_grad_bioen_log_posterior_logw", [&] {
        TempProblem P(m, n, yTilde);
        double f;
        if (bioen_b200_set_logw(P.ctx, G, YTilde, theta)) throw std::runtime_error(g_last_error);
        if (bioen_b200_eval(P.ctx, BIOEN_B200_LOGW, g, &f, gradient)) throw std::runtime_error(g_last_error);
    });
}

double _opt_lbfgs_logw(params_t p, lbfgs_config_params config, visual_params visual, int* error) {
    double fmin = kNaN;
    int err = -2000;
    guarded("_opt_lbfgs_logw", [&] {
        TempProblem P(p.m, p.n, p.yTilde);
        int info[4];
        if (bioen_b200_set_logw(P.ctx, p.G, p.YTilde, p.theta)) throw std::runtime_error(g_last_error);
        err = bioen_b200_opt_lbfgs(P.ctx, BIOEN_B200_LOGW, p.g, p.result, config, visual, &fmin, info);
        if (err == -2000) throw std::runtime_error(g_last_error);
    });
    if (error) *error = err;
    return fmin;
}

double _opt_bfgs_logw(params_t p, gsl_config_params config, visual_params visual, int* error) {
    double fmin = kNaN;
    int err = -2000;
    guarded("_opt_bfgs_logw", [&] {
        TempProblem P(p.m, p.n, p.yTilde);
        int info[4];
        if (bioen_b200_set_logw(P.ctx, p.G, p.YTilde, p.theta)) throw std::runtime_error(g_last_error);
        err = bioen_b200_opt_gsl(P.ctx, BIOEN_B200_LOGW, p.g, p.result, config, visual, &fmin, info);
        if (err == -2000) throw std::runtime_error(g_last_error);
    });
    if (error) *error = err;
    return fmin;
}

void _get_weights_from_forces(const double* w0, const double* yTilde, const double* forces, double* w,
                              int /*caching*/, const double* /*yTildeT*/, double* /*tmp_n*/, size_t m, size_t n) {
    guarded("_get_weights_from_forces", [&] {
        TempProblem P((int)m, (int)n, yTilde, false);
        std::vector<double> zeros(m, 0.0);
        if (bioen_b200_set_forces(P.ctx, w0, zeros.data(), 0.0)) throw std::runtime_error(g_last_error);
        if (bioen_b200_weights(P.ctx, BIOEN_B200_FORCES, forces, w, nullptr)) throw std::runtime_error(g_last_error);
    });
}

double _bioen_log_posterior_forces(const double* w0, const double* yTilde, const double* YTilde, const double* w,
                                   const double* /*result*/, double theta, int /*caching*/,
                                   const double* /*yTildeT*/, double* /*tmp_n*/, double* /*tmp_m*/, int m, int n) {
    double f = kNaN;
    guarded("_bioen_log_posterior_forces", [&] {
        TempProblem P(m, n, yTilde, false);
        if (bioen_b200_set_forces(P.ctx, w0, YTilde, theta)) throw std::runtime_error(g_last_error);
        if (bioen_b200_forces_from_weights(P.ctx, w, &f, nullptr)) throw std::runtime_error(g_last_error);
    });
    return f;
}

void _grad_bioen_log_posterior_forces(const double* w0, const double* yTilde, const double* YTilde, const double* w,
                                      double* gradient, double theta, int /*caching*/, const double* /*yTildeT*/,
                                      double* /*tmp_n*/, double* /*tmp_m*/, int m, int n) {
    guarded("_grad_bioen_log_posterior_forces", [&] {
        TempProblem P(m, n, yTilde, false);
        double f;
        if (bioen_b200_set_forces(P.ctx, w0, YTilde, theta)) throw std::runtime_error(g_last_error);
        if (bioen_b200_forces_from_weights(P.ctx, w, &f, gradient)) throw std::runtime_error(g_last_error);
    });
}

double _opt_lbfgs_forces(params_t p, lbfgs_config_params config, visual_params visual, int* error) {
    double fmin = kNaN;
    int err = -2000;
    guarded("_opt_lbfgs_forces", [&] {
        TempProblem P(p.m, p.n, p.yTilde);
        int info[4];
        if (bioen_b200_set_forces(P.ctx, p.w0, p.YTilde, p.theta)) throw std::runtime_error(g_last_error);
        err = bioen_b200_opt_lbfgs(P.ctx, BIOEN_B200_FORCES, p.forces, p.result, config, visual, &fmin, info);
        if (err == -2000) throw std::runtime_error(g_last_error);
    });
    if (error) *error = err;
    return fmin;
}

double _opt_bfgs_forces(params_t p, gsl_config_params config, visual_params visual, int* error) {
    double fmin = kNaN;
    int err = -2000;
    guarded("_opt_bfgs_forces", [&] {
        TempProblem P(p.m, p.n, p.yTilde);
        int info[4];
        if (bioen_b200_set_forces(P.ctx, p.w0, p.YTilde, p.theta)) throw std::runtime_error(g_last_error);
        err = bioen_b200_opt_gsl(P.ctx, BIOEN_B200_FORCES, p.forces, p.result, config, visual, &fmin, info);
        if (err == -2000) throw std::runtime_error(g_last_error);
    });
    if (error) *error = err;
    return fmin;
}

int _library_gsl(void) { return 1; }
int _library_lbfgs(void) { return 1; }
void _omp_set_num_threads(int) {}
void _set_fast_openmp_flag(int flag) { g_fast_flag = flag; }
int _get_fast_openmp_flag(void) { return g_fast_flag; }

// message texts: the public strings of GSL 2.5 err/strerror.c and of c_bioen_error.c:25-115
const char* bioen_gsl_error(int e) {
    switch (e) {
        case 0: return "success";
        case -1: return "failure";
        case -2: return "the iteration has not converged yet";
        case 1: return "input domain error";
        case 2: return "output range error";
        case 3: return "invalid pointer";
        case 4: return "invalid argument supplied by user";
        case 5: return "generic failure";
        case 6: return "factorization failed";
        case 7: return "sanity check failed - shouldn't happen";
        case 8: return "malloc failed";
        case 9: return "problem with user-supplied function";
        case 10: return "iterative process is out of control";
        case 11: return "exceeded max number of iterations";
        case 12: return "tried to divide by zero";
        case 13: return "specified tolerance is invalid or theoretically unattainable";
        case 14: return "failed to reach the specified tolerance";
        case 15: return "underflow";
        case 16: return "overflow";
        case 17: return "loss of accuracy";
        case 18: return "roundoff error";
        case 19: return "matrix/vector sizes are not conformant";
        case 20: return "matrix not square";
        case 21: return "singularity or extremely bad function behavior detected";
        case 22: return "integral or series is divergent";
        case 23: return "the required feature is not supported by this hardware platform";
        case 24: return "the requested feature is not (yet) implemented";
        case 25: return "cache limit exceeded";
        case 26: return "table limit exceeded";
        case 27: return "iteration is not making progress towards solution";
        case 28: return "jacobian evaluations are not improving the solution";
        case 29: return "cannot reach the specified tolerance in F";
        case 30: return "cannot reach the specified tolerance in X";
        case 31: return "cannot reach the specified tolerance in gradient";
        case 32: return "end of file";
        default: return "unknown error code";
    }
}

const char* lbfgs_strerror(int e) {
    static const char* const neg[] = {
        /* -1024 */ "Unknown error.",
        /* -1023 */ "Logic error.",
        /* -1022 */ "Insufficient memory.",
        /* -1021 */ "The minimization process has been canceled.",
        /* -1020 */ "Invalid number of variables specified.",
        /* -1019 */ "Invalid number of variables (for SSE) specified.",
        /* -1018 */ "The array x must be aligned to 16 (for SSE).",
        /* -1017 */ "Invalid parameter lbfgs_parameter_t::epsilon specified.",
        /* -1016 */ "Invalid parameter lbfgs_parameter_t::past specified.",
        /* -1015 */ "Invalid parameter lbfgs_parameter_t::delta specified.",
        /* -1014 */ "Invalid parameter lbfgs_parameter_t::linesearch specified.",
        /* -1013 */ "Invalid parameter lbfgs_parameter_t::max_step specified",
        /* -1012 */ "Invalid parameter lbfgs_parameter_t::max_step specified.",
        /* -1011 */ "Invalid parameter lbfgs_parameter_t::ftol specified.",
        /* -1010 */ "Invalid parameter lbfgs_parameter_t::wolfe specified.",
        /* -1009 */ "Invalid parameter lbfgs_parameter_t::gtol specified.",
        /* -1008 */ "Invalid parameter lbfgs_parameter_t::xtol specified.",
        /* -1007 */ "Invalid parameter lbfgs_parameter_t::max_linesearch specified.",
        /* -1006 */ "Invalid parameter lbfgs_parameter_t::orthantwise_c specified.",
        /* -1005 */ "Invalid parameter lbfgs_parameter_t::orthantwise_start specified.",
        /* -1004 */ "Invalid parameter lbfgs_parameter_t::orthantwise_end specified.",
        /* -1003 */ "The line-search step went out of the interval of uncertainty.",
        /* -1002 */ "A logic error occurred; alternatively, the interval of uncertainty",
        /* -1001 */
        "A rounding error occurred; alternatively, no line-search step satisfies the sufficient decrease and "
        "curvature conditions.",
        /* -1000 */ "The line-search step became smaller than lbfgs_parameter_t::min_step.",
        /*  -999 */ "The line-search step became larger than lbfgs_parameter_t::max_step.",
        /*  -998 */ "The line-search routine reaches the maximum number of evaluations.",
        /*  -997 */ "The algorithm routine reaches the maximum number of iterations.",
        /*  -996 */ "Relative width of the interval of uncertainty is at most lbfgs_parameter_t::xtol.",
        /*  -995 */ "A logic error (negative line-search step) occurred.",
        /*  -994 */ "The current search direction increases the objective function value.",
    };
    if (e == 0) return "Convergence reached.";
    if (e == 1) return "LBFGS_STOP";
    if (e == 2) return "The initial variables already minimize the objective function.";
    if (e >= -1024 && e <= -994) return neg[e + 1024];
    return "(unknown)";
}

}  // extern "C"
