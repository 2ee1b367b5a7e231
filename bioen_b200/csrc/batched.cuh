// batched.cuh -- K <= 32 problems that share yTilde are minimised TOGETHER, so that the two matrix passes of an
// evaluation become skinny fp64 GEMMs  avg[M x K] = Y . W[N x K]  and  c[N x K] = Yt . R[M x K]  and yTilde is
// streamed from HBM once per pass for all K problems instead of K times.  The problems differ in theta and start
// point (the theta scan, the L-curve) and, optionally, in YTilde, in observable weights c_i of chi^2 = 1/2 sum c r^2,
// and (forces) in the reference weights w0: bootstrap and cross-validation replicates (DESIGN.md section 4g).  This is the only place the library uses tensor cores:
// fp64 has no tcgen05 kind on Blackwell, so the GEMMs are warp-level DMMA (mma.sync.m8n8k4.f64) fed by TMA.
//
// What the reference does for the same job: a Python loop over theta calling find_optimum once per value
// (bioen/analyze/procedure.py:62-83; the ala5 notebook's run_theta_series), every evaluation streaming yTilde
// three times (SURVEY.md section 2a).
//
// Layouts
//   per-problem N-vectors  [k][j]   K planes of ldn doubles (x, grad, xp, gp, d, s[m], y[m]): every vector kernel
//                                   is launched with blockIdx.y = k and is perfectly coalesced along j
//   GEMM "B" operands      fragment-major: block (q = index/4, t = k/8) holds its 4 x 8 values in the order the
//                                   m8n8k4 B fragment wants them (lane = (k%8)*4 + index%4), so a warp reads one
//                                   fragment with ONE conflict-free 256-byte shared-memory load.  W (weights,
//                                   index = j) and R (residuals, index = i) are WRITTEN in this order by the
//                                   kernels that produce them; they never exist in any other layout.
//   GEMM "A" operand       yTilde itself (row pass) / its structure-major copy Yt (column pass), streamed as
//                                   256-row x 16-column boxes with the 128-byte TMA swizzle, which makes the
//                                   8 x 4 A-fragment loads conflict-free too.
//
// The K L-BFGS state machines (liblbfgs semantics, same code path as lbfgs.cuh: parameter checks, stop tests,
// More-Thuente / backtracking line searches, m = 6) run in lockstep rounds on the host: one batched evaluation
// per round serves one line-search trial of every active problem; problems that finish drop out (masked).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <vector>

#include "context.cuh"
#include "lbfgs.cuh"

namespace bioen {

constexpr int kBMaxK = 32;          // problems per batch (planes); padded to a multiple of 8
constexpr int kGRows = 256;         // GEMM tile: rows per CTA
constexpr int kGKdim = 16;          // GEMM tile: reduction extent per stage (16 doubles = one 128-byte swizzle row)
#ifndef BIOEN_GEMM_STAGES
#define BIOEN_GEMM_STAGES 5
#endif
constexpr int kGStages = BIOEN_GEMM_STAGES;
constexpr int kGWarps = 8;
constexpr int kGThreads = (kGWarps + 1) * 32;
constexpr int kGTileBytes = kGRows * kGKdim * 8;   // 32 KB

__device__ __forceinline__ void dmma_m8n8k4(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1])
                 : "d"(a), "d"(b));
}

// register-resident DMMA loop: the fp64 tensor-core peak this GPU can actually deliver (bench.py's roofline
// denominator for the batched GEMMs; MEASURED_PEAKS.json has no fp64 figure)
__global__ void __launch_bounds__(256) k_dmma_peak(int iters, double* sink) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = 0.0;
    const double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dmma_m8n8k4(c[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    if (s == 123.456) sink[0] = s;
}

// position of element (index, k) inside a fragment-major B operand with KP = 8*NT problems
__host__ __device__ __forceinline__ size_t frag_index(long long index, int k, int NT) {
    return ((size_t)(index >> 2) * NT + (k >> 3)) * 32 + (size_t)((k & 7) * 4 + (int)(index & 3));
}

struct GemmArgs {
    int rows, kdim;          // logical extents of A
    int RB, S;               // row blocks, segments of the reduction axis
    int ktiles, tps;         // reduction tiles in total / per segment
    int KP;                  // 8 * NT
    const double* B;         // fragment-major, zero padded to ktiles*16 indices
    double* out;             // out[(seg*KP + k)*ldo + row]
    long long ldo;
    int evict_first;
};

// D[rows x KP] (+)= A[rows x kdim] . B[kdim x KP] on fp64 tensor cores; persistent over (row block, segment) items
template <int NT>
__global__ void __launch_bounds__(kGThreads, 1)
    batched_gemm_kernel(const __grid_constant__ CUtensorMap tmap, const GemmArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // swizzle needs 1 KB
    constexpr int kBBytes = kGKdim * NT * 8 * 8;            // B slice per stage
    constexpr int kStage = kGTileBytes + 4096;              // A tile + room for the largest B slice (NT = 4)
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)kGStages * kStage);
    uint64_t* empty = full + kGStages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int items = a.RB * a.S;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kGStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kGWarps);
        }
        fence_barrier_init();
    }
    __syncthreads();

    if (warp == kGWarps) {
        if (lane == 0) {
            prefetch_tensormap(&tmap);
            const uint64_t policy = a.evict_first ? l2_policy_evict_first() : l2_policy_evict_last();
            int stage = 0;
            uint32_t phase = 1;
            for (int t = blockIdx.x; t < items; t += gridDim.x) {
                const int rb = t / a.S, seg = t - rb * a.S;
                const int k0 = seg * a.tps, k1 = min(k0 + a.tps, a.ktiles);
                for (int kt = k0; kt < k1; ++kt) {
                    unsigned char* st = smem + (size_t)stage * kStage;
                    mbar_wait(&empty[stage], phase);
                    mbar_expect_tx(&full[stage], kGTileBytes + kBBytes);
                    tma_load_2d(st, &tmap, kt * kGKdim, rb * kGRows, &full[stage], policy);
                    bulk_load_1d(st + kGTileBytes, a.B + (size_t)kt * kGKdim * a.KP, kBBytes, &full[stage]);
                    if (++stage == kGStages) { stage = 0; phase ^= 1; }
                }
            }
        }
        return;
    }

    // consumers: warp w owns rows 32w .. 32w+31 of the block = 4 m-tiles of 8 rows, all NT n-tiles
    double acc[4][NT][2];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
    // swizzled A-fragment offsets: element (row, col) lives at row*128 + ((col/2) ^ (row%8))*16 + (col%2)*8
    const int g = lane >> 2, tg = lane & 3;
    uint32_t aoff[4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) aoff[ks] = (uint32_t)((((ks * 2 + (tg >> 1)) ^ g) << 4) + ((tg & 1) << 3));
    const uint32_t rowbase = (uint32_t)(warp * 32 + g) * 128u;

    int stage = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < items; t += gridDim.x) {
        const int rb = t / a.S, seg = t - rb * a.S;
        const int k0 = seg * a.tps, k1 = min(k0 + a.tps, a.ktiles);
        for (int kt = k0; kt < k1; ++kt) {
            const unsigned char* st = smem + (size_t)stage * kStage;
            mbar_wait(&full[stage], phase);
            const double* Bs = reinterpret_cast<const double*>(st + kGTileBytes);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                double af[4], bf[NT];
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
                    af[mt] = *reinterpret_cast<const double*>(st + rowbase + (uint32_t)mt * 1024u + aoff[ks]);
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) bf[nt] = Bs[(ks * NT + nt) * 32 + lane];
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) dmma_m8n8k4(acc[mt][nt], af[mt], bf[nt]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == kGStages) { stage = 0; phase ^= 1; }
        }
        // D fragment: row = g, columns 2*tg, 2*tg+1 of each 8 x 8 tile
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            const long long row = (long long)rb * kGRows + warp * 32 + mt * 8 + g;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int k = nt * 8 + tg * 2;
                if (row < a.rows) {
                    a.out[((size_t)seg * a.KP + k) * a.ldo + row] = acc[mt][nt][0];
                    a.out[((size_t)seg * a.KP + k + 1) * a.ldo + row] = acc[mt][nt][1];
                }
                acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// batched vector kernels: blockIdx.y = problem k.  Per-problem scalars live in scb[k][SC_COUNT] with the same
// slot numbers as the single-problem path (vector_kernels.cuh); per-problem launch parameters travel by value.
// Per-problem inputs (YTilde, observable weights, forces w0) are planes read at base + k * stride (BatchBufs).
// ------------------------------------------------------------------------------------------------
struct KVec {
    double stp[kBMaxK];
    double theta[kBMaxK];
    int mask[kBMaxK];      // 0: the plane is left untouched
};

struct BatchBufs {
    int n, K, KP, NT;
    long long ldn;              // plane stride
    double *X, *Gr, *XP, *GP, *D;
    double* S;                  // [m][KP][ldn]
    double* Yv;                 // [m][KP][ldn]
    double* Wf;                 // fragment-major weights
    double* Rf;                 // fragment-major residuals
    double* avgp;               // row-pass partials [S][KP][ldo]
    double* scb;                // [KP][SC_COUNT]
    double* partials;           // [KP][pstride]
    unsigned int* ticket;       // [KP]
    long long pstride;
    // Per-problem inputs.  Problem k reads its plane at base + k * stride; stride 0 = every problem reads the shared
    // vector.  Cw == nullptr: no observable weights (chi^2 = 1/2 r.r, nothing is multiplied).
    const double* G;            // reference log-weights (logw, always shared) / reference weights w0 (forces)
    long long gld = 0;          // 0 or ldN (forces only)
    const double* Yobs;         // YTilde
    long long yld = 0;          // 0 or ldo
    const double* Cw = nullptr; // [KP][ldo] observable weights c_k,i: chi^2 = 1/2 sum_i c r^2, gradients use c r
    // forces scan only: the variables are M-dimensional planes; these are the structure-axis work planes
    int nN = 0;                 // structures
    long long ldN = 0;
    double *Xn = nullptr, *LR = nullptr, *Tn = nullptr;   // [KP][ldN]: x_j = (Yt f)_j, log(w_j/w0_j), t_j
    double* Ff = nullptr;       // fragment-major forces (index = i)
    double* avgk = nullptr;     // [KP][ldo] averages of the last objective half (both methods)
    long long ldo = 0;
};

__global__ void __launch_bounds__(kVecThreads) kb_update_lse(const BatchBufs b, const KVec p, int move) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[3 * 32];
    __shared__ bool is_last;
    double* x = b.X + (size_t)k * b.ldn;
    const double* xp = b.XP + (size_t)k * b.ldn;
    const double* d = b.D + (size_t)k * b.ldn;
    const double stp = p.stp[k];
    double m = -DBL_MAX, s = 0.0, xn = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < b.n; j += gridDim.x * blockDim.x) {
        double v;
        if (move) { v = fma(stp, d[j], xp[j]); x[j] = v; }
        else v = x[j];
        xn = fma(v, v, xn);
        if (v > m) { s = s * exp(m - v) + 1.0; m = v; }
        else s += exp(v - m);
    }
    double* partials = b.partials + (size_t)k * b.pstride;
    block_lse(m, s, xn, red);
    if (threadIdx.x == 0) {
        partials[blockIdx.x * 3 + 0] = m;
        partials[blockIdx.x * 3 + 1] = s;
        partials[blockIdx.x * 3 + 2] = xn;
        __threadfence();
        is_last = (atomicAdd(b.ticket + k, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        m = -DBL_MAX; s = 0.0; xn = 0.0;
        for (unsigned q = threadIdx.x; q < gridDim.x; q += blockDim.x) {
            lse_merge(m, s, __ldcg(&partials[q * 3]), __ldcg(&partials[q * 3 + 1]));
            xn += __ldcg(&partials[q * 3 + 2]);
        }
        block_lse(m, s, xn, red);
        if (threadIdx.x == 0) {
            double* sc = b.scb + (size_t)k * SC_COUNT;
            sc[SC_GMAX] = m;
            sc[SC_S] = s;
            sc[SC_XNORM2] = xn;
            b.ticket[k] = 0;
        }
    }
}

// weights in fragment-major order + the three weighted sums of the prior; each thread owns 4 consecutive j
__global__ void __launch_bounds__(kVecThreads) kb_weights(const BatchBufs b, const KVec p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[3 * 32];
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const double M = sc[SC_GMAX], inv = 1.0 / sc[SC_S];
    const double* x = b.X + (size_t)k * b.ldn;
    double v[3] = {0.0, 0.0, 0.0};
    const int nq = (b.n + 3) >> 2;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
        double w4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = 4 * q + e;
            double w = 0.0;
            if (j < b.n) {
                const double gj = x[j], Gj = b.G[j];
                w = exp(gj - M) * inv;
                v[0] = fma(gj - Gj, w, v[0]);
                v[1] = fma(gj, w, v[1]);
                v[2] = fma(Gj, w, v[2]);
            }
            w4[e] = w;
        }
        double* dst = b.Wf + ((size_t)q * b.NT + (k >> 3)) * 32 + (k & 7) * 4;
        *reinterpret_cast<double2*>(dst) = make_double2(w4[0], w4[1]);
        *reinterpret_cast<double2*>(dst + 2) = make_double2(w4[2], w4[3]);
    }
    grid_sum<3>(v, b.partials + (size_t)k * b.pstride, b.ticket + k, red, [=](const double(&t)[3]) {
        sc[SC_TMP0] = t[0];
        sc[SC_GBAR] = t[1];
        sc[SC_CAPGBAR] = t[2];
    });
}

// finish the batched row pass: avg, r (fragment-major), chi^2, sum_i r_i avg_i, objective   (one block per k)
__global__ void __launch_bounds__(1024) kb_finalize(const BatchBufs b, const KVec p, int m, int nseg, long long ldo) {
    const int k = blockIdx.x;
    if (!p.mask[k]) return;
    __shared__ double red[2 * 32];
    const double* Y = b.Yobs + (size_t)k * b.yld;
    const double* c = b.Cw ? b.Cw + (size_t)k * b.ldo : nullptr;
    double v[2] = {0.0, 0.0};
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < nseg; ++q) s += b.avgp[((size_t)q * b.KP + k) * ldo + i];
        b.avgk[(size_t)k * b.ldo + i] = s;
        const double r = s - Y[i];
        const double cr = c ? c[i] * r : r;
        b.Rf[frag_index(i, k, b.NT)] = cr;
        v[0] = fma(cr, r, v[0]);
        v[1] = fma(cr, s, v[1]);
    }
    block_sum<2>(v, red);
    if (threadIdx.x == 0) {
        double* sc = b.scb + (size_t)k * SC_COUNT;
        const double chi2 = 0.5 * v[0];
        const double kl = sc[SC_TMP0] - (sc[SC_GMAX] + log(sc[SC_S])) + sc[SC_LOGS0];
        const double prior = kl * p.theta[k];
        sc[SC_KL] = kl;
        sc[SC_CHI2] = chi2;
        sc[SC_PRIOR] = prior;
        sc[SC_F] = prior + chi2;
        sc[SC_TMP0 + 1] = v[1];   // sum_i r_i avg_i
    }
}

// gradient from the column-pass output (already sitting in the Gr plane), plus grad.d and ||grad||^2
__global__ void __launch_bounds__(kVecThreads) kb_grad(const BatchBufs b, const KVec p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[2 * 32];
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const double M = sc[SC_GMAX], inv = 1.0 / sc[SC_S], gbar = sc[SC_GBAR], Gbar = sc[SC_CAPGBAR];
    const double ravg = sc[SC_TMP0 + 1], theta = p.theta[k];
    const double* x = b.X + (size_t)k * b.ldn;
    const double* d = b.D + (size_t)k * b.ldn;
    double* gr = b.Gr + (size_t)k * b.ldn;
    double v[2] = {0.0, 0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < b.n; j += gridDim.x * blockDim.x) {
        const double gj = x[j];
        const double w = exp(gj - M) * inv;
        const double gv = w * theta * (gj - gbar - b.G[j] + Gbar) + w * (gr[j] - ravg);
        gr[j] = gv;
        v[0] = fma(gv, d[j], v[0]);
        v[1] = fma(gv, gv, v[1]);
    }
    grid_sum<2>(v, b.partials + (size_t)k * b.pstride, b.ticket + k, red, [=](const double(&t)[2]) {
        sc[SC_DG] = t[0];
        sc[SC_GNORM2] = t[1];
    });
}

// dst_k = alpha * src_k for masked planes (d = -g, copies)
__global__ void __launch_bounds__(kVecThreads)
    kb_scale_copy(int n, long long ldn, const double* src, double* dst, double alpha, const KVec p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    const double* s = src + (size_t)k * ldn;
    double* d = dst + (size_t)k * ldn;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) d[j] = alpha * s[j];
}

struct KSlots {
    int slot[kBMaxK];
    int mask[kBMaxK];
};

__global__ void __launch_bounds__(kVecThreads) kb_pair(const BatchBufs b, const KSlots p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[2 * 32];
    const size_t plane = (size_t)k * b.ldn;
    const size_t hist = ((size_t)p.slot[k] * b.KP + k) * b.ldn;
    const double *x = b.X + plane, *g = b.Gr + plane;
    double *xp = b.XP + plane, *gp = b.GP + plane, *s = b.S + hist, *y = b.Yv + hist;
    double v[2] = {0.0, 0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < b.n; j += gridDim.x * blockDim.x) {
        const double xj = x[j], gj = g[j];
        const double sj = xj - xp[j], yj = gj - gp[j];
        s[j] = sj; y[j] = yj; xp[j] = xj; gp[j] = gj;
        v[0] = fma(yj, sj, v[0]);
        v[1] = fma(yj, yj, v[1]);
    }
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const int slot = p.slot[k];
    grid_sum<2>(v, b.partials + (size_t)k * b.pstride, b.ticket + k, red, [=](const double(&t)[2]) {
        sc[SC_YS] = t[0];
        sc[SC_YY] = t[1];
        sc[SC_YS0 + slot] = t[0];
    });
}

// one fused step of the two-loop recursion per problem (see k_lbfgs_twoloop); op 0 = nothing to do for this k
struct KStep {
    signed char op[kBMaxK];        // 0 none, 1 active
    signed char init[kBMaxK];      // d = -g first
    signed char u_kind[kBMaxK];    // TL_NONE, TL_S, TL_Y (lbfgs.cuh)
    signed char u_slot[kBMaxK];
    signed char c_num[kBMaxK], c_den[kBMaxK], c2_num[kBMaxK];   // sc indices (c2 < 0: unused); csign below
    signed char csign[kBMaxK];
    signed char scale[kBMaxK];     // 1: d *= ys/yy
    signed char v_kind[kBMaxK];    // TL_NONE, TL_S, TL_Y, TL_G
    signed char v_slot[kBMaxK];
    signed char out[kBMaxK];
};

__global__ void __launch_bounds__(kVecThreads) kb_twoloop(const BatchBufs b, const KStep p) {
    const int k = blockIdx.y;
    if (!p.op[k]) return;
    __shared__ double red[32];
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const size_t plane = (size_t)k * b.ldn;
    double* d = b.D + plane;
    const double* g = b.Gr + plane;
    auto hist = [&](int kind, int slot) -> const double* {
        if (kind == TL_G) return g;
        return (kind == TL_S ? b.S : b.Yv) + ((size_t)slot * b.KP + k) * b.ldn;
    };
    const double* u = p.u_kind[k] ? hist(p.u_kind[k], p.u_slot[k]) : nullptr;
    const double* vv = p.v_kind[k] ? hist(p.v_kind[k], p.v_slot[k]) : nullptr;
    double coef = 0.0, scale = 1.0;
    if (u) {
        coef = (double)p.csign[k] * (sc[p.c_num[k]] / sc[p.c_den[k]]);
        if (p.c2_num[k] >= 0) coef -= sc[p.c2_num[k]] / sc[p.c_den[k]];
    }
    if (p.scale[k]) scale = sc[SC_YS] / sc[SC_YY];
    const int init = p.init[k];
    double v[1] = {0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < b.n; j += gridDim.x * blockDim.x) {
        double dj = init ? -g[j] : d[j];
        if (u) dj = fma(coef, u[j], dj);
        if (p.scale[k]) dj *= scale;
        d[j] = dj;
        if (vv) v[0] = fma(vv[j], dj, v[0]);
    }
    if (vv) {
        const int out = p.out[k];
        grid_sum<1>(v, b.partials + (size_t)k * b.pstride, b.ticket + k, red,
                    [=](const double(&t)[1]) { sc[out] = t[0]; });
    }
}

// ------------------------------------------------------------------------------------------------
// forces method, batched (c_bioen_kernels_forces.c:43-76 for K problems at once).  The variables f_k are
// M-dimensional planes; one batched evaluation is four skinny GEMMs:
//   X = Yt.F  ->  softmax with prior weights  ->  avg = Y.W  ->  T = Yt.R  ->  E  ->  grad = Y.E - avg*sum(E)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kbf_prepare(const BatchBufs b, const KVec p, int move) {
    const int k = blockIdx.x;
    if (!p.mask[k]) return;
    __shared__ double red[32];
    double* x = b.X + (size_t)k * b.ldn;
    const double* xp = b.XP + (size_t)k * b.ldn;
    const double* d = b.D + (size_t)k * b.ldn;
    double v[1] = {0.0};
    for (int i = threadIdx.x; i < b.n; i += blockDim.x) {
        double xi = x[i];
        if (move) { xi = fma(p.stp[k], d[i], xp[i]); x[i] = xi; }
        b.Ff[frag_index(i, k, b.NT)] = xi;
        v[0] = fma(xi, xi, v[0]);
    }
    block_sum<1>(v, red);
    if (threadIdx.x == 0) b.scb[(size_t)k * SC_COUNT + SC_XNORM2] = v[0];
}

__global__ void __launch_bounds__(kVecThreads) kbf_lse(const BatchBufs b, const KVec p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[3 * 32];
    __shared__ bool is_last;
    const double* x = b.Xn + (size_t)k * b.ldN;
    const double* w0p = b.G + (size_t)k * b.gld;
    double m = -DBL_MAX, s = 0.0, dummy = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < b.nN; j += gridDim.x * blockDim.x) {
        const double v = x[j], pw = w0p[j];
        if (v > m) { s = s * exp(m - v) + pw; m = v; }
        else s += pw * exp(v - m);
    }
    double* partials = b.partials + (size_t)k * b.pstride;
    block_lse(m, s, dummy, red);
    if (threadIdx.x == 0) {
        partials[blockIdx.x * 2 + 0] = m;
        partials[blockIdx.x * 2 + 1] = s;
        __threadfence();
        is_last = (atomicAdd(b.ticket + k, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        m = -DBL_MAX; s = 0.0; dummy = 0.0;
        for (unsigned q = threadIdx.x; q < gridDim.x; q += blockDim.x)
            lse_merge(m, s, __ldcg(&partials[q * 2]), __ldcg(&partials[q * 2 + 1]));
        block_lse(m, s, dummy, red);
        if (threadIdx.x == 0) {
            double* sc = b.scb + (size_t)k * SC_COUNT;
            sc[SC_GMAX] = m;
            sc[SC_S] = s;
            b.ticket[k] = 0;
        }
    }
}

// weights (fragment-major), guarded log ratio, KL   (c_bioen_kernels_forces.c:156-171, 246-274)
__global__ void __launch_bounds__(kVecThreads) kbf_weights(const BatchBufs b, const KVec p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[32];
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const double M = sc[SC_GMAX], inv = 1.0 / sc[SC_S], logS = log(sc[SC_S]);
    const double* x = b.Xn + (size_t)k * b.ldN;
    double* lrp = b.LR + (size_t)k * b.ldN;
    const double* w0p = b.G + (size_t)k * b.gld;
    double v[1] = {0.0};
    const int nq = (b.nN + 3) >> 2;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
        double w4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = 4 * q + e;
            double w = 0.0;
            if (j < b.nN) {
                const double xj = x[j], w0 = w0p[j];
                w = inv * (w0 * exp(xj - M));
                const double lr = (w >= DBL_MIN && w0 >= DBL_MIN) ? (xj - M - logS) : 0.0;
                lrp[j] = lr;
                v[0] = fma(lr, w, v[0]);
            }
            w4[e] = w;
        }
        double* dst = b.Wf + ((size_t)q * b.NT + (k >> 3)) * 32 + (k & 7) * 4;
        *reinterpret_cast<double2*>(dst) = make_double2(w4[0], w4[1]);
        *reinterpret_cast<double2*>(dst + 2) = make_double2(w4[2], w4[3]);
    }
    grid_sum<1>(v, b.partials + (size_t)k * b.pstride, b.ticket + k, red, [=](const double(&t)[1]) { sc[SC_KL] = t[0]; });
}

// avg, r (fragment-major), chi^2, objective = theta KL + chi^2   (one block per problem)
__global__ void __launch_bounds__(1024) kbf_finalize(const BatchBufs b, const KVec p, int m, int nseg) {
    const int k = blockIdx.x;
    if (!p.mask[k]) return;
    __shared__ double red[32];
    const double* Y = b.Yobs + (size_t)k * b.yld;
    const double* c = b.Cw ? b.Cw + (size_t)k * b.ldo : nullptr;
    double v[1] = {0.0};
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < nseg; ++q) s += b.avgp[((size_t)q * b.KP + k) * b.ldo + i];
        b.avgk[(size_t)k * b.ldo + i] = s;
        const double r = s - Y[i];
        const double cr = c ? c[i] * r : r;
        b.Rf[frag_index(i, k, b.NT)] = cr;      // t_j = sum_i y_ij c_i r_i: kbf_E and kbf_grad need nothing else
        v[0] = fma(cr, r, v[0]);
    }
    block_sum<1>(v, red);
    if (threadIdx.x == 0) {
        double* sc = b.scb + (size_t)k * SC_COUNT;
        const double chi2 = 0.5 * v[0], prior = sc[SC_KL] * p.theta[k];
        sc[SC_CHI2] = chi2;
        sc[SC_PRIOR] = prior;
        sc[SC_F] = prior + chi2;
    }
}

// E_j = (theta (1 + lr_j) + t_j) w_j in fragment-major order, and sum_j E_j   (kernels_forces.c:321-328)
__global__ void __launch_bounds__(kVecThreads) kbf_E(const BatchBufs b, const KVec p) {
    const int k = blockIdx.y;
    if (!p.mask[k]) return;
    __shared__ double red[32];
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const double M = sc[SC_GMAX], inv = 1.0 / sc[SC_S], theta = p.theta[k];
    const double* x = b.Xn + (size_t)k * b.ldN;
    const double* lrp = b.LR + (size_t)k * b.ldN;
    const double* t = b.Tn + (size_t)k * b.ldN;
    const double* w0p = b.G + (size_t)k * b.gld;
    double v[1] = {0.0};
    const int nq = (b.nN + 3) >> 2;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
        double e4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int j = 4 * q + e;
            double E = 0.0;
            if (j < b.nN) {
                const double w = inv * (w0p[j] * exp(x[j] - M));
                E = ((1.0 + lrp[j]) * theta + t[j]) * w;
                v[0] += E;
            }
            e4[e] = E;
        }
        double* dst = b.Wf + ((size_t)q * b.NT + (k >> 3)) * 32 + (k & 7) * 4;
        *reinterpret_cast<double2*>(dst) = make_double2(e4[0], e4[1]);
        *reinterpret_cast<double2*>(dst + 2) = make_double2(e4[2], e4[3]);
    }
    grid_sum<1>(v, b.partials + (size_t)k * b.pstride, b.ticket + k, red,
                [=](const double(&t)[1]) { sc[SC_TMP0 + 1] = t[0]; });
}

// grad_i = sum_j y_ij E_j - avg_i sum_j E_j, plus grad.d and ||grad||^2   (one block per problem)
__global__ void __launch_bounds__(1024) kbf_grad(const BatchBufs b, const KVec p, int m, int nseg) {
    const int k = blockIdx.x;
    if (!p.mask[k]) return;
    __shared__ double red[2 * 32];
    double* sc = b.scb + (size_t)k * SC_COUNT;
    const double sumE = sc[SC_TMP0 + 1];
    double* gr = b.Gr + (size_t)k * b.ldn;
    const double* d = b.D + (size_t)k * b.ldn;
    double v[2] = {0.0, 0.0};
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < nseg; ++q) s += b.avgp[((size_t)q * b.KP + k) * b.ldo + i];
        const double gv = s - b.avgk[(size_t)k * b.ldo + i] * sumE;
        gr[i] = gv;
        v[0] = fma(gv, d[i], v[0]);
        v[1] = fma(gv, gv, v[1]);
    }
    block_sum<2>(v, red);
    if (threadIdx.x == 0) {
        sc[SC_DG] = v[0];
        sc[SC_GNORM2] = v[1];
    }
}

// ------------------------------------------------------------------------------------------------
// N-sharded scan (one process per GPU): per-problem scalars that are sums over the structure axis are packed
// into a contiguous buffer, all-reduced with ONE exchange (Comm: peer-memory kernel up to its inbox size, NCCL
// above), and unpacked; the (max, sum-exp) pairs are all-gathered and merged.  slot < 0: that problem contributes nothing (finished / masked).
// ------------------------------------------------------------------------------------------------
struct KSlotTab {
    int n;                          // rows used (<= 4)
    signed char row[4];             // unpack: which buffer row feeds entry r (pack: r itself)
    signed char slot[4][kBMaxK];
};

__global__ void kb_pack(const double* scb, double* buf, const KSlotTab t, int KP) {
    const int k = threadIdx.x, r = blockIdx.x;
    if (k >= KP || r >= t.n) return;
    const int sl = t.slot[r][k];
    buf[r * KP + k] = sl >= 0 ? scb[(size_t)k * SC_COUNT + sl] : 0.0;
}

__global__ void kb_unpack(double* scb, const double* buf, const KSlotTab t, int KP) {
    const int k = threadIdx.x, r = blockIdx.x;
    if (k >= KP || r >= t.n) return;
    const int sl = t.slot[r][k];
    if (sl >= 0) scb[(size_t)k * SC_COUNT + sl] = buf[t.row[r] * KP + k];
}

// merge the ranks' (max, sum-exp) pairs: lse_all[rank][2][KP] -> sc[k][SC_GMAX], sc[k][SC_S]
__global__ void kb_lse_merge(double* scb, const double* lse_all, int nranks, int KP, const KVec p) {
    const int k = threadIdx.x;
    if (k >= KP || !p.mask[k]) return;
    double m = lse_all[k], s = lse_all[KP + k];
    for (int r = 1; r < nranks; ++r) lse_merge(m, s, lse_all[(size_t)r * 2 * KP + k], lse_all[(size_t)r * 2 * KP + KP + k]);
    scb[(size_t)k * SC_COUNT + SC_GMAX] = m;
    scb[(size_t)k * SC_COUNT + SC_S] = s;
}

// out[k][i] = sum over the reduction segments of the row-GEMM partials (the buffer that is all-reduced)
__global__ void __launch_bounds__(256) kb_reduce_avg(const double* avgp, double* out, int m, int nseg, int KP, long long ldo) {
    const int k = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double s = 0.0;
    for (int q = 0; q < nseg; ++q) s += avgp[((size_t)q * KP + k) * ldo + i];
    out[(size_t)k * ldo + i] = s;
}

// Per-problem inputs of a batch: host arrays of K rows, nullptr = every problem reads the context's shared vector.
struct BatchPlanes {
    const double* YTilde = nullptr;        // [K][M]  observed data (noise replicates)
    const double* row_weights = nullptr;   // [K][M]  c_k,i >= 0 (observable resampling, held-out folds)
    const double* w0 = nullptr;            // [K][N]  reference weights >= 0 (structure resampling), forces only
};

// Host-side checks of a batch's planes (before anything is allocated or enqueued)
inline void check_planes(const BatchPlanes& in, int K, int M, int N, bool forces) {
    auto bad = [](const char* what, int k, long long i) {
        char buf[200];
        snprintf(buf, sizeof buf, "bioen_b200: %s (problem %d, entry %lld)", what, k, i);
        throw std::invalid_argument(buf);
    };
    if (in.w0 && !forces)
        throw std::invalid_argument("bioen_b200: per-problem reference weights w0 need the forces method (log-weights "
                                    "would need G_j = -inf for a structure of weight zero)");
    for (int k = 0; k < K; ++k) {
        if (in.YTilde)
            for (int i = 0; i < M; ++i)
                if (!std::isfinite(in.YTilde[(size_t)k * M + i])) bad("YTilde must be finite", k, i);
        if (in.row_weights)
            for (int i = 0; i < M; ++i) {
                const double c = in.row_weights[(size_t)k * M + i];
                if (!(std::isfinite(c) && c >= 0.0)) bad("row weights must be finite and >= 0", k, i);
            }
        if (in.w0) {
            double sum = 0.0;
            for (long long j = 0; j < N; ++j) {
                const double w = in.w0[(size_t)k * N + j];
                if (!(std::isfinite(w) && w >= 0.0)) bad("w0 must be finite and >= 0", k, j);
                sum += w;
            }
            if (!(sum > 0.0)) bad("w0 must have a positive sum", k, -1);
        }
    }
}

struct ScanResult {
    int code = 0, iterations = 0, evaluations = 0;
    double fmin = 0.0;
};

class ThetaScan {
   public:
    Context& C;
    const bool forces;          // false: log-weights (variables = N planes), true: forces (variables = M planes)
    const int K, KP, NT, n;     // n = dimension of the variables
    const int NN, MM;           // structures, observables
    LbfgsParams prm;
    int verbose = 0;
    long long ldn, ldN;
    DevBuf<double> planes, hist, Wf, Rf, avgp, scb, partials, nplanes, Ff, avgk, redbuf, lsebuf, lse_all;
    DevBuf<double> yplanes, cplanes, wplanes;   // per-problem YTilde, row weights, w0 (allocated when given)
    bool started = false;       // run() got past the parameter check: the X planes hold the problems' points
    int vblocksN = 1;
    bool reduce = false;        // N sharded over ranks
    DevBuf<unsigned int> ticket;
    double* h_scb = nullptr;
    BatchBufs B{};
    CUtensorMap tmapRow, tmapCol;
    GemmArgs gRow{}, gCol{};
    int vblocks;
    long long rounds = 0, gemm_launches = 0;

    ThetaScan(Context& ctx, int k, const LbfgsParams& p, bool is_forces = false, const BatchPlanes& in = {})
        : C(ctx), forces(is_forces), K(k), KP((k + 7) & ~7), NT(((k + 7) & ~7) / 8),
          n(is_forces ? ctx.M : ctx.N), NN(ctx.N), MM(ctx.M), prm(p) {
        if (k < 1 || k > kBMaxK) throw std::invalid_argument("bioen_b200: theta scan batches 1..32 problems");
        if (!forces && !C.have_logw) throw std::logic_error("bioen_b200: log-weights data not set");
        if (forces && !C.have_forces) throw std::logic_error("bioen_b200: forces data not set");
        check_planes(in, K, MM, NN, forces);
        if (!C.yt_valid) C.make_transposed();
        ldn = ((long long)n + 63) & ~63LL;
        ldN = ((long long)NN + 63) & ~63LL;
        const int m = prm.m;
        planes.alloc((size_t)5 * KP * ldn);
        hist.alloc((size_t)2 * m * KP * ldn);
        const long long nq = ((long long)NN + 15) / 16 * 16;          // indices padded to whole GEMM tiles
        const long long mq = ((long long)MM + 15) / 16 * 16;
        Wf.alloc((size_t)nq * KP);
        Rf.alloc((size_t)mq * KP);
        scb.alloc((size_t)KP * SC_COUNT);
        vblocks = std::max(1, std::min((n + kVecThreads - 1) / kVecThreads, C.num_sms * 2));
        vblocksN = std::max(1, std::min((NN + kVecThreads - 1) / kVecThreads, C.num_sms * 2));
        const long long pstride = (long long)std::max(vblocks, vblocksN) * 4 + 16;
        partials.alloc((size_t)KP * pstride);
        ticket.alloc(KP);
        CUDA_CHECK(cudaHostAlloc(&h_scb, (size_t)KP * SC_COUNT * sizeof(double), cudaHostAllocDefault));
        // GEMM geometry
        gRow.rows = MM; gRow.kdim = NN; gRow.RB = (MM + kGRows - 1) / kGRows; gRow.ktiles = (NN + kGKdim - 1) / kGKdim;
        gRow.S = std::max(1, std::min(gRow.ktiles, C.num_sms / gRow.RB));
        gRow.tps = (gRow.ktiles + gRow.S - 1) / gRow.S;
        gRow.S = (gRow.ktiles + gRow.tps - 1) / gRow.tps;
        gRow.KP = KP; gRow.ldo = ((long long)C.M + 3) & ~3LL; gRow.evict_first = C.evict_first;
        avgp.alloc((size_t)gRow.S * KP * gRow.ldo);
        gRow.B = Wf.p; gRow.out = avgp.p;
        gCol.rows = NN; gCol.kdim = MM; gCol.RB = (NN + kGRows - 1) / kGRows; gCol.ktiles = (MM + kGKdim - 1) / kGKdim;
        gCol.S = 1; gCol.tps = gCol.ktiles; gCol.KP = KP; gCol.ldo = ldN; gCol.evict_first = C.evict_first;
        gCol.B = Rf.p;
        B.n = n; B.K = K; B.KP = KP; B.NT = NT; B.ldn = ldn;
        B.X = planes.p; B.Gr = B.X + (size_t)KP * ldn; B.XP = B.Gr + (size_t)KP * ldn;
        B.GP = B.XP + (size_t)KP * ldn; B.D = B.GP + (size_t)KP * ldn;
        B.S = hist.p; B.Yv = hist.p + (size_t)m * KP * ldn;
        B.Wf = Wf.p; B.Rf = Rf.p; B.avgp = avgp.p; B.scb = scb.p; B.partials = partials.p; B.ticket = ticket.p;
        B.pstride = pstride; B.G = C.Gv.p; B.Yobs = C.Yobs.p;
        gCol.out = B.Gr;          // logw: the column pass writes straight into the gradient planes (ldn == ldN)
        if (forces) {
            nplanes.alloc((size_t)3 * KP * ldN);
            Ff.alloc((size_t)mq * KP);
            B.nN = NN; B.ldN = ldN; B.Xn = nplanes.p; B.LR = B.Xn + (size_t)KP * ldN; B.Tn = B.LR + (size_t)KP * ldN;
            B.Ff = Ff.p;
        }
        avgk.alloc((size_t)KP * gRow.ldo);
        B.avgk = avgk.p;
        B.ldo = gRow.ldo;
        // per-problem planes; the padding problems k >= K are masked and keep zeros
        auto upload_planes = [&](DevBuf<double>& buf, const double* src, int len, long long ld) {
            buf.alloc((size_t)KP * ld);
            for (int q = 0; q < K; ++q) C.h2d(buf.p + (size_t)q * ld, src + (size_t)q * len, len);
            return buf.p;
        };
        if (in.YTilde) { B.Yobs = upload_planes(yplanes, in.YTilde, MM, B.ldo); B.yld = B.ldo; }
        if (in.row_weights) B.Cw = upload_planes(cplanes, in.row_weights, MM, B.ldo);
        if (in.w0) { B.G = upload_planes(wplanes, in.w0, NN, ldN); B.gld = ldN; }
        reduce = C.nranks > 1;
        if (reduce) {
            redbuf.alloc((size_t)KP * gRow.ldo + 4 * KP);
            lsebuf.alloc((size_t)2 * KP);
            lse_all.alloc((size_t)C.nranks * 2 * KP);
        }
        make_map(&tmapRow, C.Y, (cuuint64_t)NN, (cuuint64_t)MM, (cuuint64_t)C.ld);
        make_map(&tmapCol, C.Yt.p, (cuuint64_t)MM, (cuuint64_t)NN, (cuuint64_t)C.ldt);
        set_attr();
        // log s0 is a property of G: copy it into every problem's scalar row
        std::vector<double> row((size_t)KP * SC_COUNT, 0.0);
        double logs0 = 0.0;
        if (!forces) C.d2h(&logs0, C.sc.p + SC_LOGS0, 1);
        C.sync();
        for (int q = 0; q < KP; ++q) row[(size_t)q * SC_COUNT + SC_LOGS0] = logs0;
        C.h2d(scb.p, row.data(), row.size());
    }
    ~ThetaScan() {
        if (h_scb) cudaFreeHost(h_scb);
    }

    static constexpr int smem_bytes() { return kGStages * (kGTileBytes + 4096) + 2 * kGStages * 8 + 1024 + 64; }
    void make_map(CUtensorMap* map, double* base, cuuint64_t inner, cuuint64_t outer, cuuint64_t ld) {
        const cuuint64_t gdim[2] = {inner, outer};
        const cuuint64_t gstride[1] = {ld * sizeof(double)};
        const cuuint32_t box[2] = {(cuuint32_t)kGKdim, (cuuint32_t)kGRows};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = get_encode_tiled()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, gdim, gstride, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) throw CudaError("bioen_b200: cuTensorMapEncodeTiled (swizzled) failed");
    }
    void set_attr() {
        CUDA_CHECK(cudaFuncSetAttribute(batched_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes()));
        CUDA_CHECK(cudaFuncSetAttribute(batched_gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes()));
        CUDA_CHECK(cudaFuncSetAttribute(batched_gemm_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes()));
        CUDA_CHECK(cudaFuncSetAttribute(batched_gemm_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes()));
    }
    void launch_gemm(const CUtensorMap& map, const GemmArgs& g) {
        const int items = g.RB * g.S;
        const int grid = std::min(items, C.num_sms);
        const bool timed = C.pass_timing && C.pass_ev_used + 2 <= C.pass_ev.size();
        if (timed) CUDA_CHECK(cudaEventRecord(C.pass_ev[C.pass_ev_used++], C.stream));
        switch (NT) {
            case 1: batched_gemm_kernel<1><<<grid, kGThreads, smem_bytes(), C.stream>>>(map, g); break;
            case 2: batched_gemm_kernel<2><<<grid, kGThreads, smem_bytes(), C.stream>>>(map, g); break;
            case 3: batched_gemm_kernel<3><<<grid, kGThreads, smem_bytes(), C.stream>>>(map, g); break;
            default: batched_gemm_kernel<4><<<grid, kGThreads, smem_bytes(), C.stream>>>(map, g); break;
        }
        if (timed) CUDA_CHECK(cudaEventRecord(C.pass_ev[C.pass_ev_used++], C.stream));
        CUDA_CHECK(cudaGetLastError());
        ++gemm_launches;
        ++C.passes_launched;
        ++C.kernels_launched;
    }

    // ---- collectives of the sharded scan (no-ops on one GPU) -----------------------------------------------
    static KSlotTab tab_uniform(std::initializer_list<int> slots, const KVec& kv) {
        KSlotTab t{};
        t.n = (int)slots.size();
        int r = 0;
        for (int sl : slots) {
            t.row[r] = (signed char)r;
            for (int q = 0; q < kBMaxK; ++q) t.slot[r][q] = kv.mask[q] ? (signed char)sl : (signed char)-1;
            ++r;
        }
        return t;
    }
    void allreduce_tab(const KSlotTab& t, double* buf) {
        kb_pack<<<t.n, kBMaxK, 0, C.stream>>>(scb.p, buf, t, KP);
        C.comm->allreduce_sum(buf, (size_t)t.n * KP, C.stream);
        kb_unpack<<<t.n, kBMaxK, 0, C.stream>>>(scb.p, buf, t, KP);
    }
    void merge_lse(const KVec& kv) {
        if (!reduce) return;
        const KSlotTab t = tab_uniform({SC_GMAX, SC_S}, kv);
        kb_pack<<<2, kBMaxK, 0, C.stream>>>(scb.p, lsebuf.p, t, KP);
        C.comm->allgather(lsebuf.p, lse_all.p, (size_t)2 * KP, C.stream);
        kb_lse_merge<<<1, kBMaxK, 0, C.stream>>>(scb.p, lse_all.p, C.nranks, KP, kv);
    }
    // segments of the row GEMM -> one [KP][ldo] array, all-reduced together with `tail` per-problem scalars;
    // returns the BatchBufs view the finalising kernel should read (nseg = 1)
    BatchBufs reduce_rows(const KVec& kv, std::initializer_list<int> tail, int& nseg) {
        BatchBufs v = B;
        nseg = gRow.S;
        if (!reduce) return v;
        const dim3 g((MM + 255) / 256, KP);
        kb_reduce_avg<<<g, 256, 0, C.stream>>>(avgp.p, redbuf.p, MM, gRow.S, KP, gRow.ldo);
        const KSlotTab t = tab_uniform(tail, kv);
        double* tailbuf = redbuf.p + (size_t)KP * gRow.ldo;
        kb_pack<<<t.n, kBMaxK, 0, C.stream>>>(scb.p, tailbuf, t, KP);
        C.comm->allreduce_sum(redbuf.p, (size_t)KP * gRow.ldo + (size_t)t.n * KP, C.stream);
        kb_unpack<<<t.n, kBMaxK, 0, C.stream>>>(scb.p, tailbuf, t, KP);
        v.avgp = redbuf.p;
        nseg = 1;
        return v;
    }

    // one batched f+g evaluation of the masked problems; move: x = xp + stp*d first; grad = false: objective half only
    void evaluate(const KVec& kv, bool move, bool grad = true) {
        int nseg = 0;
        if (forces) {
            const dim3 gridN(vblocksN, KP);
            GemmArgs g = gCol;
            kbf_prepare<<<KP, 256, 0, C.stream>>>(B, kv, move ? 1 : 0);
            g.B = Ff.p; g.out = B.Xn;
            launch_gemm(tmapCol, g);                                   // x_j = sum_i f_i y_ij
            kbf_lse<<<gridN, kVecThreads, 0, C.stream>>>(B, kv);
            merge_lse(kv);
            kbf_weights<<<gridN, kVecThreads, 0, C.stream>>>(B, kv);
            launch_gemm(tmapRow, gRow);                                // avg_i
            {
                const BatchBufs v = reduce_rows(kv, {SC_KL}, nseg);
                kbf_finalize<<<KP, 1024, 0, C.stream>>>(v, kv, MM, nseg);
            }
            if (!grad) {
                CUDA_CHECK(cudaGetLastError());
                C.kernels_launched += 4;
                return;
            }
            g.B = Rf.p; g.out = B.Tn;
            launch_gemm(tmapCol, g);                                   // t_j = sum_i r_i y_ij
            kbf_E<<<gridN, kVecThreads, 0, C.stream>>>(B, kv);
            launch_gemm(tmapRow, gRow);                                // sum_j y_ij E_j
            {
                const BatchBufs v = reduce_rows(kv, {SC_TMP0 + 1}, nseg);
                kbf_grad<<<KP, 1024, 0, C.stream>>>(v, kv, MM, nseg);
            }
            CUDA_CHECK(cudaGetLastError());
            C.kernels_launched += 6;
            return;
        }
        const dim3 gridv(vblocks, KP);
        kb_update_lse<<<gridv, kVecThreads, 0, C.stream>>>(B, kv, move ? 1 : 0);
        merge_lse(kv);
        kb_weights<<<gridv, kVecThreads, 0, C.stream>>>(B, kv);
        launch_gemm(tmapRow, gRow);
        {
            const BatchBufs v = reduce_rows(kv, {SC_TMP0, SC_GBAR, SC_CAPGBAR, SC_XNORM2}, nseg);
            kb_finalize<<<KP, 1024, 0, C.stream>>>(v, kv, C.M, nseg, gRow.ldo);
        }
        if (!grad) {
            CUDA_CHECK(cudaGetLastError());
            C.kernels_launched += 3;
            return;
        }
        launch_gemm(tmapCol, gCol);
        kb_grad<<<gridv, kVecThreads, 0, C.stream>>>(B, kv);
        if (reduce) allreduce_tab(tab_uniform({SC_DG, SC_GNORM2}, kv), redbuf.p);
        CUDA_CHECK(cudaGetLastError());
        C.kernels_launched += 4;
    }
    void fetch() {
        C.d2h(h_scb, scb.p, (size_t)KP * SC_COUNT);
        C.spin_sync();
    }
    const double* hs(int k) const { return h_scb + (size_t)k * SC_COUNT; }

    // One evaluation of all K problems at the points in the X planes (x_host: [K][n] uploaded first when given),
    // copied out per problem: f[K], grad[K][n] (its presence selects the gradient half), avg[K][M] = yTilde . w,
    // chi2[K] (weighted by the row weights), kl[K] (the prior without the theta factor).  Any output may be nullptr.
    void evaluate_all(const double* thetas, const double* x_host, double* f, double* grad, double* avg, double* chi2,
                      double* kl) {
        if (x_host)
            for (int q = 0; q < K; ++q) C.h2d(B.X + (size_t)q * ldn, x_host + (size_t)q * n, n);
        KVec kv{};
        for (int q = 0; q < KP; ++q) { kv.mask[q] = q < K; kv.theta[q] = q < K ? thetas[q] : 0.0; }
        evaluate(kv, false, grad != nullptr);
        fetch();
        for (int q = 0; q < K; ++q) {
            if (f) f[q] = hs(q)[SC_F];
            if (chi2) chi2[q] = hs(q)[SC_CHI2];
            if (kl) kl[q] = hs(q)[SC_KL];
            if (grad) C.d2h(grad + (size_t)q * n, B.Gr + (size_t)q * ldn, n);
            if (avg) C.d2h(avg + (size_t)q * MM, avgk.p + (size_t)q * B.ldo, MM);
        }
        C.sync();
    }

    // bench.py: time `steps` batched evaluations of all K problems at fresh points (x = xp + (k+1)*d with a tiny d)
    void time_evals(const double* thetas, const double* x0_host, int warmup, int steps, float* ms, float* gemm_ms,
                    long long* launches) {
        KVec kv{};
        for (int q = 0; q < KP; ++q) { kv.mask[q] = q < K; kv.theta[q] = q < K ? thetas[q] : 0.0; kv.stp[q] = 0.0; }
        for (int q = 0; q < K; ++q) C.h2d(B.X + (size_t)q * ldn, x0_host + (size_t)q * n, n);
        const dim3 gridv(vblocks, KP);
        evaluate(kv, false);
        kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.X, B.XP, 1.0, kv);
        kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.Gr, B.D, -1e-9, kv);
        auto one = [&](int i) {
            for (int q = 0; q < K; ++q) kv.stp[q] = (double)(i + 1);
            evaluate(kv, true);
        };
        for (int i = 0; i < warmup; ++i) one(i);
        C.sync();
        cudaEvent_t e0, e1;
        CUDA_CHECK(cudaEventCreate(&e0));
        CUDA_CHECK(cudaEventCreate(&e1));
        C.begin_pass_timing(steps * 2);
        const long long k0 = C.kernels_launched;
        CUDA_CHECK(cudaEventRecord(e0, C.stream));
        for (int i = 0; i < steps; ++i) one(warmup + i);
        CUDA_CHECK(cudaEventRecord(e1, C.stream));
        CUDA_CHECK(cudaEventSynchronize(e1));
        float total = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&total, e0, e1));
        *ms = total;
        *launches = C.kernels_launched - k0;
        *gemm_ms = C.end_pass_timing();
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    }

    // The L-BFGS update of the problems in upd.mask (lbfgs.c:543-598): problem q's new pair goes to ring slot
    // upd.slot[q], then the two-loop recursion over bound[q] pairs as 2*bound+1 fused steps.  The problems of one
    // launch may sit at different (slot, bound); the others' planes are not touched.  run() and
    // bioen_b200_selftest_lbfgs_update call this.
    void update_directions(const KSlots& upd, const std::vector<int>& bound) {
        const int m = prm.m;
        const dim3 gridv(vblocks, KP);
        int maxbound = 0;
        for (int q = 0; q < K; ++q)
            if (upd.mask[q]) maxbound = std::max(maxbound, bound[q]);
        kb_pair<<<gridv, kVecThreads, 0, C.stream>>>(B, upd);
        if (reduce && !forces) {
            // y.s and y.y are sums over the structure axis; the ring copy ys[slot] follows the reduced value
            KSlotTab t{};
            t.n = 3;
            t.row[0] = 0; t.row[1] = 1; t.row[2] = 0;
            for (int q = 0; q < kBMaxK; ++q) {
                const bool on = q < K && upd.mask[q];
                t.slot[0][q] = on ? (signed char)SC_YS : (signed char)-1;
                t.slot[1][q] = on ? (signed char)SC_YY : (signed char)-1;
                t.slot[2][q] = on ? (signed char)(SC_YS0 + upd.slot[q]) : (signed char)-1;
            }
            KSlotTab pk = t;
            pk.n = 2;
            kb_pack<<<2, kBMaxK, 0, C.stream>>>(scb.p, redbuf.p, pk, KP);
            C.comm->allreduce_sum(redbuf.p, (size_t)2 * KP, C.stream);
            kb_unpack<<<3, kBMaxK, 0, C.stream>>>(scb.p, redbuf.p, t, KP);
        }
        // two-loop recursion (lbfgs.c:572-598) as 2*bound+1 fused steps per problem
        for (int t = 0; t <= 2 * maxbound; ++t) {
            KStep st{};
            for (int q = 0; q < K; ++q) {
                if (!upd.mask[q] || t > 2 * bound[q]) continue;
                const TwoLoopStep s = two_loop_step(t, (upd.slot[q] + 1) % m, bound[q], m);
                st.op[q] = 1;
                st.init[q] = (signed char)s.init;
                st.u_kind[q] = (signed char)s.u_kind; st.u_slot[q] = (signed char)s.u_slot;
                st.c_num[q] = (signed char)s.c_num; st.c_den[q] = (signed char)s.c_den; st.c2_num[q] = (signed char)s.c2_num;
                st.csign[q] = (signed char)s.csign;
                st.scale[q] = (signed char)s.scale;
                st.v_kind[q] = (signed char)s.v_kind; st.v_slot[q] = (signed char)s.v_slot;
                st.out[q] = (signed char)s.out;
            }
            kb_twoloop<<<gridv, kVecThreads, 0, C.stream>>>(B, st);
            if (reduce && !forces) {
                KSlotTab t{};
                t.n = 1;
                t.row[0] = 0;
                for (int q = 0; q < kBMaxK; ++q)
                    t.slot[0][q] = (q < K && st.op[q] && st.v_kind[q]) ? st.out[q] : (signed char)-1;
                allreduce_tab(t, redbuf.p);
            }
        }
        CUDA_CHECK(cudaGetLastError());
    }

    // x0 / x_out: [K][n] host arrays.  Returns per-problem results (liblbfgs codes).
    std::vector<ScanResult> run(const double* thetas, const double* x0_host, double* x_host) {
        std::vector<ScanResult> res(K);
        const int perr = lbfgs_check_params(n, prm);
        if (perr) {
            for (auto& r : res) r.code = perr;
            return res;
        }
        started = true;
        std::vector<LbfgsIteration> ps(K);
        std::vector<char> active(K, 0);
        KVec kv{};
        for (int q = 0; q < KP; ++q) { kv.mask[q] = q < K; kv.theta[q] = q < K ? thetas[q] : 0.0; kv.stp[q] = 0.0; }
        for (int q = 0; q < K; ++q)
            C.h2d(B.X + (size_t)q * ldn, x0_host + (size_t)q * n, n);
        const dim3 gridv(vblocks, KP);

        // ---- initial evaluation (lbfgs.c:412-459)
        evaluate(kv, false);
        fetch();
        for (int q = 0; q < K; ++q) {
            ++res[q].evaluations;
            res[q].code = ps[q].first_point(prm, hs(q));
            active[q] = res[q].code == 0;
            kv.mask[q] = active[q];
        }
        kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.Gr, B.D, -1.0, kv);
        kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.X, B.XP, 1.0, kv);
        kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.Gr, B.GP, 1.0, kv);

        auto any_active = [&] { for (char a : active) if (a) return true; return false; };
        while (any_active()) {
            ++rounds;
            for (int q = 0; q < K; ++q) {
                kv.mask[q] = active[q];
                if (active[q]) kv.stp[q] = ps[q].ls.prepare();
            }
            evaluate(kv, true);
            fetch();
            KSlots upd{};
            KVec revert{};
            bool any_upd = false, any_rev = false;
            std::vector<int> bound(K, 0);
            for (int q = 0; q < K; ++q) {
                if (!active[q]) continue;
                LbfgsIteration& p = ps[q];
                const double* h = hs(q);
                ++res[q].evaluations;
                int verdict;
                if (!p.slope_known) {   // the first trial of a search brings the slope of its direction
                    p.slope_known = true;
                    p.ls.set_slope(h[SC_DGINIT]);
                    if (0 < h[SC_DGINIT]) verdict = LBFGSERR_INCREASEGRADIENT;
                    else verdict = p.ls.update(h[SC_F], h[SC_DG]);
                } else {
                    verdict = p.ls.update(h[SC_F], h[SC_DG]);
                }
                if (verdict == 0) continue;   // next trial of the same search
                int slot = 0;
                const bool more = p.search_finished(verdict, h, slot, bound[q], res[q].code);
                res[q].iterations = p.iterations;
                if (more) {
                    upd.mask[q] = 1;
                    upd.slot[q] = slot;
                    any_upd = true;
                    continue;
                }
                active[q] = 0;
                if (verdict < 0) {
                    revert.mask[q] = 1;
                    any_rev = true;
                }
            }
            if (any_rev) {
                kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.XP, B.X, 1.0, revert);
                kb_scale_copy<<<gridv, kVecThreads, 0, C.stream>>>(n, ldn, B.GP, B.Gr, 1.0, revert);
            }
            if (any_upd) update_directions(upd, bound);
            if (verbose && rounds % 100 == 0) printf("\t\ttheta scan round %lld\n", rounds);
        }
        for (int q = 0; q < K; ++q) {
            res[q].fmin = ps[q].fx;
            C.d2h(x_host + (size_t)q * n, B.X + (size_t)q * ldn, n);
        }
        C.sync();
        return res;
    }
};

}  // namespace bioen
