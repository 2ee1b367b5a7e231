// vector_kernels.cuh -- the O(N) and O(M) kernels around the two matrix passes, and the fused vector
// kernels of the device-resident L-BFGS.  All reductions are fixed-order (block tree + last-block sum).
//
// Device scalar file: every evaluation/minimiser scalar lives in one small device array `sc[]`
// (indices below), so kernels chain through device memory and the host reads a handful of doubles once per
// line-search trial.
#pragma once
#include <float.h>

#include "comm.cuh"
#include "common.cuh"
#include "stream_pass.cuh"

namespace bioen {

enum ScalarSlot {
    SC_LSE_MAX = 0,   // local max of x            (k_update_lse)
    SC_LSE_SUM = 1,   // local sum exp(x - max)
    SC_KL = 2,        // forces: sum_j w_j (log w_j - log w0_j)
    SC_GMAX = 3,      // global max
    SC_S = 4,         // global sum exp(x - gmax)
    SC_LOGS0 = 5,     // log sum exp(G)            (constant of the problem)
    SC_GBAR = 6,      // <g> = sum g_j w_j
    SC_CAPGBAR = 7,   // <G> = sum G_j w_j
    SC_F = 8,         // objective
    SC_CHI2 = 9,      // 1/2 sum r^2
    SC_PRIOR = 10,    // theta * (...)  (logw)  or  theta * KL (forces)
    SC_DG = 11,       // grad . d      } local parts until all-reduced (3 contiguous doubles)
    SC_GNORM2 = 12,   // ||grad||^2    }
    SC_XNORM2 = 13,   // ||x||^2       }
    SC_WSCALE = 14,   // sharded log-weights: w_j = e_j * sc[SC_WSCALE], e_j = exp(g_j - rank-local max)
    SC_GINF = 15,     // max |grad_j|  (GSL stop test)
    // L-BFGS scalars
    SC_YS = 16,       // y.s of the newest pair
    SC_YY = 17,       // y.y of the newest pair
    SC_BETA = 18,     // raw y_j . d of the running second loop
    SC_DGINIT = 19,   // g . d for the new direction
    SC_DNORM2 = 20,   // ||d||^2 (initial step)
    SC_BETA2 = 21,    // second-loop dots alternate between SC_BETA and SC_BETA2
    // 22, 23 unused
    SC_YS0 = 24,      // ys[m] ring, up to 16 entries
    SC_ALPHA0 = 40,   // raw s_j . d ring, up to 16 entries
    SC_TMP0 = 56,     // generic outputs of vec_dot etc.
    SC_COUNT = 64
};

constexpr int kVecThreads = 256;

// the scalar file -> page-locked host memory (mapped), then a sequence number the host spins on (Context::fetch_scalars)
__global__ void __launch_bounds__(64) k_publish_scalars(const double* __restrict__ sc, double* host_copy, int count,
                                                        double* host_flag, double seq) {
    const int i = threadIdx.x;
    if (i < count) host_copy[i] = sc[i];
    __threadfence_system();
    __syncthreads();
    if (i == 0) {
        __threadfence_system();
        *reinterpret_cast<volatile double*>(host_flag) = seq;
    }
}

// merge two (max, sum-of-exp) pairs
__device__ __forceinline__ void lse_merge(double& m, double& s, double m2, double s2) {
    const double mm = fmax(m, m2);
    s = s * exp(m - mm) + s2 * exp(m2 - mm);
    m = mm;
}

// fixed-order block reduction of (max, sum-of-exp) pairs and one plain sum; result in thread 0
__device__ __forceinline__ void block_lse(double& m, double& s, double& xn, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
        lse_merge(m, s, m2, s2);
    }
    xn = warp_sum(xn);
    __syncthreads();
    if (lane == 0) { red[wid] = m; red[32 + wid] = s; red[64 + wid] = xn; }
    __syncthreads();
    if (wid == 0) {
        m = lane < nw ? red[lane] : -DBL_MAX;
        s = lane < nw ? red[32 + lane] : 0.0;
        xn = lane < nw ? red[64 + lane] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
            lse_merge(m, s, m2, s2);
        }
        xn = warp_sum(xn);
    }
}

// ------------------------------------------------------------------------------------------------
// K1: optional x = xp + stp*d, then local (max, sum exp(x-max)) and ||x||^2.
//     logw: the N-length softmax / log-sum-exp of the north star; forces: used on x_j = (yTilde^T f)_j with
//     the prior weights folded in (w0 != nullptr -> terms w0_j exp(x_j - max)).
//     reference: c_bioen_kernels_logw.c:55-94 (un-stabilised there), c_bioen_kernels_forces.c:151-171
// ------------------------------------------------------------------------------------------------
struct LseArgs {
    int n;
    double* x;           // in/out
    const double* xp;    // nullptr: x is used as is
    const double* d;
    double stp;
    const double* w0;    // nullptr for logw
    // forces: x_j is first assembled from the column-pass partial sums
    const double* col_partial;  // nullptr: x already holds the values
    long long col_ld;
    long long col_L, col_chunk;
    int write_xnorm;     // 1: sc[SC_XNORM2] = ||x||^2 (logw: x are the variables; forces: x_j is derived, keep ||f||^2)
    double* partials;    // gridDim.x * 3
    unsigned int* ticket;
    double* sc;
};

__global__ void __launch_bounds__(kVecThreads) k_update_lse(const LseArgs a) {
    __shared__ double red[3 * 32];
    __shared__ bool is_last;
    double m = -DBL_MAX, s = 0.0, xn = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        double x;
        if (a.col_partial) {
            const long long cb = j / kTileC;
            const int ns = pass_num_slots(cb, a.col_L, a.col_chunk);
            x = 0.0;
            for (int q = 0; q < ns; ++q) x += a.col_partial[(size_t)q * a.col_ld + j];
            a.x[j] = x;
        } else if (a.xp) {
            x = fma(a.stp, a.d[j], a.xp[j]);
            a.x[j] = x;
        } else {
            x = a.x[j];
        }
        xn = fma(x, x, xn);
        const double pw = a.w0 ? a.w0[j] : 1.0;
        if (x > m) {
            s = s * exp(m - x) + pw;
            m = x;
        } else {
            s += pw * exp(x - m);
        }
    }
    block_lse(m, s, xn, red);
    if (threadIdx.x == 0) {
        a.partials[blockIdx.x * 3 + 0] = m;
        a.partials[blockIdx.x * 3 + 1] = s;
        a.partials[blockIdx.x * 3 + 2] = xn;
        __threadfence();
        is_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        m = -DBL_MAX; s = 0.0; xn = 0.0;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
            lse_merge(m, s, __ldcg(&a.partials[b * 3]), __ldcg(&a.partials[b * 3 + 1]));
            xn += __ldcg(&a.partials[b * 3 + 2]);
        }
        block_lse(m, s, xn, red);
        if (threadIdx.x == 0) {
            a.sc[SC_LSE_MAX] = m;
            a.sc[SC_LSE_SUM] = s;
            if (a.write_xnorm) a.sc[SC_XNORM2] = xn;
            *a.ticket = 0;
        }
    }
}

// merge the per-rank (max, sum) pairs; every thread of every block of the next kernel calls this
__device__ __forceinline__ void global_lse(const double* pairs, int nranks, double& M, double& S) {
    M = pairs[0];
    S = pairs[1];
    for (int r = 1; r < nranks; ++r) lse_merge(M, S, pairs[2 * r], pairs[2 * r + 1]);
}

// ------------------------------------------------------------------------------------------------
// K2 (logw): w_j = exp(g_j - gmax) / S and the three weighted sums of the prior / gradient
//     reference: c_bioen_kernels_logw.c:96-127 (prior), 208-212 (<g>, <G>)
//     The sums are appended to the M-vector that is all-reduced after the row pass: msum[M..M+2].
// ------------------------------------------------------------------------------------------------
struct LogwWeightsArgs {
    int n;
    const double* g;
    const double* G;
    double* w;
    const double* lse_pairs;  // [nranks][2]
    int nranks;
    double* msum_tail;        // 3 doubles: sum (g-G) w, sum g w, sum G w  (local parts)
    double* partials;
    unsigned int* ticket;
    double* sc;
    // 1: sharded run whose normalisation travels WITH the row sums (one exchange per evaluation): w_j = e_j =
    //    exp(g_j - m_p) with the rank-local maximum m_p, sums of e_j-weighted terms, and tail[3..4] = (m_p, S_p)
    int local_only;
};

__global__ void __launch_bounds__(kVecThreads) k_logw_weights(const LogwWeightsArgs a) {
    __shared__ double red[3 * 32];
    double M, S;
    if (a.local_only) { M = a.sc[SC_LSE_MAX]; S = 1.0; }
    else global_lse(a.lse_pairs, a.nranks, M, S);
    const double inv = 1.0 / S;
    double v[3] = {0.0, 0.0, 0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const double g = a.g[j], G = a.G[j];
        const double w = exp(g - M) * inv;
        a.w[j] = w;
        v[0] = fma(g - G, w, v[0]);
        v[1] = fma(g, w, v[1]);
        v[2] = fma(G, w, v[2]);
    }
    double* tail = a.msum_tail;
    double* sc = a.sc;
    const int local_only = a.local_only;
    grid_sum<3>(v, a.partials, a.ticket, red, [=](const double(&t)[3]) {
        tail[0] = t[0];
        tail[1] = t[1];
        tail[2] = t[2];
        if (local_only) {
            tail[3] = M;
            tail[4] = sc[SC_LSE_SUM];
        } else {
            sc[SC_GMAX] = M;
            sc[SC_S] = S;
        }
    });
}

// ------------------------------------------------------------------------------------------------
// Sharded log-weights evaluation, the ONE exchange of the objective half, fused with what surrounds it (one block):
//   slot reduction of the local row pass  ->  this rank's M + 5 doubles {A_p,i = sum_j y_ij e_j; sum (g-G) e,
//   sum g e, sum G e; m_p; S_p} delivered to every rank's inbox  ->  combination in rank order with the factors
//   c_p = exp(m_p - m), m = max_p m_p, S = sum_p S_p c_p:  avg_i = sum_p A_p,i c_p / S (likewise the three prior sums)
//   ->  r_i, chi^2, prior, objective (what k_finalize_rows does on one GPU)  ->  sc[SC_WSCALE] = c_rank / S, the
//   factor that turns this rank's e_j into globally normalised weights in k_logw_grad.
// SURVEY 8e / north_star item 4: "one allreduce of the M-vector plus the log-sum-exp / entropy scalars".
// ------------------------------------------------------------------------------------------------
struct RowsExchangeArgs {
    int m;
    const double* partial;   // row-pass slots
    long long ld, L, chunk;
    double* msum;            // m + 5 doubles; [m..m+4] already hold the tail written by k_logw_weights(local_only)
    P2PDev p2p;
    const double* Y;
    double* ab;
    double* avg;
    double theta;
    double* sc;
};

constexpr int kRowsXThreads = 1024;

__global__ void __launch_bounds__(kRowsXThreads, 1) k_logw_rows_exchange_finalize(const RowsExchangeArgs a) {
    __shared__ double red[32];
    __shared__ double s_c[kP2PMaxRanks];
    __shared__ double s_inv;
    const int tid = threadIdx.x, R = a.p2p.nranks;
    for (int i = tid; i < a.m; i += kRowsXThreads) {
        const int ns = pass_num_slots(i / kTileR, a.L, a.chunk);
        double s = 0.0;
        for (int q = 0; q < ns; ++q) s += a.partial[(size_t)q * a.ld + i];
        a.msum[i] = s;
    }
    int fail;
    const double* in = p2p_deliver_and_wait(a.p2p, a.msum, a.m + 5, &fail);
    const long long cap = a.p2p.cap;
    if (tid == 0) {
        double mx = __ldcg(in + a.m + 3);
        for (int r = 1; r < R; ++r) mx = fmax(mx, __ldcg(in + r * cap + a.m + 3));
        double S = 0.0;
        for (int r = 0; r < R; ++r) {
            s_c[r] = exp(__ldcg(in + r * cap + a.m + 3) - mx);
            S += __ldcg(in + r * cap + a.m + 4) * s_c[r];
        }
        s_inv = 1.0 / S;
        a.sc[SC_GMAX] = mx;
        a.sc[SC_S] = S;
        a.sc[SC_WSCALE] = fail ? p2p_nan() : s_c[a.p2p.rank] * s_inv;
    }
    __syncthreads();
    const double inv = s_inv;
    double v[1] = {0.0};
    for (int i = tid; i < a.m; i += kRowsXThreads) {
        double s = 0.0;
        for (int r = 0; r < R; ++r) s = fma(__ldcg(in + r * cap + i), s_c[r], s);
        s *= inv;
        const double rr = s - a.Y[i];
        a.avg[i] = s;
        reinterpret_cast<double2*>(a.ab)[i] = make_double2(rr, s);
        v[0] = fma(rr, rr, v[0]);
    }
    block_sum<1>(v, red);
    if (tid == 0) {
        double t[3];
        for (int k = 0; k < 3; ++k) {
            double s = 0.0;
            for (int r = 0; r < R; ++r) s = fma(__ldcg(in + r * cap + a.m + k), s_c[r], s);
            t[k] = s * inv;
        }
        const double chi2 = 0.5 * v[0];
        const double val = t[0] - (a.sc[SC_GMAX] + log(a.sc[SC_S])) + a.sc[SC_LOGS0];
        const double prior = val * a.theta;
        a.sc[SC_GBAR] = t[1];
        a.sc[SC_CAPGBAR] = t[2];
        a.sc[SC_CHI2] = chi2;
        a.sc[SC_PRIOR] = prior;
        a.sc[SC_F] = fail ? p2p_nan() : prior + chi2;
    }
}

// ------------------------------------------------------------------------------------------------
// slot reduction of the row pass: msum_i = sum_slots partial[slot][i]   (only needed before an all-reduce)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kVecThreads)
    k_reduce_row_slots(int m, const double* partial, long long ld, long long L, long long chunk, double* msum) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int ns = pass_num_slots(i / kTileR, L, chunk);
    double s = 0.0;
    for (int q = 0; q < ns; ++q) s += partial[(size_t)q * ld + i];
    msum[i] = s;
}

// ------------------------------------------------------------------------------------------------
// K4: finish the row pass: avg_i, r_i = avg_i - Y_i, chi^2/2, and the objective.
//     logw:   f = theta (sum (g-G) w - log s + log s0) + chi2      c_bioen_kernels_logw.c:122-126,143-146
//     forces: f = theta KL + chi2                                   c_bioen_kernels_forces.c:244,276
//     Writes ab[i] = {r_i, avg_i} (logw column pass) or {r_i, 0} (forces t_j pass) and avg[i].
// ------------------------------------------------------------------------------------------------
struct FinalizeArgs {
    int m;
    const double* partial;   // row-pass slots (used when msum == nullptr)
    long long ld, L, chunk;
    const double* msum;      // already slot-reduced (and all-reduced) row sums + 3 tail scalars, or nullptr
    const double* tail;      // logw: the 3 weighted sums; forces: KL (local tail, or all-reduced in msum)
    const double* Y;
    double* ab;
    double* avg;
    int ab_with_avg;         // 1: ab = {r, avg}; 0: ab = {r, 0}
    int is_forces;
    double theta;
    double* partials;
    unsigned int* ticket;
    double* sc;
};

__global__ void __launch_bounds__(kVecThreads) k_finalize_rows(const FinalizeArgs a) {
    __shared__ double red[32];
    double v[1] = {0.0};
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.m) {
        double s;
        if (a.msum) {
            s = a.msum[i];
        } else {
            const int ns = pass_num_slots(i / kTileR, a.L, a.chunk);
            s = 0.0;
            for (int q = 0; q < ns; ++q) s += a.partial[(size_t)q * a.ld + i];
        }
        const double r = s - a.Y[i];
        a.avg[i] = s;
        reinterpret_cast<double2*>(a.ab)[i] = make_double2(r, a.ab_with_avg ? s : 0.0);
        v[0] = r * r;
    }
    const FinalizeArgs b = a;
    grid_sum<1>(v, a.partials, a.ticket, red, [=](const double(&t)[1]) {
        double* sc = b.sc;
        const double chi2 = 0.5 * t[0];
        double prior;
        if (b.is_forces) {
            sc[SC_KL] = b.tail[0];
            prior = b.tail[0] * b.theta;
        } else {
            // log s = gmax + log S  (the reference's un-stabilised s = sum exp(g_j))
            const double val = b.tail[0] - (sc[SC_GMAX] + log(sc[SC_S])) + sc[SC_LOGS0];
            prior = val * b.theta;
            sc[SC_GBAR] = b.tail[1];
            sc[SC_CAPGBAR] = b.tail[2];
        }
        sc[SC_CHI2] = chi2;
        sc[SC_PRIOR] = prior;
        sc[SC_F] = prior + chi2;
    });
}

// ------------------------------------------------------------------------------------------------
// K6 (logw): finish the column pass:
//     grad_j = w_j theta (g_j - <g> - G_j + <G>) + w_j sum_i r_i (y_ij - avg_i)   c_bioen_kernels_logw.c:214-217
//     plus the scalars the line search / stop tests need: grad.d, ||grad||^2, max|grad|.
// ------------------------------------------------------------------------------------------------
struct LogwGradArgs {
    int n;
    const double* col_partial;
    long long ld, L, chunk;
    const double* g;
    const double* G;
    const double* w;
    const double* d;   // may be nullptr
    double* grad;
    double theta;
    double* partials;  // gridDim.x * 3
    unsigned int* ticket;
    double* sc;
    // sharded run with the exchange fused in (p2p.nranks > 1): `wio` holds e_j and is overwritten with the normalised
    // w_j = e_j * sc[SC_WSCALE]; the block that finishes the grid reduction exchanges {grad.d, ||grad||^2, ||x||^2,
    // max|grad|} with the other ranks and leaves the global values in sc[]
    double* wio;
    P2PDev p2p;
};

__global__ void __launch_bounds__(kVecThreads) k_logw_grad(const LogwGradArgs a) {
    __shared__ double red[3 * 32];
    __shared__ double xs[4];
    const double gbar = a.sc[SC_GBAR], Gbar = a.sc[SC_CAPGBAR];
    const bool fused = a.p2p.nranks > 1;
    const double wscale = fused ? a.sc[SC_WSCALE] : 1.0;
    double dg = 0.0, gn = 0.0, gi = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const int ns = pass_num_slots(j / kTileC, a.L, a.chunk);
        double c = 0.0;
        for (int q = 0; q < ns; ++q) c += a.col_partial[(size_t)q * a.ld + j];
        double w = a.w[j];
        if (fused) {
            w *= wscale;
            a.wio[j] = w;
        }
        const double gr = w * a.theta * (a.g[j] - gbar - a.G[j] + Gbar) + w * c;
        a.grad[j] = gr;
        if (a.d) dg = fma(gr, a.d[j], dg);
        gn = fma(gr, gr, gn);
        gi = fmax(gi, fabs(gr));
    }
    double v[3] = {dg, gn, gi};
    if (!grid_sum_max_last<2>(v, a.partials, a.ticket, red)) return;
    if (!fused) {
        if (threadIdx.x == 0) {
            a.sc[SC_DG] = v[0];
            a.sc[SC_GNORM2] = v[1];
            a.sc[SC_GINF] = v[2];
        }
        return;
    }
    if (threadIdx.x == 0) {
        xs[0] = v[0];
        xs[1] = v[1];
        xs[2] = a.sc[SC_XNORM2];   // local ||x||^2 left by k_update_lse
        xs[3] = v[2];
    }
    int fail;
    const double* in = p2p_deliver_and_wait(a.p2p, xs, 4, &fail);
    if (threadIdx.x == 0) {
        double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
        for (int r = 0; r < a.p2p.nranks; ++r) {
            const double* q = in + r * a.p2p.cap;
            t0 += __ldcg(q); t1 += __ldcg(q + 1); t2 += __ldcg(q + 2); t3 = fmax(t3, __ldcg(q + 3));
        }
        if (fail) t0 = t1 = t2 = t3 = p2p_nan();
        a.sc[SC_DG] = t0;
        a.sc[SC_GNORM2] = t1;
        a.sc[SC_XNORM2] = t2;
        a.sc[SC_GINF] = t3;
    }
}

// ------------------------------------------------------------------------------------------------
// forces: normalised weights, guarded log-ratio and KL   (c_bioen_kernels_forces.c:156-171, 246-274)
//     w_j = w0_j exp(x_j - xmax) / S;   lr_j = log w_j - log w0_j = x_j - xmax - log S  where both
//     w_j >= DBL_MIN and w0_j >= DBL_MIN, else 0;  KL = sum_j w_j lr_j (local part -> msum tail[0])
// ------------------------------------------------------------------------------------------------
struct ForcesWeightsArgs {
    int n;
    const double* x;
    const double* w0;
    double* w;
    double* lr;
    const double* lse_pairs;
    int nranks;
    double* msum_tail;  // 1 double: local KL
    double* partials;
    unsigned int* ticket;
    double* sc;
};

__global__ void __launch_bounds__(kVecThreads) k_forces_weights(const ForcesWeightsArgs a) {
    __shared__ double red[32];
    double M, S;
    global_lse(a.lse_pairs, a.nranks, M, S);
    const double inv = 1.0 / S, logS = log(S);
    double v[1] = {0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const double x = a.x[j], w0 = a.w0[j];
        const double w = inv * (w0 * exp(x - M));
        const double lr = (w >= DBL_MIN && w0 >= DBL_MIN) ? (x - M - logS) : 0.0;
        a.w[j] = w;
        a.lr[j] = lr;
        v[0] = fma(lr, w, v[0]);
    }
    double* tail = a.msum_tail;
    double* sc = a.sc;
    grid_sum<1>(v, a.partials, a.ticket, red, [=](const double(&t)[1]) {
        tail[0] = t[0];
        sc[SC_GMAX] = M;
        sc[SC_S] = S;
    });
}

// forces, reference entry points that receive the WEIGHTS instead of the forces
// (c_bioen_kernels_forces.c:246-274): lr_j = log w_j - log w0_j where both >= DBL_MIN, else 0; KL = sum w_j lr_j
struct ForcesLrArgs {
    int n;
    const double* w;
    const double* w0;
    double* lr;
    double* msum_tail;
    double* partials;
    unsigned int* ticket;
};

__global__ void __launch_bounds__(kVecThreads) k_forces_lr_from_w(const ForcesLrArgs a) {
    __shared__ double red[32];
    double v[1] = {0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const double w = a.w[j], w0 = a.w0[j];
        const double lr = (w >= DBL_MIN && w0 >= DBL_MIN) ? (log(w) - log(w0)) : 0.0;
        a.lr[j] = lr;
        v[0] = fma(lr, w, v[0]);
    }
    double* tail = a.msum_tail;
    grid_sum<1>(v, a.partials, a.ticket, red, [=](const double(&t)[1]) { tail[0] = t[0]; });
}

// forces: E_j = (theta (1 + lr_j) + t_j) w_j,  t_j = column-pass sums    (c_bioen_kernels_forces.c:321-328)
struct ForcesEArgs {
    int n;
    const double* col_partial;
    long long ld, L, chunk;
    const double* w;
    const double* lr;
    double* E;
    double theta;
};

__global__ void __launch_bounds__(kVecThreads) k_forces_E(const ForcesEArgs a) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const int ns = pass_num_slots(j / kTileC, a.L, a.chunk);
        double t = 0.0;
        for (int q = 0; q < ns; ++q) t += a.col_partial[(size_t)q * a.ld + j];
        a.E[j] = ((1.0 + a.lr[j]) * a.theta + t) * a.w[j];
    }
}

// forces: finish the gradient row pass: grad_i = sum_slots, plus grad.d, ||grad||^2, max|grad| (M is small:
// one block).  When `msum` is given the slots were already reduced (and all-reduced across ranks).
struct ForcesGradArgs {
    int m;
    const double* partial;
    long long ld, L, chunk;
    const double* msum;
    const double* d;
    double* grad;
    double* sc;
};

__global__ void __launch_bounds__(1024) k_forces_grad(const ForcesGradArgs a) {
    __shared__ double red[3 * 32];
    double dg = 0.0, gn = 0.0, gi = 0.0;
    for (int i = threadIdx.x; i < a.m; i += blockDim.x) {
        double s;
        if (a.msum) {
            s = a.msum[i];
        } else {
            const int ns = pass_num_slots(i / kTileR, a.L, a.chunk);
            s = 0.0;
            for (int q = 0; q < ns; ++q) s += a.partial[(size_t)q * a.ld + i];
        }
        a.grad[i] = s;
        if (a.d) dg = fma(s, a.d[i], dg);
        gn = fma(s, s, gn);
        gi = fmax(gi, fabs(s));
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    dg = warp_sum(dg); gn = warp_sum(gn); gi = warp_max(gi);
    if (lane == 0) { red[wid] = dg; red[32 + wid] = gn; red[64 + wid] = gi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < nw; ++w) { dg += red[w]; gn += red[32 + w]; gi = fmax(gi, red[64 + w]); }
        a.sc[SC_DG] = dg;
        a.sc[SC_GNORM2] = gn;
        a.sc[SC_GINF] = gi;
    }
}

// forces: x = xp + stp*d (optional), ||x||^2, and ab[i] = {x_i, 0} for the first column pass (M is small)
struct ForcesUpdateArgs {
    int m;
    double* x;
    const double* xp;
    const double* d;
    double stp;
    double* ab;
    double* sc;
};

__global__ void __launch_bounds__(1024) k_forces_update(const ForcesUpdateArgs a) {
    __shared__ double red[32];
    double v[1] = {0.0};
    for (int i = threadIdx.x; i < a.m; i += blockDim.x) {
        double x = a.x[i];
        if (a.xp) {
            x = fma(a.stp, a.d[i], a.xp[i]);
            a.x[i] = x;
        }
        reinterpret_cast<double2*>(a.ab)[i] = make_double2(x, 0.0);
        v[0] = fma(x, x, v[0]);
    }
    block_sum<1>(v, red);
    if (threadIdx.x == 0) a.sc[SC_XNORM2] = v[0];
}

// ------------------------------------------------------------------------------------------------
// generic vector kernels (device-resident minimisers)
// ------------------------------------------------------------------------------------------------
// out[0..K) = sums of up to 3 dot products in one sweep; pairs given as pointers (nullptr = unused)
struct Dot3Args {
    int n;
    const double *a0, *b0, *a1, *b1, *a2, *b2;
    double* out;  // device, 3 doubles
    double* partials;
    unsigned int* ticket;
};

__global__ void __launch_bounds__(kVecThreads) k_dot3(const Dot3Args a) {
    __shared__ double red[3 * 32];
    double v[3] = {0.0, 0.0, 0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        v[0] = fma(a.a0[j], a.b0[j], v[0]);
        if (a.a1) v[1] = fma(a.a1[j], a.b1[j], v[1]);
        if (a.a2) v[2] = fma(a.a2[j], a.b2[j], v[2]);
    }
    double* out = a.out;
    grid_sum<3>(v, a.partials, a.ticket, red, [=](const double(&t)[3]) {
        out[0] = t[0];
        out[1] = t[1];
        out[2] = t[2];
    });
}

// z = alpha*x + beta*y  (z may alias x or y; y may be nullptr when beta == 0)
__global__ void __launch_bounds__(kVecThreads)
    k_axpby(int n, double alpha, const double* x, double beta, const double* y, double* z) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const double v = alpha * x[j];
        z[j] = y ? fma(beta, y[j], v) : v;
    }
}

// L-BFGS: s = x - xp, y = g - gp, ys = y.s, yy = y.y; then xp <- x, gp <- g for the next iteration
//     (liblbfgs lbfgs.c:543-555 and 462-463)
struct PairArgs {
    int n;
    const double *x, *g;
    double *xp, *gp;
    double *s, *y;
    int slot;          // ring index: sc[SC_YS0 + slot] = ys
    double* partials;
    unsigned int* ticket;
    double* sc;
    P2PDev p2p;        // nranks > 1: the dot products are summed over the ranks by the finishing block
};

// the block that finished a grid reduction sums its K totals (thread 0 holds them in v) over the ranks
template <int K>
__device__ __forceinline__ void p2p_sum_inline(const P2PDev& p, double (&v)[K]) {
    __shared__ double xs[K];
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) xs[k] = v[k];
    }
    int fail;
    const double* in = p2p_deliver_and_wait(p, xs, K, &fail);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            double s = 0.0;
            for (int r = 0; r < p.nranks; ++r) s += __ldcg(in + r * p.cap + k);
            v[k] = fail ? p2p_nan() : s;
        }
    }
}

__global__ void __launch_bounds__(kVecThreads) k_lbfgs_pair(const PairArgs a) {
    __shared__ double red[2 * 32];
    double v[2] = {0.0, 0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const double x = a.x[j], g = a.g[j];
        const double s = x - a.xp[j], y = g - a.gp[j];
        a.s[j] = s;
        a.y[j] = y;
        a.xp[j] = x;
        a.gp[j] = g;
        v[0] = fma(y, s, v[0]);
        v[1] = fma(y, y, v[1]);
    }
    if (!grid_sum_last<2>(v, a.partials, a.ticket, red)) return;
    if (a.p2p.nranks > 1) p2p_sum_inline<2>(a.p2p, v);
    if (threadIdx.x == 0) {
        a.sc[SC_YS] = v[0];
        a.sc[SC_YY] = v[1];
        a.sc[SC_YS0 + a.slot] = v[0];
    }
}

// One step of the two-loop recursion, fused: d <- [init ? -g : d] + coef * u ; d *= scale ; out = v . d
//     coef and scale are formed on the device from raw dot products already sitting in sc[]:
//       coef  = csign * sc[c_num] / sc[c_den]  (+ sc[c2_num]/sc[c2_den] * c2sign when c2_num >= 0)
//       scale = sc[s_num] / sc[s_den]          (when s_num >= 0)
//     so the whole recursion (liblbfgs lbfgs.c:572-598) runs without a host round trip.
struct TwoLoopArgs {
    int n;
    double* d;
    const double* g;      // used when init
    int init;
    const double* u;      // nullptr: no axpy
    int c_num, c_den; double csign;
    int c2_num, c2_den; double c2sign;
    int s_num, s_den;
    const double* v;      // nullptr: no dot
    int out;              // sc index receiving the raw dot v.d
    double* partials;
    unsigned int* ticket;
    double* sc;
    P2PDev p2p;           // nranks > 1: the dot product is summed over the ranks by the finishing block
};

__global__ void __launch_bounds__(kVecThreads) k_lbfgs_twoloop(const TwoLoopArgs a) {
    __shared__ double red[32];
    double coef = 0.0, scale = 1.0;
    if (a.u) {
        coef = a.csign * (a.sc[a.c_num] / a.sc[a.c_den]);
        if (a.c2_num >= 0) coef += a.c2sign * (a.sc[a.c2_num] / a.sc[a.c2_den]);
    }
    if (a.s_num >= 0) scale = a.sc[a.s_num] / a.sc[a.s_den];
    double v[1] = {0.0};
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        double dj = a.init ? -a.g[j] : a.d[j];
        if (a.u) dj = fma(coef, a.u[j], dj);
        if (a.s_num >= 0) dj *= scale;
        a.d[j] = dj;
        if (a.v) v[0] = fma(a.v[j], dj, v[0]);
    }
    if (a.v) {
        if (!grid_sum_last<1>(v, a.partials, a.ticket, red)) return;
        if (a.p2p.nranks > 1) p2p_sum_inline<1>(a.p2p, v);
        if (threadIdx.x == 0) a.sc[a.out] = v[0];
    }
}

// ------------------------------------------------------------------------------------------------
// L-BFGS update for SMALL n (n <= 1024: the forces method, and log-weights problems with few structures -- every
// fixture of the reference's test-suite): k_lbfgs_pair + the 2*bound+1 kernels of the two-loop recursion as ONE
// single-CTA kernel.  Thread j owns element j of every vector and keeps d_j, g_j and the six (s, y) pairs in
// registers; the 2*bound+2 dot products are block reductions (one __syncthreads each), the coefficients are formed from
// the same raw dot products in the same order as k_lbfgs_twoloop does, and the same scalar-file outputs are written
// (ys, yy, the ys and raw s.d rings, g.d; the second loop's dots stay in registers instead of SC_BETA / SC_BETA2).
// 15 launches of ~3 us become one of ~5 us -- at these sizes the update, not the evaluation, was most of an iteration.
// For n <= 256 (one block in the multi-kernel path as well) the result is bit-identical to that path.
// ------------------------------------------------------------------------------------------------
constexpr int kSmallUpdateMaxN = 1024;
constexpr int kSmallUpdateM = 6;   // history length (liblbfgs default; BioEn never changes it)

struct SmallUpdateArgs {
    int n;
    const double *x, *g;
    double *xp, *gp, *d;
    double* S[kSmallUpdateM];
    double* Y[kSmallUpdateM];
    int end;     // ring slot that receives the new pair
    int bound;   // pairs in use (including the new one)
    double* sc;
};

// all threads of the block get the sum; `red` is [2][32] and toggles so that one barrier per reduction is enough
__device__ __forceinline__ double small_block_sum(double v, double (*red)[32], int& phase) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    if (lane == 0) red[phase][wid] = v;
    __syncthreads();
    const double t = warp_sum(lane < nw ? red[phase][lane] : 0.0);
    phase ^= 1;
    return t;
}

__device__ __forceinline__ double small_pick(const double (&v)[kSmallUpdateM], int k) {
    double r = v[0];
#pragma unroll
    for (int t = 1; t < kSmallUpdateM; ++t) r = (k == t) ? v[t] : r;
    return r;
}

__global__ void __launch_bounds__(kSmallUpdateMaxN, 1) k_lbfgs_update_small(const SmallUpdateArgs a) {
    __shared__ double red[2][32];
    __shared__ double s_alpha[kSmallUpdateM], s_ys[kSmallUpdateM];
    const int j = threadIdx.x;
    const bool on = j < a.n;
    int phase = 0;
    double sv[kSmallUpdateM], yv[kSmallUpdateM];
    // pairs already in the ring: slots end-1, end-2, ... (bound - 1 of them)
#pragma unroll
    for (int t = 0; t < kSmallUpdateM; ++t) {
        const int age = (a.end - t + kSmallUpdateM) % kSmallUpdateM;   // 0 = the new pair
        const bool used = on && age != 0 && age < a.bound;
        sv[t] = used ? a.S[t][j] : 0.0;
        yv[t] = used ? a.Y[t][j] : 0.0;
    }
    if (j < kSmallUpdateM) s_ys[j] = a.sc[SC_YS0 + j];
    double g = 0.0, s_new = 0.0, y_new = 0.0;
    if (on) {
        const double x = a.x[j];
        g = a.g[j];
        s_new = x - a.xp[j];
        y_new = g - a.gp[j];
        a.xp[j] = x;
        a.gp[j] = g;
    }
#pragma unroll
    for (int t = 0; t < kSmallUpdateM; ++t) {
        if (t == a.end) {
            sv[t] = s_new;
            yv[t] = y_new;
            if (on) { a.S[t][j] = s_new; a.Y[t][j] = y_new; }
        }
    }
    // ys = y.s, yy = y.y of the new pair (lbfgs.c:543-555)
    const double ys = small_block_sum(y_new * s_new + 0.0, red, phase);
    const double yy = small_block_sum(y_new * y_new + 0.0, red, phase);
    if (j == 0) {
        s_ys[a.end] = ys;
        a.sc[SC_YS] = ys;
        a.sc[SC_YY] = yy;
        a.sc[SC_YS0 + a.end] = ys;
    }
    // two-loop recursion (lbfgs.c:572-598); slot of the i-th newest pair: (end - i) mod m
    double dj = -g;
    int slot = a.end;
    double alpha_raw = small_block_sum(small_pick(sv, slot) * dj + 0.0, red, phase);   // also publishes s_ys
    double beta_raw = 0.0;
    for (int i = 0; i < a.bound; ++i) {
        if (j == 0) { s_alpha[slot] = alpha_raw; a.sc[SC_ALPHA0 + slot] = alpha_raw; }
        const double coef = -1.0 * (alpha_raw / s_ys[slot]);
        dj = fma(coef, small_pick(yv, slot), dj);
        if (i + 1 < a.bound) {
            slot = (slot + kSmallUpdateM - 1) % kSmallUpdateM;
            alpha_raw = small_block_sum(small_pick(sv, slot) * dj + 0.0, red, phase);
        } else {
            dj *= ys / yy;
            beta_raw = small_block_sum(small_pick(yv, slot) * dj + 0.0, red, phase);
        }
    }
    // slot = oldest pair now; s_alpha is complete (the last store is ordered by the barrier of the reduction above
    // only for i + 1 < bound, so read the oldest alpha from the register)
    double dginit = 0.0;
    for (int i = a.bound - 1; i >= 0; --i) {
        const double al = (i == a.bound - 1) ? alpha_raw : s_alpha[slot];
        const double ysl = s_ys[slot];
        double coef = 1.0 * (al / ysl);
        coef += -1.0 * (beta_raw / ysl);
        dj = fma(coef, small_pick(sv, slot), dj);
        if (i > 0) {
            slot = (slot + 1) % kSmallUpdateM;
            beta_raw = small_block_sum(small_pick(yv, slot) * dj + 0.0, red, phase);
        } else {
            dginit = small_block_sum(g * dj + 0.0, red, phase);
        }
    }
    if (on) a.d[j] = dj;
    if (j == 0) a.sc[SC_DGINIT] = dginit;
}

// sharded twin of k_colgrad_finish (stream_pass.cuh): per-CTA partials summed in CTA order, then ONE exchange of
// {grad.d, ||grad||^2, ||x||^2, max|grad|} between the ranks from this block
__global__ void __launch_bounds__(256) k_colgrad_finish_sharded(int ncta, const double* cta_part, double* sc,
                                                                const P2PDev p2p) {
    __shared__ double red[3][8];
    __shared__ double xs[4];
    double t0 = 0.0, t1 = 0.0, t2 = 0.0;
    for (int b = threadIdx.x; b < ncta; b += 256) {
        t0 += cta_part[3 * b];
        t1 += cta_part[3 * b + 1];
        t2 = fmax(t2, cta_part[3 * b + 2]);
    }
    t0 = warp_sum(t0); t1 = warp_sum(t1); t2 = warp_max(t2);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = t0; red[1][threadIdx.x >> 5] = t1; red[2][threadIdx.x >> 5] = t2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { t0 += red[0][w]; t1 += red[1][w]; t2 = fmax(t2, red[2][w]); }
        xs[0] = t0; xs[1] = t1; xs[2] = sc[SC_XNORM2]; xs[3] = t2;
    }
    int fail;
    const double* in = p2p_deliver_and_wait(p2p, xs, 4, &fail);
    if (threadIdx.x == 0) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        for (int r = 0; r < p2p.nranks; ++r) {
            const double* q = in + r * p2p.cap;
            s0 += __ldcg(q); s1 += __ldcg(q + 1); s2 += __ldcg(q + 2); s3 = fmax(s3, __ldcg(q + 3));
        }
        if (fail) s0 = s1 = s2 = s3 = p2p_nan();
        sc[SC_DG] = s0; sc[SC_GNORM2] = s1; sc[SC_XNORM2] = s2; sc[SC_GINF] = s3;
    }
}

// ------------------------------------------------------------------------------------------------
// Sharded forces method on the fused two-pass kernels: the three exchanges of an evaluation issued from inside the
// kernels that produce the values (as the log-weights path does), instead of three 1-block exchange launches.
//   k_forces_lse_gather        this rank's (max, sum) pair from the CTA rows of F1, gathered over the ranks
//   k_forces_rows_finish       out_i = sum over the CTA rows of a fused pass (scaled by the global softmax pair for
//                              F1); the block that finishes last sums the M (+1: KL) values over the ranks and runs
//                              what k_finalize_rows (objective half) or k_forces_grad (gradient half) would run
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_forces_lse_gather(int nrows, const double* lse, double* sc_pair,
                                                           double* pairs_all, const P2PDev p2p) {
    __shared__ double sm[256], ss[256];
    double m = -DBL_MAX, s = 0.0;
    for (int c = threadIdx.x; c < nrows; c += 256) lse_merge(m, s, lse[2 * c], lse[2 * c + 1]);
    sm[threadIdx.x] = m;
    ss[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            double m1 = sm[threadIdx.x], s1 = ss[threadIdx.x];
            lse_merge(m1, s1, sm[threadIdx.x + o], ss[threadIdx.x + o]);
            sm[threadIdx.x] = m1;
            ss[threadIdx.x] = s1;
        }
        __syncthreads();
    }
    __shared__ double pair[2];
    if (threadIdx.x == 0) {
        sc_pair[0] = pair[0] = sm[0];
        sc_pair[1] = pair[1] = ss[0];
    }
    __syncthreads();
    p2p_exchange_block(p2p, pair, pairs_all, 2, kP2PGather);
}

struct RowsFinishArgs {
    int m, nrows;
    const double* part;
    long long ldp;
    const double* lse_rows;    // F1: per-row (max, sum) pairs; nullptr for F2
    const double* lse_pairs;   // [nranks][2] gathered pairs
    int nranks;
    double* out;               // msum: m values (+ tail)
    int ntail;                 // 1: out[m] holds this rank's KL part (objective half); 0: gradient half
    int gradient;              // 0: finish the objective half, 1: finish the gradient half
    const double* Y;
    double* ab;
    double* avg;
    double theta;
    const double* d;           // gradient half: optional direction
    double* grad;
    unsigned int* ticket;
    double* sc;
    P2PDev p2p;
};

__global__ void __launch_bounds__(256) k_forces_rows_finish(const RowsFinishArgs a) {
    __shared__ double red[8][33];
    __shared__ bool is_last;
    double M = 0.0, inv = 1.0;
    if (a.lse_rows) {
        double S;
        global_lse(a.lse_pairs, a.nranks, M, S);
        inv = 1.0 / S;
    }
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + tx;
    double s = 0.0;
    for (int c = ty; c < a.nrows; c += 8) {
        const double scale = a.lse_rows ? exp(a.lse_rows[2 * c] - M) * inv : 1.0;
        if (i < a.m) s = fma(a.part[(size_t)c * a.ldp + i], scale, s);
    }
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && i < a.m) {
        double t = red[0][tx];
#pragma unroll
        for (int g = 1; g < 8; ++g) t += red[g][tx];
        a.out[i] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        is_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x == 0) *a.ticket = 0;
    // ---- the finishing block: sum over the ranks, then the M-vector epilogue
    const int count = a.m + a.ntail;
    const double* vals = a.out;
    int fail = 0;
    const double* in = nullptr;
    if (a.p2p.nranks > 1) in = p2p_deliver_and_wait(a.p2p, a.out, count, &fail);
    auto total = [&](int k) {
        if (!in) return __ldcg(vals + k);
        double t = 0.0;
        for (int r = 0; r < a.p2p.nranks; ++r) t += __ldcg(in + r * a.p2p.cap + k);
        return t;
    };
    double* redf = &red[0][0];
    if (!a.gradient) {
        double v[1] = {0.0};
        for (int k = threadIdx.x; k < a.m; k += blockDim.x) {
            const double sum = total(k);
            const double r = sum - a.Y[k];
            a.avg[k] = sum;
            reinterpret_cast<double2*>(a.ab)[k] = make_double2(r, 0.0);
            v[0] = fma(r, r, v[0]);
        }
        block_sum<1>(v, redf);
        if (threadIdx.x == 0) {
            const double kl = total(a.m), chi2 = 0.5 * v[0];
            a.sc[SC_KL] = kl;
            a.sc[SC_CHI2] = chi2;
            a.sc[SC_PRIOR] = kl * a.theta;
            a.sc[SC_F] = fail ? p2p_nan() : kl * a.theta + chi2;
        }
    } else {
        double v[3] = {0.0, 0.0, 0.0};
        double gi = 0.0;
        for (int k = threadIdx.x; k < a.m; k += blockDim.x) {
            const double sum = total(k);
            a.grad[k] = sum;
            if (a.d) v[0] = fma(sum, a.d[k], v[0]);
            v[1] = fma(sum, sum, v[1]);
            gi = fmax(gi, fabs(sum));
        }
        v[2] = 0.0;
        block_sum<3>(v, redf);
        // max |grad| over the block
        __shared__ double gmax[8];
        gi = warp_max(gi);
        if ((threadIdx.x & 31) == 0) gmax[threadIdx.x >> 5] = gi;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) gi = fmax(gi, gmax[w]);
            a.sc[SC_DG] = fail ? p2p_nan() : v[0];
            a.sc[SC_GNORM2] = fail ? p2p_nan() : v[1];
            a.sc[SC_GINF] = gi;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// L-BFGS direction update in coefficient space (opt-in, BIOEN_B200_OPT_LBFGS_GRAM).
//
// liblbfgs' two-loop recursion (lbfgs.c:572-598) is a chain of 2*bound+1 dot products, each of which needs the vector
// the previous one produced: 2*bound+2 kernels and -- sharded -- as many exchanges per iteration.  All vectors of the
// recursion lie in the span of the 2*bound+1 basis vectors {s_i, y_i, g}, so the same recursion can run on the
// (2*bound+1)-dimensional coefficient vector once the Gram matrix of the basis is known (Chen et al., "Large-scale
// L-BFGS using MapReduce", NIPS 2014).  Only three basis vectors change per iteration (the new s, the new y and g):
//   kernel 1  k_lbfgs_gram_pair   s = x - xp, y = g - gp (stored in the ring), xp <- x, gp <- g, and the 3 x 13 dot
//                                 products of {s, y, g} with the whole basis in the SAME sweep; the finishing block
//                                 sums them over the ranks (ONE exchange), updates the resident Gram matrix, runs the
//                                 recursion on 13 coefficients and leaves them with g.d, y.s, y.y in device memory
//   kernel 2  k_lbfgs_combine     d = sum_k c_k b_k
// i.e. 2 kernels, 1 exchange and ~35 vector streams per iteration instead of 14 kernels, 13 exchanges and ~60.
// The arithmetic is algebraically that of the two-loop recursion but rounds differently (dot products with the running
// vector are replaced by combinations of Gram entries), so trajectories differ from the default path in the last bits
// from the first iteration on: that is why it is an option and not the default.
// ------------------------------------------------------------------------------------------------
constexpr int kGramM = 6;                       // history length this path supports (liblbfgs default, BioEn never changes it)
constexpr int kGramB = 2 * kGramM + 1;          // basis: s[0..5], y[0..5], g
constexpr int kGramK = 3 * kGramB;              // dot products per iteration

struct GramPairArgs {
    int n;
    const double *x, *g;
    double *xp, *gp;
    double* S[kGramM];
    double* Y[kGramM];
    int end;            // ring slot receiving the new pair
    int bound;          // pairs in the ring INCLUDING the new one
    double* gram;       // [kGramB][kGramB] resident Gram matrix, then kGramB coefficients at gram + kGramB*kGramB
    double* partials;   // gridDim.x * kGramK
    unsigned int* ticket;
    double* sc;
    P2PDev p2p;
};

__global__ void __launch_bounds__(kVecThreads) k_lbfgs_gram_pair(const GramPairArgs a) {
    __shared__ double red[kGramK * 32];
    double v[kGramK];
#pragma unroll
    for (int k = 0; k < kGramK; ++k) v[k] = 0.0;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        const double x = a.x[j], g = a.g[j];
        const double s = x - a.xp[j], y = g - a.gp[j];
        a.xp[j] = x;
        a.gp[j] = g;
#pragma unroll
        for (int t = 0; t < kGramM; ++t) {
            double sv = 0.0, yv = 0.0;
            if (t == a.end) {
                a.S[t][j] = s;
                a.Y[t][j] = y;
                sv = s;
                yv = y;
            } else if (t < a.bound) {        // slots fill up in order 0, 1, ...: valid slots are [0, bound)
                sv = a.S[t][j];
                yv = a.Y[t][j];
            }
            v[3 * t + 0] = fma(s, sv, v[3 * t + 0]);
            v[3 * t + 1] = fma(y, sv, v[3 * t + 1]);
            v[3 * t + 2] = fma(g, sv, v[3 * t + 2]);
            v[3 * (kGramM + t) + 0] = fma(s, yv, v[3 * (kGramM + t) + 0]);
            v[3 * (kGramM + t) + 1] = fma(y, yv, v[3 * (kGramM + t) + 1]);
            v[3 * (kGramM + t) + 2] = fma(g, yv, v[3 * (kGramM + t) + 2]);
        }
        v[3 * (kGramB - 1) + 0] = fma(s, g, v[3 * (kGramB - 1) + 0]);
        v[3 * (kGramB - 1) + 1] = fma(y, g, v[3 * (kGramB - 1) + 1]);
        v[3 * (kGramB - 1) + 2] = fma(g, g, v[3 * (kGramB - 1) + 2]);
    }
    if (!grid_sum_last<kGramK>(v, a.partials, a.ticket, red)) return;
    if (a.p2p.nranks > 1) p2p_sum_inline<kGramK>(a.p2p, v);
    if (threadIdx.x != 0) return;
    // ---- the finishing thread: Gram update + the recursion on the coefficients
    double* Gm = a.gram;
    const int is = a.end, iy = kGramM + a.end, ig = kGramB - 1;
    for (int k = 0; k < kGramB; ++k) {
        Gm[is * kGramB + k] = Gm[k * kGramB + is] = v[3 * k + 0];
        Gm[iy * kGramB + k] = Gm[k * kGramB + iy] = v[3 * k + 1];
        Gm[ig * kGramB + k] = Gm[k * kGramB + ig] = v[3 * k + 2];
    }
    double c[kGramB], alpha[kGramM];
    for (int k = 0; k < kGramB; ++k) c[k] = 0.0;
    c[ig] = -1.0;                                             // q = -g
    auto dotq = [&](int row) {                                 // b_row . q
        double s = 0.0;
        for (int k = 0; k < kGramB; ++k) s = fma(c[k], Gm[row * kGramB + k], s);
        return s;
    };
    int jslot = (a.end + 1) % kGramM;                          // liblbfgs: j = end (after its increment), then --j
    for (int i = 0; i < a.bound; ++i) {
        jslot = (jslot + kGramM - 1) % kGramM;                 // newest ... oldest
        const double ys = Gm[jslot * kGramB + kGramM + jslot];
        alpha[jslot] = dotq(jslot) / ys;
        c[kGramM + jslot] -= alpha[jslot];
    }
    const double ys_new = Gm[is * kGramB + iy], yy_new = Gm[iy * kGramB + iy];
    const double h0 = ys_new / yy_new;
    for (int k = 0; k < kGramB; ++k) c[k] *= h0;
    for (int i = 0; i < a.bound; ++i) {                        // oldest ... newest
        const double ys = Gm[jslot * kGramB + kGramM + jslot];
        const double beta = dotq(kGramM + jslot) / ys;
        c[jslot] += alpha[jslot] - beta;
        jslot = (jslot + 1) % kGramM;
    }
    for (int k = 0; k < kGramB; ++k) Gm[kGramB * kGramB + k] = c[k];
    a.sc[SC_DGINIT] = dotq(ig);
    a.sc[SC_YS] = ys_new;
    a.sc[SC_YY] = yy_new;
    a.sc[SC_YS0 + a.end] = ys_new;
}

struct GramCombineArgs {
    int n;
    const double* S[kGramM];
    const double* Y[kGramM];
    const double* g;
    const double* coef;   // kGramB coefficients (device)
    int bound;
    double* d;
};

__global__ void __launch_bounds__(kVecThreads) k_lbfgs_combine(const GramCombineArgs a) {
    __shared__ double c[kGramB];
    if (threadIdx.x < kGramB) c[threadIdx.x] = a.coef[threadIdx.x];
    __syncthreads();
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < a.n; j += gridDim.x * blockDim.x) {
        double dj = c[kGramB - 1] * a.g[j];
#pragma unroll
        for (int t = 0; t < kGramM; ++t) {
            if (t < a.bound) {
                dj = fma(c[t], a.S[t][j], dj);
                dj = fma(c[kGramM + t], a.Y[t][j], dj);
            }
        }
        a.d[j] = dj;
    }
}

// fp64 -> fp32 copy of the resident matrix (opt-in reduced-precision STORAGE, BIOEN_B200_OPT_FP32_STORAGE);
// round-to-nearest; columns >= n of the destination stay zero
__global__ void __launch_bounds__(256) k_convert_f32(const double* Y, long long ld, int m, int n, float* Y32, long long ld32) {
    const long long total = (long long)m * n;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / n);
        const long long j = t - (long long)i * n;
        Y32[(size_t)i * ld32 + j] = (float)Y[(size_t)i * ld + j];
    }
}

// ------------------------------------------------------------------------------------------------
// In-place row-affine transform of the resident matrix:  y_ij <- scale_i * y_ij + offset_i   (columns j < n only: the
// padding stays zero).  This is how a nuisance-parameter refit (DEER modulation depth, scattering scale factor:
// bioen/analyze/observables/observables.py:110-143 rebuilds the whole matrix in a Python double loop) is committed
// to the matrix that lives in HBM: one read + one write pass, 2*M*N*8 bytes, HBM-bound.
__global__ void __launch_bounds__(256) k_affine_rows(double* Y, long long ld, int m, int n, const double* scale,
                                                     const double* offset) {
    const long long npair = (n + 1) / 2, total = (long long)m * npair;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / npair);
        const long long jp = t - (long long)i * npair;
        const double s = scale[i], o = offset[i];
        double2* p = reinterpret_cast<double2*>(Y + (size_t)i * ld) + jp;
        double2 v = *p;
        v.x = fma(s, v.x, o);
        if (2 * jp + 1 < n) v.y = fma(s, v.y, o);
        *p = v;
    }
}

// ------------------------------------------------------------------------------------------------
// Plain read-only stream over the resident matrix: every thread sums 16-byte loads, nothing is written.  An upper
// reference for what a read-only pass over yTilde can reach on this device (the copy figure in
// MEASURED_PEAKS.json mixes reads and writes and is lower).
template <int U>
__global__ void __launch_bounds__(1024, 2) k_read_stream(const double2* __restrict__ p, size_t n2, double* sink) {
    double s0 = 0.0, s1 = 0.0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (U - 1) * stride < n2; i += U * stride) {
        double2 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = __ldcs(p + i + u * stride);
#pragma unroll
        for (int u = 0; u < U; ++u) { s0 += v[u].x; s1 += v[u].y; }
    }
    for (; i < n2; i += stride) {
        const double2 v = __ldcs(p + i);
        s0 += v.x;
        s1 += v.y;
    }
    if (s0 + s1 == 1.2345e-300) *sink = s0;   // keeps the loads alive, never true in practice
}

// The same read-only measurement with the ACCESS ORDER of the matrix passes: a block reads 32-row x 128-column
// tiles (32 segments of 1 KB, one row pitch apart) in one of four orders.  Separates "what the tile order costs at
// the DRAM" from "what the TMA pipeline costs".  order 0: row pass, contiguous chunk of tiles per block (tiles of a
// row tile are adjacent column blocks); 1: row pass, tiles dealt round-robin to the blocks; 2: column pass,
// contiguous chunk (a run walks down the rows of one column block); 3: column pass, runs dealt round-robin;
// 4: column pass, contiguous chunk, a run covers two adjacent column blocks.
__global__ void __launch_bounds__(1024, 2)
    k_read_tiles(const double* __restrict__ Y, long long ld, int M, int nRT, int nCB, int order, double* sink) {
    const long long T = (long long)nRT * nCB, G = gridDim.x, b = blockIdx.x;
    const long long chunk = (T + G - 1) / G;
    const int r = threadIdx.x >> 5, c = threadIdx.x & 31;
    double s0 = 0.0, s1 = 0.0;
    auto tile = [&](long long rt, long long cb) {
        const long long row = rt * 32 + r;
        if (row < M) {
            const double2* p = reinterpret_cast<const double2*>(Y + row * ld + cb * 128);
            const double2 u = __ldcs(p + c), v = __ldcs(p + 32 + c);
            s0 += u.x + v.x;
            s1 += u.y + v.y;
        }
    };
    if (order == 0 || order == 2) {
        const long long t0 = b * chunk, t1 = (t0 + chunk < T) ? t0 + chunk : T;
        const long long L = (order == 0) ? nCB : nRT;
        for (long long t = t0; t < t1; ++t) {
            const long long run = t / L, k = t - run * L;
            if (order == 0) tile(run, k); else tile(k, run);
        }
    } else if (order == 1) {
        for (long long t = b; t < T; t += G) tile(t / nCB, t % nCB);
    } else if (order == 4) {
        // column pass whose runs cover TWO adjacent column blocks: 2 KB contiguous per row, contiguous chunks
        const long long npair = (nCB + 1) / 2, Tp = npair * nRT, chunkp = (Tp + G - 1) / G;
        const long long t0 = b * chunkp, t1 = (t0 + chunkp < Tp) ? t0 + chunkp : Tp;
        for (long long t = t0; t < t1; ++t) {
            const long long p = t / nRT, rt = t - p * nRT;
            tile(rt, 2 * p);
            if (2 * p + 1 < nCB) tile(rt, 2 * p + 1);
        }
    } else {
        for (long long cb = b; cb < nCB; cb += G)
            for (long long rt = 0; rt < nRT; ++rt) tile(rt, cb);
    }
    if (s0 + s1 == 1.2345e-300) *sink = s0;
}

}  // namespace bioen
