// persistent_eval.cuh -- one whole evaluation (objective, or objective + gradient) as ONE cooperative kernel.
//
// The stand-alone path launches 6 kernels per log-weights evaluation (10-11 per forces evaluation on the tile
// kernels).  That is invisible next to two 1.1 ms passes over an 8 GB matrix, but it IS the evaluation when yTilde
// is small: at the ala5 shape (28 x 50 001, 11 MB, L2-resident) a forces evaluation took 0.129 ms of which the four
// passes over the matrix are ~0.03 ms; at config 2 (500 x 1e5) the small kernels are 25 % of a step; and with N = 1e6
// split over 8 GPUs (1 GB per GPU) launch gaps, kernel ramp-up / tail and the separate exchange kernels cost 0.07 ms
// next to 0.30 ms of passes.  Here one persistent CTA per SM runs the phases of the evaluation back to back, separated
// by grid barriers (sense-reversing: an arrival count and a generation word in global memory, no state from the
// host; the kernel is launched cooperatively so all CTAs are resident):
//
//   log-weights   V0 x = xp + stp d, local (max, sum exp)  | V1 global (max, S), w_j, prior sums | P2 row pass  avg
//                 V3 (CTA 0) slots -> avg, r, chi^2, f [+ the ONE exchange of a sharded run]   -- objective done --
//                 P4 column pass  c_j | V5 grad_j, grad.d, |grad|^2, max|grad| [+ exchange of 4 scalars]
//   forces        V0 (CTA 0) f = xp + stp d, ab | P1 column pass x_j | V2 x_j, local (max, sum w0 exp)
//   (tile path)   V3 w_j, lr_j, KL | P4 row pass avg | V5 (CTA 0) avg, r, chi^2, f             -- objective done --
//                 P6 column pass t_j | V7 E_j | P8 row pass grad | V9 (CTA 0) grad, grad.d, |grad|^2, max|grad|
//
// The passes are the SAME producer / consumer code as stream_pass_kernel (pass_produce / pass_consume: TMA tiles,
// 4-stage mbarrier ring, register accumulators, fixed-order slots); the ring simply keeps turning from one pass to
// the next.  Vectors that a later pass reads through bulk copies (w, ab, E, avg) are written with ordinary stores in
// an earlier phase, so every grid barrier is preceded by a generic->async proxy fence.  A matrix that fits in L2 is
// loaded with the evict_last policy and the second pass of a step is served from L2 (profiles/: lts hit rate).
// All reductions are fixed-order: results are bit-reproducible run to run (not bit-identical to the stand-alone
// kernels: the partial sums are cut at CTA borders instead of 256-thread blocks).
#pragma once
#include "vector_kernels.cuh"

namespace bioen {

constexpr int kPEvalThreads = kPassThreads;   // 8 consumer warps + 1 producer warp
constexpr int kPEvalVec = kConsumerWarps * 32;
constexpr int kPSlots = 12;                   // doubles per CTA in the partials table

enum PEvalMode { kPEvalObjective = 0, kPEvalBoth = 1, kPEvalGradient = 2 };

struct PEvalArgs {
    int method;   // 0 log-weights, 1 forces (tile path)
    int mode;     // PEvalMode
    int M, N;
    PassArgs row, col;   // geometry and partial-sum buffers; the vector pointers are filled in per phase
    double* x;           // variables: N (logw) / M (forces)
    const double* xp;
    const double* d;
    double stp;
    const double* Gv;    // G (logw) / w0 (forces)
    double* w;
    double* aux_n;       // forces: x_j, later E_j
    double* aux_n2;      // forces: lr_j
    double* grad;
    const double* ddir;
    const double* Yobs;
    double* ab;
    double* avg;
    double* msum;        // sharded logw: M + 5 doubles sent to the peers
    double theta;
    double* sc;
    double* part;        // [gridDim.x][kPSlots]
    unsigned long long* bar;       // [0] arrival count, [16] generation (grid barrier)
    unsigned int* ticket;
    P2PDev p2p;          // nranks > 1: sharded log-weights run, exchanges inside the kernel
};

// barriers a launch passes (diagnostics)
__host__ __device__ inline int peval_num_barriers(int method, int mode, bool sharded) {
    if (method == 0) return mode == kPEvalObjective ? 3 : mode == kPEvalBoth ? (sharded ? 5 : 4) : 1;
    return mode == kPEvalObjective ? 4 : mode == kPEvalBoth ? 7 : 3;
}

// what replaces a grid barrier where every CTA has just written the SAME values redundantly (M-vectors finished by
// all CTAs instead of by CTA 0 + barrier): the CTA's own stores must be complete and visible to its bulk copies
__device__ __forceinline__ void peval_cta_fence() {
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncthreads();
    asm volatile("fence.proxy.async;" ::: "memory");
}

__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// all threads of all CTAs; `nbar` counts the barriers this CTA has passed in this launch
__device__ __forceinline__ void peval_grid_barrier(const PEvalArgs& a, unsigned int& nbar) {
    // ordinary stores of this phase must be visible to the bulk / tensor copies (async proxy) of the next one
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncthreads();
    ++nbar;
    if (threadIdx.x == 0) {
        // Sense-reversing barrier that needs no state from the host:
        // a.bar[0] counts arrivals, a.bar[16] (its own cache line) is the generation.  Every CTA reads the generation
        // BEFORE it arrives; the CTA that completes the count resets it and publishes generation + 1; the others poll
        // the generation word, so the spinning loads do not contend with the arriving atomics.
        unsigned long long* count = a.bar;
        unsigned long long* gen = a.bar + 16;
        const unsigned long long my_gen = ld_acquire_gpu_u64(gen);
        __threadfence();
        if (atomicAdd(count, 1ULL) + 1 == (unsigned long long)gridDim.x) {
            *count = 0;
            __threadfence();
            asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(gen), "l"(my_gen + 1) : "memory");
        } else {
            while (ld_acquire_gpu_u64(gen) == my_gen) {
            }
        }
        __threadfence();
    }
    __syncthreads();
    asm volatile("fence.proxy.async;" ::: "memory");
}

template <int MODE, bool SUB, typename T>
__device__ __forceinline__ void peval_pass(unsigned char* smem, const CUtensorMap* tmap, const PassArgs& pa,
                                           RingPos& prod, RingPos& cons) {
    TileWalk tw;
    tw.init(MODE, pa, (int)blockIdx.x, (int)gridDim.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == kConsumerWarps) {
        if (lane == 0 && tw.left > 0) pass_produce<MODE, SUB, T>(smem, tmap, pa, tw, prod);
    } else if (tw.left > 0) {
        pass_consume<MODE, SUB, T>(smem, pa, tw, cons);
    }
}

// block-wide merge of (max, sum-of-exp) pairs and one plain sum, result in thread 0: the maximum first (shuffles
// only), then ONE rescaling exp per thread and plain sums -- instead of the exp chain of pairwise lse_merge steps
// (5 + 5 dependent merges of two exps each in block_lse), which is latency a persistent CTA feels in every phase
__device__ __forceinline__ void block_lse2(double& m, double& s, double& xn, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double mm = warp_max(m);
    __syncthreads();
    if (lane == 0) red[wid] = mm;
    __syncthreads();
    mm = red[0];
    for (int w = 1; w < nw; ++w) mm = fmax(mm, red[w]);
    s = (s == 0.0) ? 0.0 : s * exp(m - mm);
    s = warp_sum(s);
    xn = warp_sum(xn);
    __syncthreads();
    if (lane == 0) { red[32 + wid] = s; red[64 + wid] = xn; }
    __syncthreads();
    if (wid == 0) {
        s = warp_sum(lane < nw ? red[32 + lane] : 0.0);
        xn = warp_sum(lane < nw ? red[64 + lane] : 0.0);
    }
    m = mm;
}

// Row sums of a row pass from its per-CTA slots, for the rows this thread / warp is responsible for.  When a run of
// tiles is spread over many CTAs (few row tiles, many column blocks: the ala5 shape has 131 slots per row) a thread
// that adds its row's slots one after the other is a chain of 131 L2 latencies; then a WARP takes a row (lanes stride
// over the slots, fixed-order shuffle sum).  The choice depends only on the geometry, so results stay reproducible.
//   f(i, sum) is called once per row, by the lane / thread that owns the row.
template <class F>
__device__ __forceinline__ void peval_row_sums(const PassArgs& row, int M, F f) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    const int max_slots = pass_num_slots(0, row.nCB, row.chunk);
    if (max_slots >= 16) {
        for (int i = wid; i < M; i += nw) {
            const int ns = pass_num_slots(i / kTileR, row.nCB, row.chunk);
            double sum = 0.0;
            for (int q = lane; q < ns; q += 32) sum += __ldcg(row.partial + (size_t)q * row.ld + i);
            sum = warp_sum(sum);
            if (lane == 0) f(i, sum);
        }
    } else {
        for (int i = tid; i < M; i += blockDim.x) {
            const int ns = pass_num_slots(i / kTileR, row.nCB, row.chunk);
            double sum = 0.0;
            for (int q = 0; q < ns; ++q) sum += __ldcg(row.partial + (size_t)q * row.ld + i);
            f(i, sum);
        }
    }
}

// block-wide (all kPEvalThreads threads) fixed-order reduction of 2 sums and 1 max; result in thread 0
__device__ __forceinline__ void block_sum2_max(double& a0, double& a1, double& mx, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    a0 = warp_sum(a0); a1 = warp_sum(a1); mx = warp_max(mx);
    __syncthreads();
    if (lane == 0) { red[wid] = a0; red[32 + wid] = a1; red[64 + wid] = mx; }
    __syncthreads();
    if (wid == 0) {
        a0 = warp_sum(lane < nw ? red[lane] : 0.0);
        a1 = warp_sum(lane < nw ? red[32 + lane] : 0.0);
        mx = warp_max(lane < nw ? red[64 + lane] : 0.0);
    }
}

template <typename T>
__global__ void __launch_bounds__(kPEvalThreads, 1)
    persistent_eval_kernel(const __grid_constant__ CUtensorMap tmap, const PEvalArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
    __shared__ double red[3 * 32];
    __shared__ double s_val[8];
    const int tid = threadIdx.x, b = blockIdx.x, G = gridDim.x;
    const bool vec = tid < kPEvalVec;                      // the producer warp has no vector elements
    const int j0 = b * kPEvalVec + tid, jstride = G * kPEvalVec;
    unsigned int nbar = 0;
    RingPos prod{0, 1}, cons{0, 0};
    pass_ring_init<T>(smem);
    if (tid == kConsumerWarps * 32) prefetch_tensormap(&tmap);
    __syncthreads();
    double* mypart = a.part + (size_t)b * kPSlots;
    const bool sharded = a.p2p.nranks > 1;

    if (a.method == 0) {
        // =========================================================================== log-weights
        if (a.mode != kPEvalGradient) {
            // ---- V0: trial point, CTA-local (max, sum exp(x - max)), ||x||^2
            double m = -DBL_MAX, s = 0.0, xn = 0.0;
            if (vec) {
                for (int j = j0; j < a.N; j += jstride) {
                    double x;
                    if (a.xp) { x = fma(a.stp, a.d[j], a.xp[j]); a.x[j] = x; }
                    else x = a.x[j];
                    xn = fma(x, x, xn);
                    if (x > m) { s = s * exp(m - x) + 1.0; m = x; }
                    else s += exp(x - m);
                }
            }
            block_lse2(m, s, xn, red);
            if (tid == 0) { mypart[0] = m; mypart[1] = s; mypart[2] = xn; }
            peval_grid_barrier(a, nbar);
            // ---- V1: every CTA merges the G pairs in the same fixed order; weights and the prior sums
            m = -DBL_MAX; s = 0.0; xn = 0.0;
            for (int q = tid; q < G; q += kPEvalThreads) {
                lse_merge(m, s, __ldcg(a.part + (size_t)q * kPSlots), __ldcg(a.part + (size_t)q * kPSlots + 1));
                xn += __ldcg(a.part + (size_t)q * kPSlots + 2);
            }
            block_lse2(m, s, xn, red);
            if (tid == 0) {
                s_val[0] = m; s_val[1] = s;
                if (b == 0) { a.sc[SC_LSE_MAX] = m; a.sc[SC_LSE_SUM] = s; a.sc[SC_XNORM2] = xn; }
            }
            __syncthreads();
            const double Mx = s_val[0], S = s_val[1];
            // sharded: e_j = exp(g_j - rank-local max); the normalisation travels with the row sums (V3)
            const double inv = sharded ? 1.0 : 1.0 / S;
            double v[3] = {0.0, 0.0, 0.0};
            if (vec) {
                for (int j = j0; j < a.N; j += jstride) {
                    const double g = a.x[j], Gj = a.Gv[j];
                    const double w = exp(g - Mx) * inv;
                    a.w[j] = w;
                    v[0] = fma(g - Gj, w, v[0]);
                    v[1] = fma(g, w, v[1]);
                    v[2] = fma(Gj, w, v[2]);
                }
            }
            block_sum<3>(v, red);
            if (tid == 0) { mypart[3] = v[0]; mypart[4] = v[1]; mypart[5] = v[2]; }
            peval_grid_barrier(a, nbar);
            // ---- P2: row pass  avg ~ Y . w
            {
                PassArgs pa = a.row;
                pa.vN = a.w;
                peval_pass<kRowPass, false, T>(smem, &tmap, pa, prod, cons);
            }
            peval_grid_barrier(a, nbar);
            // ---- V3: finish the objective.  One GPU: EVERY CTA does it (identical values, fixed order; only CTA 0
            // writes the scalar file), which saves the grid barrier that would otherwise publish avg / ab to the
            // column pass.  Sharded: CTA 0 alone (it runs the exchange), then a barrier.
            if (a.mode == kPEvalObjective && b != 0) return;
            if (b == 0 || !sharded) {
                double t[3] = {0.0, 0.0, 0.0};
                for (int q = tid; q < G; q += kPEvalThreads) {
                    t[0] += __ldcg(a.part + (size_t)q * kPSlots + 3);
                    t[1] += __ldcg(a.part + (size_t)q * kPSlots + 4);
                    t[2] += __ldcg(a.part + (size_t)q * kPSlots + 5);
                }
                block_sum<3>(t, red);
                if (tid == 0) { s_val[2] = t[0]; s_val[3] = t[1]; s_val[4] = t[2]; }
                __syncthreads();
                if (!sharded) {
                    double c[1] = {0.0};
                    peval_row_sums(a.row, a.M, [&](int i, double sum) {
                        const double r = sum - a.Yobs[i];
                        a.avg[i] = sum;
                        reinterpret_cast<double2*>(a.ab)[i] = make_double2(r, sum);
                        c[0] = fma(r, r, c[0]);
                    });
                    block_sum<1>(c, red);
                    if (tid == 0 && b == 0) {
                        const double chi2 = 0.5 * c[0];
                        const double prior = (s_val[2] - (Mx + log(S)) + a.sc[SC_LOGS0]) * a.theta;
                        a.sc[SC_GMAX] = Mx; a.sc[SC_S] = S;
                        a.sc[SC_GBAR] = s_val[3]; a.sc[SC_CAPGBAR] = s_val[4];
                        a.sc[SC_CHI2] = chi2; a.sc[SC_PRIOR] = prior; a.sc[SC_F] = prior + chi2;
                    }
                } else {
                    // this rank's M + 5 doubles -> every rank; combination in rank order (see
                    // k_logw_rows_exchange_finalize, the stand-alone twin of this block)
                    __shared__ double s_c[kP2PMaxRanks];
                    peval_row_sums(a.row, a.M, [&](int i, double sum) { a.msum[i] = sum; });
                    if (tid == 0) {
                        a.msum[a.M] = s_val[2]; a.msum[a.M + 1] = s_val[3]; a.msum[a.M + 2] = s_val[4];
                        a.msum[a.M + 3] = Mx; a.msum[a.M + 4] = S;
                    }
                    int fail;
                    const double* in = p2p_deliver_and_wait(a.p2p, a.msum, a.M + 5, &fail);
                    const long long cap = a.p2p.cap;
                    const int R = a.p2p.nranks;
                    if (tid == 0) {
                        double mx = __ldcg(in + a.M + 3);
                        for (int r = 1; r < R; ++r) mx = fmax(mx, __ldcg(in + r * cap + a.M + 3));
                        double Sg = 0.0;
                        for (int r = 0; r < R; ++r) {
                            s_c[r] = exp(__ldcg(in + r * cap + a.M + 3) - mx);
                            Sg += __ldcg(in + r * cap + a.M + 4) * s_c[r];
                        }
                        s_val[5] = 1.0 / Sg;
                        a.sc[SC_GMAX] = mx; a.sc[SC_S] = Sg;
                        a.sc[SC_WSCALE] = fail ? p2p_nan() : s_c[a.p2p.rank] / Sg;
                    }
                    __syncthreads();
                    const double ginv = s_val[5];
                    double c[1] = {0.0};
                    for (int i = tid; i < a.M; i += kPEvalThreads) {
                        double sum = 0.0;
                        for (int r = 0; r < R; ++r) sum = fma(__ldcg(in + r * cap + i), s_c[r], sum);
                        sum *= ginv;
                        const double rr = sum - a.Yobs[i];
                        a.avg[i] = sum;
                        reinterpret_cast<double2*>(a.ab)[i] = make_double2(rr, sum);
                        c[0] = fma(rr, rr, c[0]);
                    }
                    block_sum<1>(c, red);
                    if (tid == 0) {
                        double t3[3];
                        for (int k = 0; k < 3; ++k) {
                            double sum = 0.0;
                            for (int r = 0; r < R; ++r) sum = fma(__ldcg(in + r * cap + a.M + k), s_c[r], sum);
                            t3[k] = sum * ginv;
                        }
                        const double chi2 = 0.5 * c[0];
                        const double prior = (t3[0] - (a.sc[SC_GMAX] + log(a.sc[SC_S])) + a.sc[SC_LOGS0]) * a.theta;
                        a.sc[SC_GBAR] = t3[1]; a.sc[SC_CAPGBAR] = t3[2];
                        a.sc[SC_CHI2] = chi2; a.sc[SC_PRIOR] = prior;
                        a.sc[SC_F] = fail ? p2p_nan() : prior + chi2;
                    }
                }
            }
            if (a.mode == kPEvalObjective) return;
            if (sharded) peval_grid_barrier(a, nbar);
            else peval_cta_fence();   // (V5 reads <g>, <G> from the scalar file after the barrier that follows P4)
        }
        // ---- P4: column pass  c_j = sum_i r_i (y_ij - avg_i)
        {
            PassArgs pa = a.col;
            pa.ab = a.ab;
            peval_pass<kColPass, true, T>(smem, &tmap, pa, prod, cons);
        }
        peval_grid_barrier(a, nbar);
        // ---- V5: gradient and its scalars; the CTA that arrives last finishes (and exchanges, sharded)
        {
            const double gbar = a.sc[SC_GBAR], Gbar = a.sc[SC_CAPGBAR];
            const double wscale = sharded ? a.sc[SC_WSCALE] : 1.0;
            double dg = 0.0, gn = 0.0, gi = 0.0;
            if (vec) {
                for (int j = j0; j < a.N; j += jstride) {
                    const int ns = pass_num_slots(j / kTileC, a.col.nRT, a.col.chunk);
                    double c = 0.0;
                    for (int q = 0; q < ns; ++q) c += __ldcg(a.col.partial + (size_t)q * a.col.ld + j);
                    double w = a.w[j];
                    if (sharded) { w *= wscale; a.w[j] = w; }
                    const double gr = w * a.theta * (a.x[j] - gbar - a.Gv[j] + Gbar) + w * c;
                    a.grad[j] = gr;
                    if (a.ddir) dg = fma(gr, a.ddir[j], dg);
                    gn = fma(gr, gr, gn);
                    gi = fmax(gi, fabs(gr));
                }
            }
            double v[3] = {dg, gn, gi};
            if (!grid_sum_max_last<2>(v, a.part, a.ticket, red)) return;
            if (!sharded) {
                if (tid == 0) { a.sc[SC_DG] = v[0]; a.sc[SC_GNORM2] = v[1]; a.sc[SC_GINF] = v[2]; }
                return;
            }
            __shared__ double xs[4];
            if (tid == 0) { xs[0] = v[0]; xs[1] = v[1]; xs[2] = a.sc[SC_XNORM2]; xs[3] = v[2]; }
            int fail;
            const double* in = p2p_deliver_and_wait(a.p2p, xs, 4, &fail);
            if (tid == 0) {
                double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
                for (int r = 0; r < a.p2p.nranks; ++r) {
                    const double* q = in + r * a.p2p.cap;
                    t0 += __ldcg(q); t1 += __ldcg(q + 1); t2 += __ldcg(q + 2); t3 = fmax(t3, __ldcg(q + 3));
                }
                if (fail) t0 = t1 = t2 = t3 = p2p_nan();
                a.sc[SC_DG] = t0; a.sc[SC_GNORM2] = t1; a.sc[SC_XNORM2] = t2; a.sc[SC_GINF] = t3;
            }
        }
        return;
    }

    // =============================================================================== forces (tile path)
    if (a.mode != kPEvalGradient) {
        // ---- V0 (every CTA, identical values: no grid barrier): f = xp + stp d, ab = {f_i, 0}, ||f||^2
        {
            double c[1] = {0.0};
            for (int i = tid; i < a.M; i += kPEvalThreads) {
                double x;
                if (a.xp) { x = fma(a.stp, a.d[i], a.xp[i]); a.x[i] = x; }
                else x = a.x[i];
                reinterpret_cast<double2*>(a.ab)[i] = make_double2(x, 0.0);
                c[0] = fma(x, x, c[0]);
            }
            block_sum<1>(c, red);
            if (tid == 0 && b == 0) a.sc[SC_XNORM2] = c[0];
        }
        peval_cta_fence();
        // ---- P1: column pass  x_j = sum_i f_i y_ij
        {
            PassArgs pa = a.col;
            pa.ab = a.ab;
            peval_pass<kColPass, false, T>(smem, &tmap, pa, prod, cons);
        }
        peval_grid_barrier(a, nbar);
        // ---- V2: assemble x_j, CTA-local (max, sum w0 exp(x - max))
        double m = -DBL_MAX, s = 0.0, xn = 0.0;
        if (vec) {
            for (int j = j0; j < a.N; j += jstride) {
                const int ns = pass_num_slots(j / kTileC, a.col.nRT, a.col.chunk);
                double x = 0.0;
                for (int q = 0; q < ns; ++q) x += __ldcg(a.col.partial + (size_t)q * a.col.ld + j);
                a.aux_n[j] = x;
                const double pw = a.Gv[j];
                if (x > m) { s = s * exp(m - x) + pw; m = x; }
                else s += pw * exp(x - m);
            }
        }
        block_lse2(m, s, xn, red);
        if (tid == 0) { mypart[0] = m; mypart[1] = s; }
        peval_grid_barrier(a, nbar);
        // ---- V3: global (max, S); w_j, guarded log-ratio, KL
        m = -DBL_MAX; s = 0.0; xn = 0.0;
        for (int q = tid; q < G; q += kPEvalThreads)
            lse_merge(m, s, __ldcg(a.part + (size_t)q * kPSlots), __ldcg(a.part + (size_t)q * kPSlots + 1));
        block_lse2(m, s, xn, red);
        if (tid == 0) {
            s_val[0] = m; s_val[1] = s;
            if (b == 0) { a.sc[SC_LSE_MAX] = m; a.sc[SC_LSE_SUM] = s; a.sc[SC_GMAX] = m; a.sc[SC_S] = s; }
        }
        __syncthreads();
        {
            const double Mx = s_val[0], S = s_val[1];
            const double inv = 1.0 / S, logS = log(S);
            double v[1] = {0.0};
            if (vec) {
                for (int j = j0; j < a.N; j += jstride) {
                    const double x = a.aux_n[j], w0 = a.Gv[j];
                    const double w = inv * (w0 * exp(x - Mx));
                    const double lr = (w >= DBL_MIN && w0 >= DBL_MIN) ? (x - Mx - logS) : 0.0;
                    a.w[j] = w;
                    a.aux_n2[j] = lr;
                    v[0] = fma(lr, w, v[0]);
                }
            }
            block_sum<1>(v, red);
            if (tid == 0) mypart[3] = v[0];
        }
        peval_grid_barrier(a, nbar);
        // ---- P4: row pass  avg = Y . w
        {
            PassArgs pa = a.row;
            pa.vN = a.w;
            peval_pass<kRowPass, false, T>(smem, &tmap, pa, prod, cons);
        }
        peval_grid_barrier(a, nbar);
        // ---- V5 (every CTA, identical values; CTA 0 writes the scalars): avg, r, chi^2, objective; ab = {r_i, 0}
        if (a.mode == kPEvalObjective && b != 0) return;
        {
            double t[1] = {0.0};
            for (int q = tid; q < G; q += kPEvalThreads) t[0] += __ldcg(a.part + (size_t)q * kPSlots + 3);
            block_sum<1>(t, red);
            if (tid == 0) s_val[2] = t[0];
            __syncthreads();
            double c[1] = {0.0};
            peval_row_sums(a.row, a.M, [&](int i, double sum) {
                const double r = sum - a.Yobs[i];
                a.avg[i] = sum;
                reinterpret_cast<double2*>(a.ab)[i] = make_double2(r, 0.0);
                c[0] = fma(r, r, c[0]);
            });
            block_sum<1>(c, red);
            if (tid == 0 && b == 0) {
                const double chi2 = 0.5 * c[0], kl = s_val[2];
                a.sc[SC_KL] = kl; a.sc[SC_CHI2] = chi2; a.sc[SC_PRIOR] = kl * a.theta;
                a.sc[SC_F] = kl * a.theta + chi2;
            }
        }
        if (a.mode == kPEvalObjective) return;
        peval_cta_fence();
    }
    // ---- P6: column pass  t_j = sum_i r_i y_ij
    {
        PassArgs pa = a.col;
        pa.ab = a.ab;
        peval_pass<kColPass, false, T>(smem, &tmap, pa, prod, cons);
    }
    peval_grid_barrier(a, nbar);
    // ---- V7: E_j = (theta (1 + lr_j) + t_j) w_j
    if (vec) {
        for (int j = j0; j < a.N; j += jstride) {
            const int ns = pass_num_slots(j / kTileC, a.col.nRT, a.col.chunk);
            double t = 0.0;
            for (int q = 0; q < ns; ++q) t += __ldcg(a.col.partial + (size_t)q * a.col.ld + j);
            a.aux_n[j] = ((1.0 + a.aux_n2[j]) * a.theta + t) * a.w[j];
        }
    }
    peval_grid_barrier(a, nbar);
    // ---- P8: row pass  grad_i = sum_j (y_ij - avg_i) E_j
    {
        PassArgs pa = a.row;
        pa.vN = a.aux_n;
        pa.vMb = a.avg;
        peval_pass<kRowPass, true, T>(smem, &tmap, pa, prod, cons);
    }
    peval_grid_barrier(a, nbar);
    // ---- V9 (CTA 0): gradient and its scalars
    if (b == 0) {
        double dg = 0.0, gn = 0.0, gi = 0.0;
        peval_row_sums(a.row, a.M, [&](int i, double sum) {
            a.grad[i] = sum;
            if (a.ddir) dg = fma(sum, a.ddir[i], dg);
            gn = fma(sum, sum, gn);
            gi = fmax(gi, fabs(sum));
        });
        block_sum2_max(dg, gn, gi, red);
        if (tid == 0) { a.sc[SC_DG] = dg; a.sc[SC_GNORM2] = gn; a.sc[SC_GINF] = gi; }
    }
}

}  // namespace bioen
